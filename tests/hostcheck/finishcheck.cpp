// Host build of sf_list_finished / sf_reset_finished on top of the host-check build with arena records.
//
// TEST INFRASTRUCTURE ONLY, like hostcheck.cpp and snapcheck.cpp, which this file compiles as they are:
// hc_reset_finished / hc_list_finished loop over the arenas with the same per-arena functions of sf_core.cuh as
// the CUDA kernels (sf_reset_finished_body, sf_misc_finished), and hc_save is in the same library, so the tests can
// compare the records of a run that resets finished arenas with those of an auto-reset run byte for byte.
#include "snapcheck.cpp"

extern "C" {

// sf_reset_finished: every arena whose episode has ended since its last reset
void hc_reset_finished(HcHandle *h)
{
    for (int env = 0; env < h->d.n_envs; ++env) sf_reset_finished_body(h->d, h->k, h->t, env);
}

// sf_list_finished: the ids of those arenas, ascending, into ids[n_envs]; their number into *count
void hc_list_finished(HcHandle *h, int32_t *ids, int32_t *count)
{
    int32_t n = 0;
    for (int env = 0; env < h->d.n_envs; ++env)
        if (sf_misc_finished(h->d.misc[env])) ids[n++] = env;
    *count = n;
}

} // extern "C"
