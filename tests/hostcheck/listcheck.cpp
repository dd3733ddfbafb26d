// Host build of sf_step_list on top of the host-check build with finished-arena calls and arena records.
//
// TEST INFRASTRUCTURE ONLY, like hostcheck.cpp, snapcheck.cpp and finishcheck.cpp, which this file compiles as
// they are: hc_step_list loops over the list entries with the ownership rule of the CUDA path (the lowest live
// index of an id steps it) and calls the same sf_step_body as the kernel, so the tests can compare a handle stepped
// in parts with one stepped whole (hc_step), record for record.
#include <climits>

#include "finishcheck.cpp"

extern "C" {

// sf_step_list: entry i < n steps arena ids[i] with actions row i ([n][n_agents]) if the id is in range and no
// entry below i lists it
void hc_step_list(HcHandle *h, const int32_t *ids, int n, const uint8_t *actions)
{
    std::vector<int32_t> claim((size_t)h->d.n_envs, INT32_MAX);
    for (int i = n - 1; i >= 0; --i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs) claim[ids[i]] = i;
    SfStatDelta sd = {};
    for (int i = 0; i < n; ++i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs && claim[ids[i]] == i)
            sf_step_body(h->d, h->k, h->t, ids[i], true, actions + (size_t)i * h->k.n_agents, SF_HALF_BOTH, sd);
    add_stats(h, sd);
}

} // extern "C"
