// Host build of sf_action_mask on top of the host-check build with arena records, finished-arena calls, sf_step_list
// and the record lists.
//
// TEST INFRASTRUCTURE ONLY, like the files of the chain this one compiles as they are (reclistcheck.cpp and what it
// includes).  hc_action_mask runs the predicate of the CUDA kernel (sf_action_mask_slot after sf_bt_rebuild<false>);
// hc_action_mask_brute applies the definition of the mask (strikeforce_b200.h) literally, with the same sf_obey the
// step runs on copies of the arena, so that the tests pin the predicate against the rules themselves.
#include "reclistcheck.cpp"

#include <cstring>

extern "C" {

// sf_action_mask of arena env: out[a] for every agent slot a < agents_per_env
void hc_action_mask(HcHandle *h, int env, uint32_t *out)
{
    SfEnv e;
    sf_load_env(h->d, env, e);
    sf_bt_rebuild<false>(h->d, h->t, env, e);
    for (int a = 0; a < h->k.n_agents; ++a) out[a] = sf_action_mask_slot(h->d, h->k, h->t, env, e, a);
}

// the same masks by brute force: for every controllable slot and every symbol, save the arena's record, pick the
// arena up as a kernel does (sf_load_env, sf_bt_rebuild), obey the delivered symbol, store, take the canonical hash
// and the status, and load the record back.  Returns 0, or -1 if a restored arena's record is not byte for byte
// the one saved.
int hc_action_mask_brute(HcHandle *h, int env, uint32_t *out)
{
    const SfDev &d = h->d;
    const SfConst &k = h->k;
    const long bytes = hc_snapshot_bytes(h);
    std::vector<uint8_t> rec(bytes), back(bytes);
    hc_save(h, env, rec.data());
    auto obey = [&](int a, int c, unsigned long long *hash, int *status) {
        SfEnv e;
        sf_load_env(d, env, e);
        sf_bt_rebuild(d, h->t, env, e);
        sf_obey(d, k, h->t, env, e, a, c, SF_AT(d.h_pw, a), SF_AT(d.h_sel, a));
        sf_store_env(d, env, e);
        *hash = hc_hash(h, env);
        *status = hc_status(h, env);
        hc_load(h, env, rec.data());
        hc_save(h, env, back.data());
        return memcmp(rec.data(), back.data(), bytes) == 0;
    };
    const bool running = hc_status(h, env) == SF_RUNNING;
    const uint64_t live = d.mh[env];
    for (int a = 0; a < k.n_agents; ++a) {
        out[a] = 0;
        const uint32_t sel = SF_AT(d.h_sel, a);
        const bool rnpc = (sel & HS_RNPC) != 0;
        const bool player = a == k.ind || (k.mode == SF_MODE_ROYALE && a < k.n_players && !rnpc);
        const bool agent = !player && (sel & HS_AGENT) && a < k.n_agents && !rnpc;
        if (!running || !((live >> a) & 1) || !(player || agent)) continue;
        unsigned long long idle_hash;
        int idle_status;
        if (!obey(a, '+', &idle_hash, &idle_status)) return -1;
        for (int j = 0; j < SF_N_COMMANDS; ++j) {
            const int s = SF_COMMANDS[j];
            const int c = player || strchr("+xzqeawsd", s) ? s : '+';
            bool bit;
            if (s == '+') bit = true;
            else if (s == '_') bit = c == '_';
            else {
                unsigned long long hash;
                int status;
                if (!obey(a, c, &hash, &status)) return -1;
                bit = hash != idle_hash || status != idle_status;
            }
            if (bit) out[a] |= 1u << j;
        }
    }
    return 0;
}

const char *hc_commands(void) { return SF_COMMANDS; }

} // extern "C"
