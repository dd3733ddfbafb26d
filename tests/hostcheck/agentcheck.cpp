// Host build of the per-agent step outputs (sf_enable_agent_out) on top of the host-check build with arena records,
// finished-arena calls, sf_step_list, the record lists and sf_action_mask.
//
// TEST INFRASTRUCTURE ONLY, like the files of the chain this one compiles as they are (maskcheck.cpp and what it
// includes).  A handle's rows live beside it here ([field][slot][n_envs], the layout of the CUDA buffer), and the
// stepping calls run the same sf_step_body<true> as the AGENTS kernels: the whole step, either half, and the list
// step with the lowest-index owner rule of hc_step_list.
#include <map>

#include "maskcheck.cpp"

static std::map<HcHandle *, std::vector<int32_t>> g_agent_out;

static int32_t *agent_rows(HcHandle *h)
{
    auto it = g_agent_out.find(h);
    return it == g_agent_out.end() ? nullptr : it->second.data();
}

extern "C" {

// sf_enable_agent_out: zeroed rows; a second call does nothing
void hc_enable_agent_out(HcHandle *h)
{
    if (!agent_rows(h)) g_agent_out[h].assign((size_t)h->d.n_envs * h->k.n_agents * 5, 0);
}

// hc_step with agent outputs (the AGENTS kernels of sf_step, sf_step_a and sf_step_b)
void hc_step_agents(HcHandle *h, const uint8_t *actions, int half)
{
    int32_t *ao = agent_rows(h);
    SfStatDelta sd = {};
    for (int env = 0; env < h->d.n_envs; ++env)
        sf_step_body<true>(h->d, h->k, h->t, env, true, actions ? actions + (size_t)env * h->k.n_agents : nullptr, half, sd,
                           ao);
    add_stats(h, sd);
}

// hc_step_list with agent outputs
void hc_step_list_agents(HcHandle *h, const int32_t *ids, int n, const uint8_t *actions)
{
    int32_t *ao = agent_rows(h);
    std::vector<int32_t> claim((size_t)h->d.n_envs, INT32_MAX);
    for (int i = n - 1; i >= 0; --i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs) claim[ids[i]] = i;
    SfStatDelta sd = {};
    for (int i = 0; i < n; ++i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs && claim[ids[i]] == i)
            sf_step_body<true>(h->d, h->k, h->t, ids[i], true, actions + (size_t)i * h->k.n_agents, SF_HALF_BOTH, sd, ao);
    add_stats(h, sd);
}

// sf_get(SF_FIELD_AGENT_OUT) for arena env: out[a][field] for a < agents_per_env.  -1 if not enabled.
int hc_agent_out(HcHandle *h, int env, int32_t *out)
{
    const int32_t *ao = agent_rows(h);
    if (!ao) return -1;
    const size_t n = (size_t)h->d.n_envs, na = (size_t)h->k.n_agents;
    for (size_t a = 0; a < na; ++a)
        for (size_t f = 0; f < 5; ++f) out[a * 5 + f] = ao[(f * na + a) * n + (size_t)env];
    return 0;
}

void hc_disable_agent_out(HcHandle *h) { g_agent_out.erase(h); }

} // extern "C"
