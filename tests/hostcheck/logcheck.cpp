// Host build of the match logs (sf_enable_log / sf_log_list) on top of the host-check build with arena records,
// finished-arena calls, sf_step_list, the record lists, sf_action_mask and the per-agent step outputs.
//
// TEST INFRASTRUCTURE ONLY, like the files of the chain this one compiles as they are (agentcheck.cpp and what it
// includes).  A handle's tapes live beside it here (the row layout of the CUDA buffer), and the stepping calls run
// the same sf_step_body<true> as the EXTRAS kernels, with the handle's agent rows when those are on: the whole step,
// either half, and the list step with the lowest-index owner rule of hc_step_list.  The loads clear
// SF_LOG_COMPLETE as sf_log_unload_kernel does.
#include "agentcheck.cpp"

static std::map<HcHandle *, std::vector<uint8_t>> g_log_rows;
static std::map<HcHandle *, SfLog> g_log;

static SfLog log_of(HcHandle *h)
{
    auto it = g_log.find(h);
    return it == g_log.end() ? SfLog{nullptr, 0, 0} : it->second;
}

static void log_unload(HcHandle *h, int env)
{
    const SfLog lg = log_of(h);
    if (lg.rows) sf_log_at(lg, env)->flags &= ~SF_LOG_COMPLETE;
}

extern "C" {

// sf_enable_log: zeroed tapes; 0, or -1 for a capacity out of range or another capacity than the first call's
int hc_enable_log(HcHandle *h, int cap)
{
    if (cap < 1 || cap > SF_LOG_CAP_MAX) return -1;
    if (log_of(h).rows) return cap == log_of(h).cap ? 0 : -1;
    const int32_t row_bytes = (int32_t)sizeof(sf_log_head) + ((cap + 15) & ~15);
    std::vector<uint8_t> &rows = g_log_rows[h];
    rows.assign((size_t)h->d.n_envs * (size_t)row_bytes, 0);
    g_log[h] = SfLog{rows.data(), row_bytes, cap};
    return 0;
}

int hc_log_row_bytes(HcHandle *h) { return log_of(h).row_bytes; }

// hc_step with logs (the EXTRAS kernels of sf_step, sf_step_a and sf_step_b)
void hc_step_log(HcHandle *h, const uint8_t *actions, int half)
{
    int32_t *ao = agent_rows(h);
    const SfLog lg = log_of(h);
    SfStatDelta sd = {};
    for (int env = 0; env < h->d.n_envs; ++env)
        sf_step_body<true>(h->d, h->k, h->t, env, true, actions ? actions + (size_t)env * h->k.n_agents : nullptr, half, sd,
                           ao, lg);
    add_stats(h, sd);
}

// hc_step_list with logs
void hc_step_list_log(HcHandle *h, const int32_t *ids, int n, const uint8_t *actions)
{
    int32_t *ao = agent_rows(h);
    const SfLog lg = log_of(h);
    std::vector<int32_t> claim((size_t)h->d.n_envs, INT32_MAX);
    for (int i = n - 1; i >= 0; --i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs) claim[ids[i]] = i;
    SfStatDelta sd = {};
    for (int i = 0; i < n; ++i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs && claim[ids[i]] == i)
            sf_step_body<true>(h->d, h->k, h->t, ids[i], true, actions + (size_t)i * h->k.n_agents, SF_HALF_BOTH, sd, ao, lg);
    add_stats(h, sd);
}

// sf_log_list: row i < n of out is the tape of arena ids[i] (ids NULL: arena i), zeros for an id out of range.
// -1 if logs are off.
int hc_log_list(HcHandle *h, const int32_t *ids, int n, uint8_t *out)
{
    const SfLog lg = log_of(h);
    if (!lg.rows) return -1;
    for (int i = 0; i < n; ++i) {
        const int id = ids ? ids[i] : i;
        uint8_t *row = out + (size_t)i * lg.row_bytes;
        if (id >= 0 && id < h->d.n_envs) memcpy(row, sf_log_at(lg, id), (size_t)lg.row_bytes);
        else memset(row, 0, (size_t)lg.row_bytes);
    }
    return 0;
}

// hc_load, then SF_LOG_COMPLETE cleared on the arena if the record was accepted
int hc_load_log(HcHandle *h, int env, const uint8_t *rec)
{
    const int rc = hc_load(h, env, rec);
    if (rc == 0) log_unload(h, env);
    return rc;
}

// hc_load_list, then SF_LOG_COMPLETE cleared on every listed arena if no owner was refused
int hc_load_list_log(HcHandle *h, const uint8_t *records, int n_records, const int32_t *rows, const int32_t *ids, int n)
{
    const int refused = hc_load_list(h, records, n_records, rows, ids, n);
    if (refused == 0)
        for (int i = 0; i < n; ++i)
            if (ids[i] >= 0 && ids[i] < h->d.n_envs) log_unload(h, ids[i]);
    return refused;
}

void hc_disable_log(HcHandle *h)
{
    g_log.erase(h);
    g_log_rows.erase(h);
}

} // extern "C"
