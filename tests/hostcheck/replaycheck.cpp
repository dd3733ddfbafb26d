// Host build of replay (sf_enable_replay / sf_replay_load) on top of the host-check build with match logs, arena
// records, finished-arena calls, sf_step_list, the record lists, sf_action_mask and the per-agent step outputs.
//
// TEST INFRASTRUCTURE ONLY, like the files of the chain this one compiles as they are (logcheck.cpp and what it
// includes).  A handle's tapes, states and dealt rows live beside it here (the layout of the CUDA buffer), and the
// stepping calls run the same sf_step_body<true> as the EXTRAS kernels, with the handle's agent rows and tapes when
// those are on: the whole step, either half, and the list step with the lowest-index owner rule of hc_step_list.
// hc_replay_load checks and applies as sf_replay_check_kernel / sf_replay_apply_kernel do (lowest-index owner, all
// or nothing); the resets and loads disarm as sf_replay_disarm_kernel does.
#include "logcheck.cpp"

struct HcReplay {
    std::vector<uint8_t> tapes, dealt;
    std::vector<sf_replay_state> st;
    SfReplay rp;
};
static std::map<HcHandle *, HcReplay> g_replay;

static SfReplay replay_of(HcHandle *h)
{
    auto it = g_replay.find(h);
    return it == g_replay.end() ? SfReplay{nullptr, nullptr, nullptr, 0, 0} : it->second.rp;
}

static void replay_disarm(HcHandle *h, int env)
{
    const SfReplay rp = replay_of(h);
    if (rp.st) rp.st[env].flags &= ~SF_REPLAY_ARMED;
}

extern "C" {

// sf_enable_replay: zeroed tapes, states and dealt rows; 0, or -1 for a capacity out of range or another capacity
int hc_enable_replay(HcHandle *h, int cap)
{
    if (cap < 1 || cap > SF_LOG_CAP_MAX) return -1;
    if (replay_of(h).st) return cap == replay_of(h).cap ? 0 : -1;
    const int32_t row_bytes = (int32_t)sizeof(sf_log_head) + ((cap + 15) & ~15);
    HcReplay &r = g_replay[h];
    r.tapes.assign((size_t)h->d.n_envs * (size_t)row_bytes, 0);
    r.st.assign((size_t)h->d.n_envs, sf_replay_state{0, 0, 0, 0, 0});
    r.dealt.assign((size_t)h->d.n_envs * (size_t)h->k.n_agents, 0);
    r.rp = SfReplay{r.tapes.data(), r.st.data(), r.dealt.data(), row_bytes, cap};
    return 0;
}

int hc_replay_row_bytes(HcHandle *h) { return replay_of(h).row_bytes; }

// the whole step or a half, with every extra that is on (the EXTRAS kernels of sf_step, sf_step_a and sf_step_b)
void hc_step_replay(HcHandle *h, const uint8_t *actions, int half)
{
    int32_t *ao = agent_rows(h);
    const SfLog lg = log_of(h);
    const SfReplay rp = replay_of(h);
    SfStatDelta sd = {};
    for (int env = 0; env < h->d.n_envs; ++env)
        sf_step_body<true>(h->d, h->k, h->t, env, true, actions ? actions + (size_t)env * h->k.n_agents : nullptr, half, sd,
                           ao, lg, rp);
    add_stats(h, sd);
}

// the list step with every extra that is on
void hc_step_list_replay(HcHandle *h, const int32_t *ids, int n, const uint8_t *actions)
{
    int32_t *ao = agent_rows(h);
    const SfLog lg = log_of(h);
    const SfReplay rp = replay_of(h);
    std::vector<int32_t> claim((size_t)h->d.n_envs, INT32_MAX);
    for (int i = n - 1; i >= 0; --i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs) claim[ids[i]] = i;
    SfStatDelta sd = {};
    for (int i = 0; i < n; ++i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs && claim[ids[i]] == i)
            sf_step_body<true>(h->d, h->k, h->t, ids[i], true, actions + (size_t)i * h->k.n_agents, SF_HALF_BOTH, sd, ao, lg,
                               rp);
    add_stats(h, sd);
}

// sf_replay_load of rows [n][row_bytes] into arenas ids: the number of refused owning entries (nothing changes
// unless it is 0), or -1 if replay is off
int hc_replay_load(HcHandle *h, const uint8_t *rows, const int32_t *ids, int n)
{
    const SfReplay rp = replay_of(h);
    if (!rp.st) return -1;
    std::vector<int32_t> claim((size_t)h->d.n_envs, INT32_MAX);
    for (int i = n - 1; i >= 0; --i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs) claim[ids[i]] = i;
    auto head = [&](int i) { return *reinterpret_cast<const sf_log_head *>(rows + (size_t)i * rp.row_bytes); };
    int refused = 0;
    for (int i = 0; i < n; ++i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs && claim[ids[i]] == i && sf_replay_refused(head(i), rp.cap, h->k.mode)) ++refused;
    if (refused) return refused;
    for (int i = 0; i < n; ++i) {
        if (!(ids[i] >= 0 && ids[i] < h->d.n_envs && claim[ids[i]] == i)) continue;
        const sf_log_head hd = head(i);
        sf_reset_body<true>(h->d, h->k, h->t, ids[i], hd.tb, hd.serial, hd.episode, hd.level);
        sf_replay_arm(rp, ids[i], hd.n_symbols);
        memcpy(rp.tapes + (size_t)ids[i] * rp.row_bytes, rows + (size_t)i * rp.row_bytes, (size_t)rp.row_bytes);
    }
    return 0;
}

// sf_get(SF_FIELD_REPLAY) of arena env (5 int32) and sf_get(SF_FIELD_REPLAY_DEALT) of arena env (agents_per_env
// bytes); -1 if replay is off
int hc_replay_state(HcHandle *h, int env, int32_t *out, uint8_t *dealt)
{
    const SfReplay rp = replay_of(h);
    if (!rp.st) return -1;
    memcpy(out, &rp.st[env], sizeof(sf_replay_state));
    for (int a = 0; a < h->k.n_agents; ++a) dealt[a] = rp.dealt[(size_t)a * h->d.n_envs + env];
    return 0;
}

// hc_reset, then the arena's tape disarmed
void hc_reset_replay(HcHandle *h, int env, long long tb, long long serial)
{
    hc_reset(h, env, tb, serial);
    replay_disarm(h, env);
}

// hc_load_log, then the arena's tape disarmed if the record was accepted
int hc_load_replay(HcHandle *h, int env, const uint8_t *rec)
{
    const int rc = hc_load_log(h, env, rec);
    if (rc == 0) replay_disarm(h, env);
    return rc;
}

// hc_load_list_log, then every listed arena's tape disarmed if no owner was refused
int hc_load_list_replay(HcHandle *h, const uint8_t *records, int n_records, const int32_t *rows, const int32_t *ids, int n)
{
    const int refused = hc_load_list_log(h, records, n_records, rows, ids, n);
    if (refused == 0)
        for (int i = 0; i < n; ++i)
            if (ids[i] >= 0 && ids[i] < h->d.n_envs) replay_disarm(h, ids[i]);
    return refused;
}

void hc_disable_replay(HcHandle *h) { g_replay.erase(h); }

} // extern "C"
