/*
 * sf_lib.cu -- CUDA kernels (sm_100a) and the C ABI of include/strikeforce_b200.h.
 *
 * Execution model (DESIGN.md): one thread per arena, one warp per 32 neighbouring arenas,
 * persistent CTAs (one per SM) whose warps take 32-arena chunks round-robin.  The discrete
 * exp table of the RNG (128 KB) and the static map (9 KB) are staged in shared memory once
 * per CTA; per-arena state streams from / to HBM as structure-of-arrays (sf_state.h).  There
 * is no tensor-core work on this path (no dense contraction) and no CPU fallback: every entry
 * point fails with SF_ERR_NO_DEVICE when no CUDA device is usable.
 */
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "sf_canon_dev.cuh"
#include "sf_core.cuh"
#include "sf_host_setup.h"
#include "sf_obs.cuh"
#include "sf_snapshot.cuh"

#ifndef SF_CTA
#define SF_CTA 896 /* threads per CTA = arenas in flight per SM (one CTA per SM); 28 warps x 148 SMs = 4144 >= the 4096 chunks of 131072 arenas, 72 registers per thread */
#endif
#ifdef SF_FULL_EXP
#define SF_SMEM_EXP 131072
#else
#define SF_SMEM_EXP 65536 /* the first half of the exp table (sf_exp_m1) */
#endif
#define SF_SMEM_MAP SF_TCELLS /* 9,984, a multiple of 16 */
#define SF_SMEM_BT (SF_CTA * SF_BT_ENTRIES * 2) /* the bullet-flag tables of the CTA's arenas, [entry][thread] */
#define SF_SMEM_BYTES (SF_SMEM_EXP + SF_SMEM_MAP + SF_SMEM_BT) /* 161,536 B: the 164 KB carve-out, 92 KB of L1 */
#define SF_POW_LUT_LEN (1 << 21)
#define SF_EXPORT_CAP (1 << 18)

extern __shared__ __align__(16) uint8_t sf_smem[];

/* stage the shared tables: exp table (uint4 copies) and the static map */
__device__ __forceinline__ void sf_stage_tables(const SfDev &d, SfTabs &t)
{
    const uint4 *src = reinterpret_cast<const uint4 *>(d.exp_tab);
    uint4 *dst = reinterpret_cast<uint4 *>(sf_smem);
    for (int i = threadIdx.x; i < SF_SMEM_EXP / 16; i += blockDim.x) dst[i] = __ldg(src + i);
    const uint4 *msrc = reinterpret_cast<const uint4 *>(d.smap); /* padded to SF_SMEM_MAP on the host */
    uint4 *mdst = reinterpret_cast<uint4 *>(sf_smem + SF_SMEM_EXP);
    for (int i = threadIdx.x; i < SF_SMEM_MAP / 16; i += blockDim.x) mdst[i] = __ldg(msrc + i);
    __syncthreads();
    t.exp_tab = reinterpret_cast<const uint16_t *>(sf_smem);
    t.smap = sf_smem + SF_SMEM_EXP;
    t.log_tab = d.log_tab;
    t.rng_cst = d.rng_cst, t.E = d.E;
    /* entry i of this thread's table at [i][thread]: two neighbouring lanes share a bank, no more */
    t.bt = reinterpret_cast<uint16_t *>(sf_smem + SF_SMEM_EXP + SF_SMEM_MAP) + threadIdx.x;
    t.bt_stride = SF_CTA;
}

__device__ __forceinline__ void sf_flush_stats(const SfDev &d, const SfStatDelta &sd)
{
    const unsigned full = 0xffffffffu;
#define SF_RED(field, slot)                                                        \
    do {                                                                           \
        unsigned v = __reduce_add_sync(full, (unsigned)(sd.field));                \
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&d.stats[slot], (unsigned long long)v); \
    } while (0)
#define SF_RED_S(field, slot)                                                      \
    do {                                                                           \
        int v = (int)__reduce_add_sync(full, (unsigned)(sd.field));                \
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&d.stats[slot], (unsigned long long)(long long)v); \
    } while (0)
    SF_RED(steps, SF_STAT_STEPS);
    SF_RED(episodes, SF_STAT_EPISODES);
    SF_RED(wins, SF_STAT_WINS);
    SF_RED(deaths, SF_STAT_DEATHS);
    SF_RED(timeouts, SF_STAT_TIMEOUTS);
    SF_RED(truncated, SF_STAT_TRUNCATED);
    SF_RED(overflows, SF_STAT_OVERFLOWS);
    SF_RED(ub_guards, SF_STAT_UB_GUARDS);
    SF_RED(draws, SF_STAT_RNG_DRAWS);
    SF_RED(algo_bytes, SF_STAT_ALGO_BYTES);
    SF_RED_S(kills, SF_STAT_KILLS);
    SF_RED_S(tkills, SF_STAT_TEAMS_KILLS);
    SF_RED_S(loot, SF_STAT_LOOT);
#undef SF_RED
#undef SF_RED_S
}

/* one env-step (HALF: both halves, A only, B only) for every arena of the handle.
 *
 * lpw = arenas per warp (a power of two).  A full batch puts 32 arenas into every warp: one wave of
 * 131,072 arenas is what the machine holds.  A step of ONE warp lasts ~0.8 ms however few warps there
 * are (the tick is a serial chain, and the 32 arenas of a warp execute the union of their
 * branches), so a batch that would leave warp slots empty is spread over more warps with fewer
 * arenas each (sf_launch_step picks lpw): the extra lanes idle, the chain of every warp gets
 * shorter because fewer arenas diverge in it. */
template <int HALF>
__global__ void __launch_bounds__(SF_CTA, 1)
sf_step_kernel(const SfDev d, const __grid_constant__ SfConst k, const uint8_t *__restrict__ actions, int lpw)
{
    SfTabs t;
    sf_stage_tables(d, t);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nchunks = (d.n_envs + lpw - 1) / lpw;
#ifndef SF_NO_PHASE_BARRIERS
    /* every warp of the CTA makes the same number of passes (a pass without a chunk walks through
       with all lanes off), so that the phase barriers of sf_step_halves line up */
    const int per_pass = gridDim.x * (SF_CTA / 32);
    for (int base = 0; base < nchunks; base += per_pass) {
        const int chunk = base + blockIdx.x + gridDim.x * warp;
        bool valid = chunk < nchunks && lane < lpw && chunk * lpw + lane < d.n_envs;
        int env = valid ? chunk * lpw + lane : lane; /* an idle lane reads some arena's header and writes nothing */
#else
    for (int chunk = blockIdx.x + gridDim.x * warp; chunk < nchunks; chunk += gridDim.x * (SF_CTA / 32)) {
        bool valid = lane < lpw && chunk * lpw + lane < d.n_envs;
        int env = valid ? chunk * lpw + lane : lane;
#endif
        SfStatDelta sd;
        memset(&sd, 0, sizeof sd);
        sf_step_body(d, k, t, env, valid, (actions && valid) ? actions + (size_t)env * k.n_agents : nullptr, HALF, sd);
        __syncwarp();
        sf_flush_stats(d, sd);
    }
}

/* setup() + load_data() + _srand for the listed arenas (all when env_ids == NULL) */
__global__ void __launch_bounds__(SF_CTA, 1)
sf_reset_kernel(const SfDev d, const __grid_constant__ SfConst k, const int32_t *__restrict__ env_ids, int n,
                const int64_t *__restrict__ tb, const int64_t *__restrict__ serial)
{
    SfTabs t;
    sf_stage_tables(d, t);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int env = env_ids ? env_ids[i] : i;
        int64_t ge = k.env_id_base + env;
        int64_t tbv = tb ? tb[i] : sf_synth_tb(ge);
        int64_t sv = serial ? serial[i] : sf_synth_serial(ge, 0);
        sf_reset_body(d, k, t, env, tbv, sv, 0);
    }
}

/* the synthetic action stream of sf_synth.h for global step t */
__global__ void sf_synth_actions_kernel(uint8_t *actions, int n_envs, int n_agents, int64_t env_id_base, uint64_t step,
                                        const uint8_t *table, int table_len)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_envs * n_agents) return;
    int env = i / n_agents, a = i % n_agents;
    uint64_t z = sf_synth_draw_at(env_id_base + env, a, step);
    actions[i] = table[z % (uint64_t)table_len];
}

__device__ __forceinline__ void sf_global_tabs(const SfDev &d, SfTabs &t)
{
    t.exp_tab = d.exp_tab, t.log_tab = d.log_tab, t.smap = d.smap;
    t.rng_cst = d.rng_cst, t.E = d.E;
    t.bt = nullptr, t.bt_stride = 0; /* no tick runs in these kernels */
}

__global__ void sf_hash_kernel(const SfDev d, const __grid_constant__ SfConst k, uint64_t *out)
{
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= d.n_envs) return;
    SfTabs t;
    sf_global_tabs(d, t);
    SfHashSink sink{0};
    sf_canon_emit(d, k, t, env, sink);
    out[env] = sink.sum;
}

__global__ void sf_export_kernel(const SfDev d, const __grid_constant__ SfConst k, int env, int32_t *buf, long cap,
                                 long long *n_out)
{
    SfTabs t;
    sf_global_tabs(d, t);
    SfBufSink sink{buf, cap, 0, false};
    sf_canon_emit(d, k, t, env, sink);
    *n_out = sink.overflow ? -1 : sink.n;
}

__global__ void sf_counters_kernel(const SfDev d, const __grid_constant__ SfConst k, int32_t *out)
{
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= d.n_envs) return;
    uint32_t misc = d.misc[env];
    int32_t *o = out + (size_t)env * 8;
    o[0] = (int32_t)d.frame[env], o[1] = d.kills[env], o[2] = d.tkills[env], o[3] = d.loot[env];
    o[4] = d.chest[env], o[5] = (int32_t)d.steps[env], o[6] = (int32_t)((misc >> 8) & 0xFFu), o[7] = SF_AT(d.h_hp, k.ind);
}

__global__ void sf_population_kernel(const SfDev d, const __grid_constant__ SfConst k, int32_t *out)
{
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= d.n_envs) return;
    int32_t *o = out + (size_t)env * 6;
    o[0] = __popcll(d.mh[env]);
    o[1] = __popcll(SF_AT(d.mz, 0)) + __popcll(SF_AT(d.mz, 1));
    o[2] = __popcll(SF_AT(d.mb, 0)) + __popcll(SF_AT(d.mb, 1));
    o[3] = d.chest[env];
    o[4] = (int32_t)d.ntemp[env];
    o[5] = __popcll(SF_AT(d.mp, 0)) + __popcll(SF_AT(d.mp, 1));
}

/* gameplay::bot() up to Agent::predict (bots/bot-0.5/Custom.hpp:137-158).
 *
 * The product is 123,008 contiguous bytes per (arena, observer), almost all zeros (floor, cells
 * outside the map) -- a pure HBM-write problem whose enemy is latency: a CTA that waits (for a
 * load, for a barrier, for a store engine to release a buffer) writes nothing, and the bytes it
 * has in flight are all the bandwidth it gets.  So the kernel keeps nothing of the OUTPUT in
 * shared memory: it builds a small description of the window and then streams the 7,688 16-byte
 * chunks of the observation straight from registers with plain coalesced stores (512 contiguous
 * bytes per warp instruction; a store holds no resource of the CTA once it has issued, and 25 KB
 * of shared memory per CTA leave room for 8 CTAs per SM).
 *   1. entity -> window maps for the owning bullets and player-built cells (shared memory);
 *   2. the window is classified into a CODE per cell: 0 = nothing to show (floor, outside the map),
 *      1..15 = the static flags of a cell with nothing on it (wall, stairs, exit), 16 + i = the
 *      i-th DYNAMIC cell (anything in the overlay, or a bullet flag);
 *   3. describe() runs ONCE per dynamic cell -- all its entity loads in one round -- and its 32
 *      transformed features become row 16 + i of a table whose rows 1..15 hold what describe()
 *      gives for the static flags alone (filled once per CTA);
 *   4. the copy-out: 961 = 1 (mod 4), so every four channels are exactly 961 chunks and chunk q
 *      covers the same (channel offset, cell) quadruple in each of the eight 4-channel groups; a
 *      thread reads the four codes of its chunk once and then writes the chunk of every group:
 *      four predicated table reads and one 16-byte store each. */
#ifndef SF_OBS_CTA
#define SF_OBS_CTA 128
#endif
#ifndef SF_OBS_CTAS_PER_SM
#define SF_OBS_CTAS_PER_SM 8
#endif
#ifndef SF_OBS_CACHE
#define SF_OBS_CACHE 112 /* dynamic cells with a table row; any beyond are described again during the copy-out */
#endif
#define SF_OBS_ROWS (16 + SF_OBS_CACHE)
#define SF_OBS_PITCH (SF_OBS_CH + 1) /* floats per table row: odd, so that rows fall into different banks */
#define SF_OBS_LIST 976              /* entries per per-cell array (>= 961, keeps the arrays 16-byte aligned) */
#define SF_OBS_BEYOND 0xFFFFu        /* code of a dynamic cell without a table row */
#define SF_OBS_GROUP (SF_OBS_CELLS)  /* chunks per 4-channel group: 4 * 961 floats / 4 */
#define SF_OBS_SMEM (SF_OBS_ROWS * SF_OBS_PITCH * 4 + 4 * SF_OBS_LIST * 2 + 16)
static_assert(SF_OBS_CELLS % 4 == 1 && SF_OBS_CH % 4 == 0, "the copy-out relies on 4 channels = 961 whole chunks");
static_assert(SF_OBS_ROWS % 4 == 0, "the arrays behind the table stay 16-byte aligned");

/* (arena, observed human slot) of work item `item` */
__device__ __forceinline__ void sf_obs_item(int item, int nsel, uint32_t agent_mask, int *env, int *slot)
{
    uint32_t m = agent_mask;
    for (int i = item % nsel; i > 0; --i) m &= m - 1;
    *env = item / nsel, *slot = __ffs(m) - 1;
}

/* NHWC: the same values with the channel innermost, SF_OBS_NHWC of the header.  LIST (sf_observe_list): the
   arena of row r is env_ids[r / nsel] instead of r / nsel, an id outside [0, n_envs) gives a zero row, and the
   rows written are min(*list_n, n_items / nsel) (list_n == NULL: all); the launch shape is chosen for n_items. */
template <bool NHWC, bool LIST>
__global__ void __launch_bounds__(SF_OBS_CTA, SF_OBS_CTAS_PER_SM)
sf_observe_kernel(const SfDev d, const __grid_constant__ SfConst k, float *__restrict__ obs, uint32_t agent_mask,
                  int nsel, int n_items, int rows, int run_len, const int32_t *__restrict__ env_ids,
                  const int32_t *__restrict__ list_n)
{
    float *feat = reinterpret_cast<float *>(sf_smem);                         /* [row][SF_OBS_PITCH] */
    uint16_t *code = reinterpret_cast<uint16_t *>(feat + SF_OBS_ROWS * SF_OBS_PITCH); /* per window cell */
    uint16_t *dlist = code + SF_OBS_LIST;                                     /* window index of dynamic cell i */
    int16_t *bmap = reinterpret_cast<int16_t *>(dlist + SF_OBS_LIST);
    int16_t *tmap = bmap + SF_OBS_LIST;
    int *count = reinterpret_cast<int *>(tmap + SF_OBS_LIST);
    SfTabs t;
    sf_global_tabs(d, t);
    uint32_t fb = 0;
    if (threadIdx.x < 16) { /* describe() of a cell with nothing on it depends on its static flags only (no memory access) */
        SfEnv e0;
        e0.mb[0] = e0.mb[1] = 0, e0.ntemp = 0, e0.level = 1, e0.hw_h = 0, e0.env = 0;
        int32_t f[32];
        sf_describe_cell(d, k, 0, e0, 0, threadIdx.x, 0u, 0u, -1, -1, f);
#pragma unroll
        for (int c = 0; c < SF_OBS_CH; ++c) feat[threadIdx.x * SF_OBS_PITCH + c] = f[c] ? sf_obs_transform(d, f[c], &fb) : 0.f;
    }
    constexpr int PER = (SF_OBS_CELLS + SF_OBS_CTA - 1) / SF_OBS_CTA;
    if constexpr (LIST) {
        if (list_n) n_items = min(max(*list_n, 0), n_items / nsel) * nsel; /* CTAs whose runs lie beyond it exit */
    }
    for (int run = blockIdx.x; run * run_len < n_items; run += gridDim.x)
    for (int item = run * run_len, end = min(n_items, item + run_len); item < end; ++item) {
        int env, slot;
        sf_obs_item(item, nsel, agent_mask, &env, &slot);
        bool listed = true;
        if constexpr (LIST) { /* an id outside the handle reads arena 0 and observes nothing: a zero row */
            const int id = env_ids[env];
            listed = id >= 0 && id < d.n_envs;
            env = listed ? id : 0;
        }
        float *out = obs + (size_t)item * SF_OBS_LEN;
        /* the few header words the features need */
        SfEnv e;
        const uint32_t misc = d.misc[env];
        e.level = (int)(misc & 0xFFu), e.hw_h = (int)((misc >> 16) & 0xFFu);
        e.mb[0] = SF_AT(d.mb, 0), e.mb[1] = SF_AT(d.mb, 1);
        e.ntemp = d.ntemp[env];
        e.env = env;
        const bool observer = listed && slot < e.hw_h; /* a slot this episode never used sees nothing */
        const int vcell = observer ? (int)(SF_AT(d.h_pw, slot) & POS_CELL) : 0;
        const uint32_t team = observer ? (SF_AT(d.h_sel, slot) & HS_TEAM) : 0u;
        int vf, vr, vc;
        sf_tcell_decode(vcell, &vf, &vr, &vc);
        const int r0 = vr - SF_OBS_R, c0 = vc - SF_OBS_R;
        /* the loads of a thread's window cells are issued first: they are in flight while the entity
           maps are filled */
        uint32_t cv[PER];
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int w = threadIdx.x + q * SF_OBS_CTA;
            const int cell = (observer && w < SF_OBS_CELLS) ? sf_obs_cell(vcell, w / SF_OBS_WIN, w % SF_OBS_WIN) : -1;
            cv[q] = cell >= 0 ? ((uint32_t)SF_G(cell) | ((uint32_t)t.smap[cell] << 16)) : 0u;
        }
        __syncthreads(); /* every thread is done with the last window's codes and table */
        for (int i = threadIdx.x; i < SF_OBS_CELLS; i += SF_OBS_CTA) bmap[i] = -1, tmap[i] = -1;
        if (threadIdx.x == 0) *count = 0;
        __syncthreads();
        if (observer) {
            for (int b = threadIdx.x; b < SF_LIM_BULLETS; b += SF_OBS_CTA)
                if (m2_test(e.mb, b) && (SF_AT(d.b_meta, b) & BF_OWNS)) {
                    int bf, br, bc;
                    sf_tcell_decode((int)(SF_AT(d.b_pw, b) & POS_CELL), &bf, &br, &bc);
                    int wi = br - r0, wj = bc - c0;
                    if (bf == vf && wi >= 0 && wi < SF_OBS_WIN && wj >= 0 && wj < SF_OBS_WIN)
                        bmap[wi * SF_OBS_WIN + wj] = (int16_t)b;
                }
            for (int q = threadIdx.x; q < (int)e.ntemp; q += SF_OBS_CTA) {
                int tf, tr, tc;
                sf_tcell_decode((int)SF_T(d.t_cell, q), &tf, &tr, &tc);
                int wi = tr - r0, wj = tc - c0;
                if (tf == vf && wi >= 0 && wi < SF_OBS_WIN && wj >= 0 && wj < SF_OBS_WIN)
                    tmap[wi * SF_OBS_WIN + wj] = (int16_t)q;
            }
        }
        __syncthreads();
        /* classification (a cell that carries nothing but a bullet flag has an empty overlay word:
           bmap tells); one atomic per warp, not one per cell */
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int w = threadIdx.x + q * SF_OBS_CTA;
            const bool dyn = w < SF_OBS_CELLS && ((cv[q] & 0xFFFFu) || bmap[w] >= 0);
            const unsigned md = __ballot_sync(0xffffffffu, dyn);
            const unsigned lane = threadIdx.x & 31u;
            int base = 0;
            if (lane == 0 && md) base = atomicAdd(count, __popc(md));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (w < SF_OBS_CELLS) {
                uint32_t cd = (cv[q] >> 16) & 0xFu; /* M_WALL | M_UP | M_DOWN | M_EXIT: rows 1..15 of the table */
                if (dyn) {
                    const int i = base + __popc(md & ((1u << lane) - 1u));
                    cd = i < rows ? 16u + (uint32_t)i : SF_OBS_BEYOND;
                    if (i < rows) dlist[i] = (uint16_t)w;
                }
                code[w] = (uint16_t)cd;
            }
        }
        __syncthreads();
        /* describe() once per dynamic cell; its 32 transformed features become a table row */
        const int n_dyn = *count < rows ? *count : rows;
        for (int i = threadIdx.x; i < n_dyn; i += SF_OBS_CTA) {
            const int w = dlist[i], cell = sf_obs_cell(vcell, w / SF_OBS_WIN, w % SF_OBS_WIN);
            int32_t f[32];
            sf_describe_cell(d, k, env, e, cell, t.smap[cell], SF_G(cell), team, bmap[w], tmap[w], f);
#pragma unroll
            for (int c = 0; c < SF_OBS_CH; ++c) feat[(16 + i) * SF_OBS_PITCH + c] = f[c] ? sf_obs_transform(d, f[c], &fb) : 0.f;
        }
        __syncthreads();
        /* the copy-out: no barrier, no shared-memory buffer between the table and HBM; every store instruction
           of a warp covers 512 contiguous bytes.  What HBM makes of a pure store stream depends on its shape
           (tools/gpu_write_peak.py, profiles/r02_write_peak.txt): a plain store kernel in which every CTA writes
           one 123 KB observation front to back and then moves on reaches 5.1 TB/s, 6.1 TB/s when a CTA writes
           four or more consecutive observations (hence run_len).  Measured and rejected: storing the all-zero
           chunks first and the others in a second pass, lane-dense (41% slower: partial-warp stores); a warp
           vote that sends 128 empty cells in a row down a store-only path (7% slower) */
        float4 *dst = reinterpret_cast<float4 *>(out);
        if constexpr (NHWC) {
            /* channel-innermost: the 32 features of a cell are one table row = eight chunks; chunk idx
               covers features 4p..4p+3 of window cell idx / 8 */
#pragma unroll 4
            for (int idx = threadIdx.x; idx < SF_OBS_CELLS * (SF_OBS_CH / 4); idx += SF_OBS_CTA) {
                const int w = idx / (SF_OBS_CH / 4), p = idx % (SF_OBS_CH / 4);
                const uint32_t cd = code[w];
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (cd == SF_OBS_BEYOND) { /* more dynamic cells than table rows (rare) */
                    const int cell = sf_obs_cell(vcell, w / SF_OBS_WIN, w % SF_OBS_WIN);
                    int32_t f[32];
                    sf_describe_cell(d, k, env, e, cell, t.smap[cell], SF_G(cell), team, bmap[w], tmap[w], f);
                    int32_t g0 = 0, g1 = 0, g2 = 0, g3 = 0;
#pragma unroll
                    for (int c = 0; c < SF_OBS_CH / 4; ++c)
                        if (c == p) g0 = f[4 * c], g1 = f[4 * c + 1], g2 = f[4 * c + 2], g3 = f[4 * c + 3];
                    v.x = g0 ? sf_obs_transform(d, g0, &fb) : 0.f, v.y = g1 ? sf_obs_transform(d, g1, &fb) : 0.f;
                    v.z = g2 ? sf_obs_transform(d, g2, &fb) : 0.f, v.w = g3 ? sf_obs_transform(d, g3, &fb) : 0.f;
                } else if (cd) {
                    const float *r = feat + cd * SF_OBS_PITCH + 4 * p;
                    v = make_float4(r[0], r[1], r[2], r[3]);
                }
                __stcs(dst + idx, v);
            }
        } else {
            /* [32][31][31]: 961 = 1 (mod 4), so every four channels are exactly 961 chunks and chunk q covers
               the same (channel offset, cell) quadruple in each of the eight 4-channel groups; a thread reads
               the four codes of its chunk once and then writes the chunk of every group: four predicated table
               reads (the group is an immediate) and one 16-byte store each.  The price is alignment: the warp
               stores of group g start 16 g bytes off a 512-byte boundary, and a plain store kernel shows what
               HBM makes of that (tools/gpu_write_peak.py: 6.1 TB/s aligned, 5.75 TB/s on any other 32-byte
               boundary, 4.4 TB/s from the middle of a 32-byte sector).  Measured and rejected
               (profiles/r02_variants.txt): a walk with every warp store on a 512-byte boundary (chunk
               g * 960 + r, the codes packed once per window into one word per chunk) has to unpack and
               address the four codes per chunk AND per group -- twice the instructions of this loop,
               3.76 ms; this loop with a thread owning chunk q of the even groups and q - 1 of the odd ones
               (every warp store then starts on a sector boundary) decodes twice, 3.89 ms. */
            for (int q = threadIdx.x; q < SF_OBS_GROUP; q += SF_OBS_CTA) {
                int cc = (4 * q) / SF_OBS_CELLS, w = 4 * q - cc * SF_OBS_CELLS; /* channel offset in the group, window cell */
                int row[4];  /* table offset of element j of the chunk: row * pitch + channel offset, -1 = zero */
                bool beyond = false;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t cd = code[w];
                    row[j] = cd ? (int)cd * SF_OBS_PITCH + cc : -1;
                    if (cd == SF_OBS_BEYOND) beyond = true, row[j] = -2 - w;
                    if (++w == SF_OBS_CELLS) w = 0, ++cc;
                }
                if (!beyond) {
#pragma unroll
                    for (int g = 0; g < SF_OBS_CH / 4; ++g) {
                        float4 v;
                        v.x = row[0] >= 0 ? feat[row[0] + 4 * g] : 0.f;
                        v.y = row[1] >= 0 ? feat[row[1] + 4 * g] : 0.f;
                        v.z = row[2] >= 0 ? feat[row[2] + 4 * g] : 0.f;
                        v.w = row[3] >= 0 ? feat[row[3] + 4 * g] : 0.f;
                        __stcs(dst + g * SF_OBS_GROUP + q, v);
                    }
                } else { /* more dynamic cells than table rows (rare): those are described here, once per chunk */
                    float val[4][SF_OBS_CH / 4];
                    int cj = (4 * q) / SF_OBS_CELLS, wj = 4 * q - cj * SF_OBS_CELLS;
#pragma unroll 1
                    for (int j = 0; j < 4; ++j) {
                        if (row[j] <= -2) {
                            const int cell = sf_obs_cell(vcell, wj / SF_OBS_WIN, wj % SF_OBS_WIN);
                            int32_t f[32];
                            sf_describe_cell(d, k, env, e, cell, t.smap[cell], SF_G(cell), team, bmap[wj], tmap[wj], f);
                            for (int g = 0; g < SF_OBS_CH / 4; ++g) val[j][g] = f[4 * g + cj] ? sf_obs_transform(d, f[4 * g + cj], &fb) : 0.f;
                        } else {
                            for (int g = 0; g < SF_OBS_CH / 4; ++g) val[j][g] = row[j] >= 0 ? feat[row[j] + 4 * g] : 0.f;
                        }
                        if (++wj == SF_OBS_CELLS) wj = 0, ++cj;
                    }
                    for (int g = 0; g < SF_OBS_CH / 4; ++g)
                        __stcs(dst + g * SF_OBS_GROUP + q, make_float4(val[0][g], val[1][g], val[2][g], val[3][g]));
                }
            }
        }
    }
    if (fb) atomicAdd(&d.stats[SF_STAT_RESERVED0], (unsigned long long)fb);
}

/* Measured and rejected (profiles/r02_variants.txt; the code is in the history of this file): a
   warp-specialised version of this kernel -- four producer warps describing window i+1 into one of two
   description buffers while four consumer warps stream window i out of the other, named barriers in
   between -- 4.80 ms against 3.71 ms: half the CTA's threads issue no stores. */

/* Random::_srand + n _rand() draws for a batch of independent streams (random.hpp:54-76) */
__global__ void __launch_bounds__(SF_CTA, 1)
sf_rng_kernel(const SfDev d, const int64_t *tb, const int64_t *serial, int n_streams, int n_draws, int32_t *out)
{
    SfTabs t;
    sf_stage_tables(d, t);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_streams; i += gridDim.x * blockDim.x) {
        /* stand-alone stream: seed, warm up and draw in registers (no arena state is touched) */
        uint32_t Lp[9], c[18];
        int64_t a = tb[i], b = serial[i];
        for (int q = 0; q < 18; ++q) {
            c[q] = (2u * (uint32_t)(a % 10 + 1)) | ((2u * (uint32_t)t.log_tab[(uint32_t)(b % 10)]) << 8);
            a /= 10, b /= 10;
        }
        for (int q = 0; q < 9; ++q) Lp[q] = 0u;
        uint32_t n = 0;
        for (; n < SF_WARM_DRAWS; ++n) sf_warm_draw(t, Lp, c, n);
        for (int j = 0; j < n_draws; ++j, ++n) {
            sf_warm_draw(t, Lp, c, n);
            out[(size_t)j * n_streams + i] = (int32_t)((sf_exp_m1(t, 2u * (Lp[8] >> 16)) + 1u) & 1023u);
        }
    }
}

/* sf_save / sf_load: arena records (sf_snapshot.cuh) to and from a device buffer.
 *
 * A pure HBM copy.  The list is cut into tiles of 32 entries and each (tile, work item of the layout) pair
 * is one turn of a CTA, so even a short list keeps every SM busy.  A block item (overlay, built list,
 * sf_step_out) is a straight 16-byte (8-byte for an odd built-list tail) vector copy of each arena's
 * contiguous bytes.  A SoA item covers consecutive [slot][E] sections: row s of the tile's 32 arenas is
 * read with one lane per arena (coalesced when the ids are consecutive, as in the all-arenas case; scattered
 * otherwise, by the same code), transposed through shared memory into each arena's contiguous run of the
 * record, and that run written with vector stores.  A load runs the same steps backwards.  Record-side
 * stores of a save and record-side loads of a load are streaming (.cs): the records are not read again
 * soon, the state is. */
#define SF_SNAP_CTA 256
#define SF_SNAP_CTAS_PER_SM 8
#define SF_SNAP_STAGE (SF_SNAP_TILE * (SF_SNAP_STAGE_RUN + 16))

/* stage stride of a run of P bytes per arena: an odd number of 16-byte chunks, so that the arenas of a row
   do not all fall into the same shared-memory banks */
__device__ __forceinline__ uint32_t sf_snap_stride(uint32_t P) { return ((P >> 4) | 1u) << 4; }

/* row-by-row transpose of one SoA section between the arenas' columns in the state and the stage */
template <bool SAVE, class T>
__device__ __forceinline__ void sf_snap_soa(const SfSnapSeg &g, int E, uint8_t *st, uint32_t S, int nv, const int *s_env)
{
    T *dev = reinterpret_cast<T *>(g.dev);
    /* a save also writes the zero padding at the end of the section (rows beyond g.rows) */
    const int rows = SAVE ? (int)(sf_snap_seg_bytes(g) / sizeof(T)) : (int)g.rows;
#pragma unroll 4
    for (int q = threadIdx.x; q < rows * SF_SNAP_TILE; q += SF_SNAP_CTA) {
        const int r = q >> 5, j = q & 31;
        if (j >= nv) continue;
        T *s = reinterpret_cast<T *>(st + (size_t)j * S) + r;
        if (SAVE) *s = r < (int)g.rows ? __ldg(dev + (size_t)r * E + s_env[j]) : T(0);
        else dev[(size_t)r * E + s_env[j]] = *s;
    }
}

/* bytes [lo, hi) of the per-arena block g for the tile's arenas; bytes at or beyond g.elem are the record's
   padding (written as zeros by a save, skipped by a load) */
template <bool SAVE, class V>
__device__ __forceinline__ void sf_snap_block(const SfSnapSeg &g, uint32_t lo, uint32_t hi, uint8_t *records, int nv,
                                              const int *s_env, const size_t *s_rec)
{
    const int per = (int)((hi - lo) / sizeof(V));
    auto one = [&](int j, int c) {
        const uint32_t b = lo + (uint32_t)c * (uint32_t)sizeof(V);
        V *dev = reinterpret_cast<V *>(g.dev + (size_t)s_env[j] * g.elem + b);
        V *rec = reinterpret_cast<V *>(records + s_rec[j] + g.off + b);
        if (SAVE) {
            V v;
            if (b < g.elem) v = __ldg(dev);
            else memset(&v, 0, sizeof v);
            __stcs(rec, v);
        } else if (b < g.elem) {
            *dev = __ldcs(rec);
        }
    };
    if (per >= SF_SNAP_CTA) { /* large blocks: the CTA walks one arena at a time, fully coalesced */
#pragma unroll 4
        for (int j = 0; j < nv; ++j)
            for (int c = threadIdx.x; c < per; c += SF_SNAP_CTA) one(j, c);
    } else {
        for (int q = threadIdx.x; q < nv * per; q += SF_SNAP_CTA) one(q / per, q % per);
    }
}

/* SAVE: records[i] = arena ids[i] (ids NULL: arena i).  LOAD: arena ids[i] = records[rows[i]] (rows NULL:
   row i), unless sf_snap_check_kernel refused a referenced record. */
template <bool SAVE>
__global__ void __launch_bounds__(SF_SNAP_CTA)
sf_snap_kernel(const __grid_constant__ SfSnapLayout L, int64_t env_id_base, const int32_t *__restrict__ ids, int n,
               uint8_t *records, const int32_t *__restrict__ rows, const int *refused)
{
    __shared__ __align__(16) uint8_t stage[SF_SNAP_STAGE];
    __shared__ int s_env[SF_SNAP_TILE];
    __shared__ size_t s_rec[SF_SNAP_TILE]; /* byte offset of the entry's record */
    if (!SAVE && *reinterpret_cast<const volatile int *>(refused)) return;
    const long n_work = (long)((n + SF_SNAP_TILE - 1) / SF_SNAP_TILE) * L.n_item;
    for (long w = blockIdx.x; w < n_work; w += gridDim.x) {
        const int tile = (int)(w / L.n_item), item = (int)(w % L.n_item);
        const SfSnapItem it = L.item[item];
        const int nv = min(SF_SNAP_TILE, n - tile * SF_SNAP_TILE);
        __syncthreads(); /* the last turn is done with the stage and the entry table */
        if (threadIdx.x < nv) {
            const int i = tile * SF_SNAP_TILE + threadIdx.x;
            s_env[threadIdx.x] = ids ? ids[i] : i;
            s_rec[threadIdx.x] = (size_t)(SAVE || !rows ? i : rows[i]) * L.bytes;
        }
        __syncthreads();
        if (it.first >= L.n_soa) {
            const SfSnapSeg &g = L.seg[it.first];
            const uint32_t hi = it.hi == g.elem ? sf_snap_end(L, it.first) - g.off : it.hi; /* the last piece covers the padding */
            if (g.elem % 16 == 0) sf_snap_block<SAVE, uint4>(g, it.lo, hi, records, nv, s_env, s_rec);
            else sf_snap_block<SAVE, uint2>(g, it.lo, hi, records, nv, s_env, s_rec);
            continue;
        }
        const uint32_t lo = L.seg[it.first].off;
        const uint32_t P = sf_snap_end(L, it.last - 1) - lo, S = sf_snap_stride(P);
        const int chunks = (int)(P / 16);
        if (!SAVE) {
            for (int q = threadIdx.x; q < nv * chunks; q += SF_SNAP_CTA) {
                const int j = q / chunks, c = q - j * chunks;
                *reinterpret_cast<uint4 *>(stage + (size_t)j * S + 16 * c) =
                    __ldcs(reinterpret_cast<const uint4 *>(records + s_rec[j] + lo + 16 * c));
            }
            __syncthreads();
        }
        for (int s = it.first; s < it.last; ++s) {
            const SfSnapSeg &g = L.seg[s];
            uint8_t *st = stage + (g.off - lo);
            switch (g.elem) {
            case 1: sf_snap_soa<SAVE, uint8_t>(g, L.E, st, S, nv, s_env); break;
            case 2: sf_snap_soa<SAVE, uint16_t>(g, L.E, st, S, nv, s_env); break;
            case 4: sf_snap_soa<SAVE, uint32_t>(g, L.E, st, S, nv, s_env); break;
            default: sf_snap_soa<SAVE, unsigned long long>(g, L.E, st, S, nv, s_env); break;
            }
        }
        if (SAVE) {
            __syncthreads();
            for (int q = threadIdx.x; q < nv * chunks; q += SF_SNAP_CTA) {
                const int j = q / chunks, c = q - j * chunks;
                __stcs(reinterpret_cast<uint4 *>(records + s_rec[j] + lo + 16 * c),
                       *reinterpret_cast<const uint4 *>(stage + (size_t)j * S + 16 * c));
            }
            if (item == 0 && threadIdx.x < 4 * nv) { /* the header, 4 chunks per record */
                const int j = threadIdx.x >> 2, c = threadIdx.x & 3;
                const int64_t ge = env_id_base + s_env[j];
                __stcs(reinterpret_cast<uint4 *>(records + s_rec[j]) + c,
                       make_uint4(sf_snap_header_word(L, ge, 4 * c), sf_snap_header_word(L, ge, 4 * c + 1),
                                  sf_snap_header_word(L, ge, 4 * c + 2), sf_snap_header_word(L, ge, 4 * c + 3)));
            }
        }
    }
}

/* magic, version, size and fingerprint of every record a load references */
__global__ void sf_snap_check_kernel(const __grid_constant__ SfSnapLayout L, const uint8_t *records, const int32_t *rows,
                                     int n, int *refused)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t *w = reinterpret_cast<const uint32_t *>(records + (size_t)(rows ? rows[i] : i) * L.bytes);
    if (!sf_snap_compatible(w, L)) atomicOr(refused, 1);
}

/* after the copy: the pending stream of every arena that took a record of another global id */
__global__ void sf_snap_reseed_kernel(const SfDev d, const __grid_constant__ SfConst k, const uint8_t *records, uint32_t bytes,
                                      const int32_t *ids, const int32_t *rows, int n, const int *refused)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || *refused) return;
    SfTabs t;
    sf_global_tabs(d, t);
    const uint32_t *w = reinterpret_cast<const uint32_t *>(records + (size_t)(rows ? rows[i] : i) * bytes);
    sf_snap_reseed(d, k, t, ids ? ids[i] : i, sf_snap_global_id(w));
}

/* sf_list_finished / sf_reset_finished: a stable compaction of the arenas whose state is not SF_RUNNING.
 *
 * Tiles of SF_LIST_TILE consecutive arenas, one CTA each, four arenas per thread (one 16-byte load of their
 * header words).  sf_list_count_kernel writes the number of finished arenas of every tile; sf_list_scatter_kernel
 * adds up the counts of the tiles before its own, scans its tile and writes the ids, and its last CTA writes the
 * total.  An id's position is the number of finished arenas below it, so the list is ascending and the same on
 * every run (no atomics); the header words are read twice, the second time from L2 (512 KB at 131,072 arenas). */
#define SF_LIST_CTA 256
#define SF_LIST_TILE (4 * SF_LIST_CTA)
#define SF_FIN_CTA 32 /* sf_reset_finished_kernel: one warp per CTA, so that a short list spreads over the SMs */

/* bit j: arena tile * SF_LIST_TILE + 4 * thread + j is finished (E is a multiple of 32: the load stays in the array) */
__device__ __forceinline__ uint32_t sf_list_flags(const SfDev &d, int tile)
{
    const int base = tile * SF_LIST_TILE + 4 * (int)threadIdx.x;
    if (base >= d.n_envs) return 0u;
    const uint4 m = __ldg(reinterpret_cast<const uint4 *>(d.misc + base));
    uint32_t f = (sf_misc_finished(m.x) ? 1u : 0u) | (sf_misc_finished(m.y) ? 2u : 0u) | (sf_misc_finished(m.z) ? 4u : 0u) |
                 (sf_misc_finished(m.w) ? 8u : 0u);
    const int left = d.n_envs - base;
    return left >= 4 ? f : f & ((1u << left) - 1u);
}

/* sum of v over the CTA, in every thread */
__device__ __forceinline__ int sf_list_sum(int v, int *s_warp)
{
    v = (int)__reduce_add_sync(0xffffffffu, (unsigned)v);
    __syncthreads(); /* s_warp is free */
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
    __syncthreads();
    int sum = 0;
#pragma unroll
    for (int w = 0; w < SF_LIST_CTA / 32; ++w) sum += s_warp[w];
    return sum;
}

__global__ void __launch_bounds__(SF_LIST_CTA) sf_list_count_kernel(const SfDev d, int32_t *__restrict__ tile_n)
{
    __shared__ int s_warp[SF_LIST_CTA / 32];
    const int n = sf_list_sum(__popc(sf_list_flags(d, blockIdx.x)), s_warp);
    if (threadIdx.x == 0) tile_n[blockIdx.x] = n;
}

__global__ void __launch_bounds__(SF_LIST_CTA)
sf_list_scatter_kernel(const SfDev d, const int32_t *__restrict__ tile_n, int32_t *__restrict__ ids, int32_t *__restrict__ count)
{
    __shared__ int s_warp[SF_LIST_CTA / 32];
    int before = 0;
    for (int i = threadIdx.x; i < (int)blockIdx.x; i += SF_LIST_CTA) before += tile_n[i];
    const int base = sf_list_sum(before, s_warp); /* finished arenas in the tiles below this one */
    const uint32_t f = sf_list_flags(d, blockIdx.x);
    const int c = __popc(f), lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = c; /* inclusive scan over the warp */
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    __syncthreads(); /* every thread has read s_warp */
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int pos = base + incl - c, total = base;
#pragma unroll
    for (int w = 0; w < SF_LIST_CTA / 32; ++w) {
        pos += w < warp ? s_warp[w] : 0;
        total += s_warp[w];
    }
    const int env = blockIdx.x * SF_LIST_TILE + 4 * (int)threadIdx.x;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if ((f >> j) & 1u) ids[pos++] = env + j;
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) *count = total;
}

/* sf_reset_finished: the listed arenas (the count is read here, not on the host), lpw consecutive entries of the
 * list per one-warp CTA.  As in sf_launch_step, lpw is the smallest power of two that still fits the list into one
 * pass of the grid: a reset is a long serial chain per lane (the 19,968-byte overlay cleared with 16-byte stores,
 * the rest of the stream warm-up, the digit split of the next seeds), so the few dozen arenas that finish in a
 * typical step run one per SM, and a long list fills whole warps instead of looping. */
__global__ void __launch_bounds__(SF_FIN_CTA, 1)
sf_reset_finished_kernel(const SfDev d, const __grid_constant__ SfConst k, const int32_t *__restrict__ ids,
                         const int32_t *__restrict__ count)
{
    const int n = *count;
    int lpw = 1;
    while (lpw < SF_FIN_CTA && (n + lpw - 1) / lpw > (int)gridDim.x) lpw *= 2;
    SfTabs t;
    sf_global_tabs(d, t);
    for (int c = blockIdx.x; c * lpw < n; c += gridDim.x) {
        const int i = c * lpw + (int)threadIdx.x;
        if ((int)threadIdx.x < lpw && i < n) sf_reset_finished_body(d, k, t, ids[i]);
    }
}

/* ====================================================================== host side */

struct sf_handle {
    SfDev d;
    SfConst k;
    sfhost::Tables tabs;
    void *arena = nullptr;       /* one device allocation holding every array */
    size_t arena_bytes = 0;
    uint8_t *d_actions = nullptr; /* [n_envs][n_agents] staging for sf_step_host / synthetic streams */
    uint8_t *d_table = nullptr;   /* action alphabet of sf_synth_actions */
    int32_t *d_export = nullptr;
    long long *d_export_n = nullptr;
    int32_t *d_ids = nullptr;
    int64_t *d_tb = nullptr, *d_serial = nullptr;
    int32_t *d_rows = nullptr;   /* sf_load: record row of each entry */
    int *d_refused = nullptr;    /* sf_load: set when a referenced record is not one of this configuration */
    int32_t *d_fin_ids = nullptr; /* sf_reset_finished: the finished arenas, ascending ... */
    int32_t *d_fin_n = nullptr;   /* ... and their number */
    int32_t *d_tile_n = nullptr;  /* sf_list_finished / sf_reset_finished: finished arenas per tile of SF_LIST_TILE */
    SfSnapLayout snap;           /* the record layout of sf_save / sf_load (sf_snapshot.cuh) */
    int device = 0, n_sm = 0;
    bool between_halves = false; /* sf_step_a has run, sf_step_b has not: the P2 observation point */
    int lanes_per_warp = 0;      /* 0 = chosen from the batch size; SF_LANES_PER_WARP overrides (measurements) */
    int obs_run = 0;             /* consecutive observations a CTA writes before it moves on; 0 = chosen from the
                                    batch size, SF_OBS_RUN overrides (measurements) */
    int obs_rows = SF_OBS_CACHE; /* table rows for dynamic cells; SF_OBS_TABLE_ROWS lowers it (tests of the path beyond the table) */
    long long launches = 0;
    std::string err;
};

static thread_local std::string g_create_err;

static int sf_fail(sf_handle *h, int code, const std::string &msg)
{
    if (h) h->err = msg;
    else g_create_err = msg;
    return code;
}

#define SF_CUDA(h, call)                                                                         \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return sf_fail(h, e_ == cudaErrorMemoryAllocation ? SF_ERR_NOMEM : SF_ERR_CUDA,      \
                           std::string(#call) + ": " + cudaGetErrorString(e_));                  \
    } while (0)

/* A handle lives on the device that was current in sf_create; every entry point runs there,
 * whatever device the calling thread has current, and puts the caller's device back. */
struct SfDeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit SfDeviceGuard(const sf_handle *h);
    ~SfDeviceGuard()
    {
        if (switched) cudaSetDevice(prev);
    }
};

static int sf_require_device(sf_handle *h)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return sf_fail(h, SF_ERR_NO_DEVICE, "no usable CUDA device: strikeforce_b200 has no CPU path");
    }
    return SF_OK;
}

SfDeviceGuard::SfDeviceGuard(const sf_handle *h)
{
    if (h && cudaGetDevice(&prev) == cudaSuccess && prev != h->device) switched = cudaSetDevice(h->device) == cudaSuccess;
}

namespace {
struct Carver {
    size_t off = 0;
    uint8_t *base = nullptr;
    template <class T> void take(T *&p, size_t n)
    {
        off = (off + 255) & ~(size_t)255;
        if (base) p = reinterpret_cast<T *>(base + off);
        off += n * sizeof(T);
    }
};

void carve(Carver &c, sf_handle &h)
{
    SfDev &d = h.d;
    const SfConst &k = h.k;
    size_t E = (size_t)d.E;
    c.take(d.frame, E), c.take(d.kills, E), c.take(d.tkills, E), c.take(d.loot, E), c.take(d.chest, E);
    c.take(d.misc, E), c.take(d.steps, E), c.take(d.episode, E), c.take(d.ntemp, E);
    c.take(d.mh, E), c.take(d.mz, 2 * E), c.take(d.mb, 2 * E), c.take(d.mp, 2 * E);
    c.take(d.rng_log, 9 * E), c.take(d.rng_cst, 36 * E), c.take(d.rng_w, E), c.take(d.jomle, E);
    c.take(d.pend_log, 9 * E), c.take(d.pend_n, E);
    size_t H = (size_t)k.cap_h * E, Z = (size_t)k.cap_z * E, B = (size_t)k.cap_b * E, T = (size_t)d.cap_t * E;
    c.take(d.h_pw, H), c.take(d.h_sel, H), c.take(d.h_bp, H), c.take(d.h_hp, H), c.take(d.h_mind, H);
    c.take(d.h_stam, H), c.take(d.h_kills, H), c.take(d.h_dmg, H), c.take(d.h_eff, H), c.take(d.h_cons, H);
    c.take(d.h_thr, H), c.take(d.h_cmd, H);
    c.take(d.z_pos, Z), c.take(d.z_hp, Z), c.take(d.z_mind, Z);
    c.take(d.b_pw, B), c.take(d.b_meta, B), c.take(d.b_dmg, B), c.take(d.b_eff, B);
    c.take(d.t_cell, T), c.take(d.t_dmg, T), c.take(d.t_pidx, T);
    c.take(d.p_cell, (size_t)k.cap_p * E);
    c.take(d.grid, E * SF_GRID_STRIDE);
    c.take(d.out, E);
    c.take(d.stats, (size_t)SF_STAT_COUNT);
    uint8_t *smap = nullptr;
    uint16_t *exp_tab = nullptr, *log_tab = nullptr;
    float *lut = nullptr;
    c.take(smap, (size_t)SF_SMEM_MAP), c.take(exp_tab, (size_t)65536), c.take(log_tab, (size_t)65536);
    c.take(lut, (size_t)SF_POW_LUT_LEN);
    d.smap = smap, d.exp_tab = exp_tab, d.log_tab = log_tab, d.pow_lut = lut, d.pow_lut_len = SF_POW_LUT_LEN;
    c.take(h.d_actions, E * (size_t)k.n_agents);
    c.take(h.d_table, (size_t)256);
    c.take(h.d_export, (size_t)SF_EXPORT_CAP);
    c.take(h.d_export_n, (size_t)1);
    c.take(h.d_ids, E), c.take(h.d_tb, E), c.take(h.d_serial, E);
    c.take(h.d_rows, E), c.take(h.d_refused, (size_t)1);
    c.take(h.d_fin_ids, E), c.take(h.d_fin_n, (size_t)1), c.take(h.d_tile_n, (E + SF_LIST_TILE - 1) / SF_LIST_TILE);
}
} // namespace

static int sf_launch_reset(sf_handle *h, const int32_t *d_ids, int n, const int64_t *d_tb, const int64_t *d_serial,
                           cudaStream_t s)
{
    int grid = (n + SF_CTA - 1) / SF_CTA;
    if (grid > h->n_sm) grid = h->n_sm;
    sf_reset_kernel<<<grid, SF_CTA, SF_SMEM_BYTES, s>>>(h->d, h->k, d_ids, n, d_tb, d_serial);
    h->launches += 1;
    SF_CUDA(h, cudaGetLastError());
    return SF_OK;
}

extern "C" {

int32_t sf_abi_version(void) { return SF_ABI_VERSION; }

const char *sf_last_error(const sf_handle *h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int sf_create(const sf_config *cfg, sf_handle **out)
{
    if (!cfg || !out) return sf_fail(nullptr, SF_ERR_ARG, "sf_create: null argument");
    *out = nullptr;
    int rc = sf_require_device(nullptr);
    if (rc) return rc;
    sf_handle *h = new (std::nothrow) sf_handle();
    if (!h) return sf_fail(nullptr, SF_ERR_NOMEM, "host allocation failed");
    std::string err = sfhost::build_const(*cfg, h->k, h->tabs);
    if (!err.empty()) {
        delete h;
        return sf_fail(nullptr, SF_ERR_ARG, "sf_create: " + err);
    }
    memset(&h->d, 0, sizeof h->d);
    h->d.n_envs = cfg->n_envs;
    h->d.E = (cfg->n_envs + 31) / 32 * 32;
    h->d.cap_t = (h->k.cap_t + 7) / 8 * 8;
    if (const char *v = getenv("SF_OBS_RUN")) {
        int n = atoi(v);
        if (n >= 1 && n <= 4096) h->obs_run = n;
    }
    if (const char *v = getenv("SF_OBS_TABLE_ROWS")) {
        int n = atoi(v);
        if (n >= 0 && n < SF_OBS_CACHE) h->obs_rows = n;
    }
    if (const char *v = getenv("SF_LANES_PER_WARP")) {
        const int n = atoi(v);
        if (n == 1 || n == 2 || n == 4 || n == 8 || n == 16 || n == 32) h->lanes_per_warp = n;
    }
    cudaError_t ce = cudaGetDevice(&h->device);
    if (ce == cudaSuccess) ce = cudaDeviceGetAttribute(&h->n_sm, cudaDevAttrMultiProcessorCount, h->device);
    int smem_optin = 0;
    if (ce == cudaSuccess) ce = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device);
    if (ce != cudaSuccess) {
        std::string m = std::string("device query: ") + cudaGetErrorString(ce);
        delete h;
        return sf_fail(nullptr, SF_ERR_CUDA, m);
    }
    if (smem_optin < SF_SMEM_BYTES) {
        delete h;
        return sf_fail(nullptr, SF_ERR_UNSUPPORTED, "device offers too little shared memory per block (need 161,536 B)");
    }
    Carver sizer;
    carve(sizer, *h);
    h->arena_bytes = sizer.off + 256;
    ce = cudaMalloc(&h->arena, h->arena_bytes);
    if (ce != cudaSuccess) {
        std::string m = "cudaMalloc of " + std::to_string(h->arena_bytes) + " bytes: " + cudaGetErrorString(ce);
        delete h;
        return sf_fail(nullptr, SF_ERR_NOMEM, m);
    }
    Carver placer;
    placer.base = static_cast<uint8_t *>(h->arena);
    carve(placer, *h);
    sf_snap_layout(h->d, h->k, sf_snap_fingerprint(h->k, h->tabs.smap.data(), h->d.cap_t), h->snap);
#define SF_CREATE_CUDA(call)                                                        \
    do {                                                                            \
        cudaError_t e_ = (call);                                                    \
        if (e_ != cudaSuccess) {                                                    \
            std::string m_ = std::string(#call) + ": " + cudaGetErrorString(e_);    \
            cudaFree(h->arena);                                                     \
            delete h;                                                               \
            return sf_fail(nullptr, SF_ERR_CUDA, m_);                               \
        }                                                                           \
    } while (0)
    SF_CREATE_CUDA(cudaMemset(h->arena, 0, h->arena_bytes));
    sfhost::build_pow_lut(h->tabs, SF_POW_LUT_LEN);
    h->tabs.smap.resize(SF_SMEM_MAP, 0);
    SF_CREATE_CUDA(cudaMemcpy(const_cast<uint8_t *>(h->d.smap), h->tabs.smap.data(), SF_SMEM_MAP, cudaMemcpyHostToDevice));
    SF_CREATE_CUDA(cudaMemcpy(const_cast<uint16_t *>(h->d.exp_tab), h->tabs.exp_tab.data(), 65536 * 2, cudaMemcpyHostToDevice));
    SF_CREATE_CUDA(cudaMemcpy(const_cast<uint16_t *>(h->d.log_tab), h->tabs.log_tab.data(), 65536 * 2, cudaMemcpyHostToDevice));
    SF_CREATE_CUDA(cudaMemcpy(const_cast<float *>(h->d.pow_lut), h->tabs.pow_lut.data(), (size_t)SF_POW_LUT_LEN * 4,
                              cudaMemcpyHostToDevice));
    SF_CREATE_CUDA(cudaFuncSetAttribute(sf_step_kernel<SF_HALF_BOTH>, cudaFuncAttributeMaxDynamicSharedMemorySize, SF_SMEM_BYTES));
    SF_CREATE_CUDA(cudaFuncSetAttribute(sf_step_kernel<SF_HALF_A>, cudaFuncAttributeMaxDynamicSharedMemorySize, SF_SMEM_BYTES));
    SF_CREATE_CUDA(cudaFuncSetAttribute(sf_step_kernel<SF_HALF_B>, cudaFuncAttributeMaxDynamicSharedMemorySize, SF_SMEM_BYTES));
    SF_CREATE_CUDA(cudaFuncSetAttribute(sf_reset_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SF_SMEM_BYTES));
    SF_CREATE_CUDA(cudaFuncSetAttribute(sf_rng_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SF_SMEM_BYTES));
    SF_CREATE_CUDA(cudaFuncSetAttribute(sf_observe_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SF_OBS_SMEM));
    SF_CREATE_CUDA(cudaFuncSetAttribute(sf_observe_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SF_OBS_SMEM));
    SF_CREATE_CUDA(cudaFuncSetAttribute(sf_observe_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SF_OBS_SMEM));
    SF_CREATE_CUDA(cudaFuncSetAttribute(sf_observe_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SF_OBS_SMEM));
    rc = sf_launch_reset(h, nullptr, h->d.n_envs, nullptr, nullptr, 0);
    if (rc == SF_OK) {
        cudaError_t e_ = cudaDeviceSynchronize();
        if (e_ != cudaSuccess) rc = sf_fail(nullptr, SF_ERR_CUDA, std::string("initial reset: ") + cudaGetErrorString(e_));
    } else
        g_create_err = h->err;
    if (rc != SF_OK) {
        cudaFree(h->arena);
        delete h;
        return rc;
    }
#undef SF_CREATE_CUDA
    *out = h;
    return SF_OK;
}

int sf_destroy(sf_handle *h)
{
    if (!h) return SF_ERR_ARG;
    {
        SfDeviceGuard guard(h);
        cudaDeviceSynchronize();
        cudaFree(h->arena);
    }
    delete h;
    return SF_OK;
}

int sf_reset(sf_handle *h, const int32_t *env_ids, int32_t n, const int64_t *tb, const int64_t *serial, void *stream)
{
    if (!h) return SF_ERR_ARG;
    SfDeviceGuard guard(h);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!env_ids) n = h->d.n_envs;
    if (n <= 0 || n > h->d.n_envs) return sf_fail(h, SF_ERR_ARG, "sf_reset: bad arena count");
    if ((tb == nullptr) != (serial == nullptr)) return sf_fail(h, SF_ERR_ARG, "sf_reset: tb and serial go together");
    if (env_ids) {
        for (int i = 0; i < n; ++i)
            if (env_ids[i] < 0 || env_ids[i] >= h->d.n_envs) return sf_fail(h, SF_ERR_ARG, "sf_reset: arena id out of range");
        SF_CUDA(h, cudaMemcpyAsync(h->d_ids, env_ids, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    }
    if (tb) {
        for (int i = 0; i < n; ++i)
            if (tb[i] < 0 || serial[i] < 0) return sf_fail(h, SF_ERR_ARG, "sf_reset: seeds must be non-negative");
        SF_CUDA(h, cudaMemcpyAsync(h->d_tb, tb, (size_t)n * 8, cudaMemcpyHostToDevice, s));
        SF_CUDA(h, cudaMemcpyAsync(h->d_serial, serial, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    }
    int rc = sf_launch_reset(h, env_ids ? h->d_ids : nullptr, n, tb ? h->d_tb : nullptr, tb ? h->d_serial : nullptr, s);
    if (rc) return rc;
    h->between_halves = false;
    /* the staging buffers are reused by the next call */
    SF_CUDA(h, cudaStreamSynchronize(s));
    return SF_OK;
}

static int sf_launch_step(sf_handle *h, int half, const uint8_t *d_actions, cudaStream_t s)
{
    SfDeviceGuard guard(h);
    if ((half == SF_HALF_B) != h->between_halves)
        return sf_fail(h, SF_ERR_ARG, half == SF_HALF_B ? "sf_step_b: no sf_step_a before it"
                                                        : "sf_step / sf_step_a: the step opened by sf_step_a is still waiting for sf_step_b");
    h->between_halves = half == SF_HALF_A;
    /* arenas per warp: as few as still fit the batch into one wave of warps (see sf_step_kernel) */
    const int slots = h->n_sm * (SF_CTA / 32);
    int lpw = h->lanes_per_warp;
    if (lpw <= 0) {
        lpw = 1;
        while (lpw < 32 && (h->d.n_envs + lpw - 1) / lpw > slots) lpw *= 2;
    }
    const int nchunks = (h->d.n_envs + lpw - 1) / lpw;
    int grid = nchunks < h->n_sm ? nchunks : h->n_sm; /* one persistent CTA per SM; warps take chunks round-robin over the CTAs */
    if (half == SF_HALF_BOTH) sf_step_kernel<SF_HALF_BOTH><<<grid, SF_CTA, SF_SMEM_BYTES, s>>>(h->d, h->k, d_actions, lpw);
    else if (half == SF_HALF_A) sf_step_kernel<SF_HALF_A><<<grid, SF_CTA, SF_SMEM_BYTES, s>>>(h->d, h->k, nullptr, lpw);
    else sf_step_kernel<SF_HALF_B><<<grid, SF_CTA, SF_SMEM_BYTES, s>>>(h->d, h->k, d_actions, lpw);
    h->launches += 1;
    SF_CUDA(h, cudaGetLastError());
    return SF_OK;
}

int sf_step(sf_handle *h, const uint8_t *actions, void *stream)
{
    if (!h || !actions) return h ? sf_fail(h, SF_ERR_ARG, "sf_step: null actions") : SF_ERR_ARG;
    return sf_launch_step(h, SF_HALF_BOTH, actions, static_cast<cudaStream_t>(stream));
}

int sf_step_a(sf_handle *h, void *stream)
{
    if (!h) return SF_ERR_ARG;
    return sf_launch_step(h, SF_HALF_A, nullptr, static_cast<cudaStream_t>(stream));
}

int sf_step_b(sf_handle *h, const uint8_t *actions, void *stream)
{
    if (!h || !actions) return h ? sf_fail(h, SF_ERR_ARG, "sf_step_b: null actions") : SF_ERR_ARG;
    return sf_launch_step(h, SF_HALF_B, actions, static_cast<cudaStream_t>(stream));
}

int sf_step_host(sf_handle *h, const uint8_t *actions_host, sf_step_out *out_host, void *stream)
{
    if (!h || !actions_host || !out_host) return h ? sf_fail(h, SF_ERR_ARG, "sf_step_host: null argument") : SF_ERR_ARG;
    SfDeviceGuard guard(h);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    size_t na = (size_t)h->d.n_envs * (size_t)h->k.n_agents;
    /* page-locked buffers (cudaHostAlloc / cudaHostRegister) are used in place: the kernel reads each
       arena's commands from the action buffer when human_action needs them and stores each arena's
       result as its warp finishes, so both transfers overlap the step; pageable ones are copied */
    auto device_view = [](const void *p) -> void * {
        cudaPointerAttributes pa;
        if (cudaPointerGetAttributes(&pa, p) == cudaSuccess && pa.type == cudaMemoryTypeHost && pa.devicePointer)
            return pa.devicePointer;
        cudaGetLastError();
        return nullptr;
    };
    const uint8_t *actions = static_cast<const uint8_t *>(device_view(actions_host));
    if (!actions) {
        SF_CUDA(h, cudaMemcpyAsync(h->d_actions, actions_host, na, cudaMemcpyHostToDevice, s));
        actions = h->d_actions;
    }
    sf_step_out *mirror = static_cast<sf_step_out *>(device_view(out_host));
    h->d.out_mirror = mirror;
    int rc = sf_launch_step(h, SF_HALF_BOTH, actions, s);
    h->d.out_mirror = nullptr;
    if (rc) return rc;
    if (!mirror)
        SF_CUDA(h, cudaMemcpyAsync(out_host, h->d.out, (size_t)h->d.n_envs * sizeof(sf_step_out), cudaMemcpyDeviceToHost, s));
    SF_CUDA(h, cudaStreamSynchronize(s));
    return SF_OK;
}

int sf_synth_actions(sf_handle *h, uint8_t *actions, uint64_t t, const char *table, int32_t table_len, void *stream)
{
    if (!h || !actions || !table || table_len <= 0 || table_len > 256)
        return h ? sf_fail(h, SF_ERR_ARG, "sf_synth_actions: bad argument") : SF_ERR_ARG;
    SfDeviceGuard guard(h);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    SF_CUDA(h, cudaMemcpyAsync(h->d_table, table, (size_t)table_len, cudaMemcpyHostToDevice, s));
    int n = h->d.n_envs * h->k.n_agents;
    sf_synth_actions_kernel<<<(n + 255) / 256, 256, 0, s>>>(actions, h->d.n_envs, h->k.n_agents, h->k.env_id_base, t,
                                                            h->d_table, table_len);
    h->launches += 1;
    SF_CUDA(h, cudaGetLastError());
    return SF_OK;
}

/* the checks and the launch sf_observe and sf_observe_list share: n_rows rows of observations (arenas 0..n_rows-1,
   or env_ids[0..n_rows) with *count of them written) */
static int sf_launch_observe(sf_handle *h, const char *fn, float *obs, int32_t phase, uint32_t agent_mask, int n_rows,
                             const int32_t *env_ids, const int32_t *count, cudaStream_t s)
{
    const bool nhwc = (phase & SF_OBS_NHWC) != 0;
    phase &= ~SF_OBS_NHWC;
    if (phase != SF_OBS_P1 && phase != SF_OBS_P2) return sf_fail(h, SF_ERR_ARG, std::string(fn) + ": phase must be SF_OBS_P1 or SF_OBS_P2");
    /* the kernel describes the arena as it stands; the phase says WHERE in the step the caller claims
       to be, and a claim that does not match the handle is an error: P2 is the point between
       sf_step_a and sf_step_b (get_command inside human_action), P1 the loop top */
    if ((phase == SF_OBS_P2) != h->between_halves)
        return sf_fail(h, SF_ERR_ARG, std::string(fn) + (phase == SF_OBS_P2 ? ": SF_OBS_P2 is the point between sf_step_a and sf_step_b"
                                                                             : ": between sf_step_a and sf_step_b the observation point is SF_OBS_P2"));
    SfDeviceGuard guard(h);
    int nsel = __builtin_popcount(agent_mask);
    if (nsel == 0) return sf_fail(h, SF_ERR_ARG, std::string(fn) + ": empty agent mask");
    if (reinterpret_cast<uintptr_t>(obs) & 15u) return sf_fail(h, SF_ERR_ARG, std::string(fn) + ": obs must be 16-byte aligned");
    int n_items = n_rows * nsel;
    /* a CTA writes runs of consecutive observations: HBM takes 1,184 store streams that each run on for
       megabytes better than a front of 123 KB pieces (profiles/r02_obs_run.txt: 73 -> 80% of the peak); the
       longest run of up to 16 that still leaves every CTA four turns */
    const int ctas = SF_OBS_CTAS_PER_SM * h->n_sm;
    int run_len = h->obs_run;
    if (run_len == 0)
        for (run_len = 16; run_len > 1 && n_items / run_len < 4 * ctas; run_len >>= 1) {}
    int runs = (n_items + run_len - 1) / run_len;
    int grid = runs < ctas ? runs : ctas;
#define SF_OBS_LAUNCH(NHWC, LIST)                                                                                          \
    sf_observe_kernel<NHWC, LIST><<<grid, SF_OBS_CTA, SF_OBS_SMEM, s>>>(h->d, h->k, obs, agent_mask, nsel, n_items, h->obs_rows, \
                                                                        run_len, env_ids, count)
    if (env_ids) {
        if (nhwc) SF_OBS_LAUNCH(true, true);
        else SF_OBS_LAUNCH(false, true);
    } else {
        if (nhwc) SF_OBS_LAUNCH(true, false);
        else SF_OBS_LAUNCH(false, false);
    }
#undef SF_OBS_LAUNCH
    h->launches += 1;
    SF_CUDA(h, cudaGetLastError());
    return SF_OK;
}

int sf_observe(sf_handle *h, float *obs, int32_t phase, uint32_t agent_mask, void *stream)
{
    if (!h || !obs) return h ? sf_fail(h, SF_ERR_ARG, "sf_observe: null buffer") : SF_ERR_ARG;
    return sf_launch_observe(h, "sf_observe", obs, phase, agent_mask, h->d.n_envs, nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

int sf_observe_list(sf_handle *h, float *obs, int32_t phase, uint32_t agent_mask, const int32_t *env_ids, const int32_t *count,
                    int32_t n_max, void *stream)
{
    if (!h || !obs || !env_ids) return h ? sf_fail(h, SF_ERR_ARG, "sf_observe_list: null buffer") : SF_ERR_ARG;
    if (n_max < 1 || n_max > h->d.n_envs) return sf_fail(h, SF_ERR_ARG, "sf_observe_list: n_max must be in [1, n_envs]");
    if ((reinterpret_cast<uintptr_t>(env_ids) | reinterpret_cast<uintptr_t>(count)) & 3u)
        return sf_fail(h, SF_ERR_ARG, "sf_observe_list: env_ids and count must be 4-byte aligned");
    return sf_launch_observe(h, "sf_observe_list", obs, phase, agent_mask, n_max, env_ids, count, static_cast<cudaStream_t>(stream));
}

/* the two launches of the compaction (see sf_list_count_kernel) */
static int sf_launch_list(sf_handle *h, int32_t *ids, int32_t *count, cudaStream_t s)
{
    const int tiles = (h->d.n_envs + SF_LIST_TILE - 1) / SF_LIST_TILE;
    sf_list_count_kernel<<<tiles, SF_LIST_CTA, 0, s>>>(h->d, h->d_tile_n);
    sf_list_scatter_kernel<<<tiles, SF_LIST_CTA, 0, s>>>(h->d, h->d_tile_n, ids, count);
    h->launches += 2;
    SF_CUDA(h, cudaGetLastError());
    return SF_OK;
}

int sf_list_finished(sf_handle *h, int32_t *env_ids, int32_t *count, void *stream)
{
    if (!h || !env_ids || !count) return h ? sf_fail(h, SF_ERR_ARG, "sf_list_finished: null buffer") : SF_ERR_ARG;
    if ((reinterpret_cast<uintptr_t>(env_ids) | reinterpret_cast<uintptr_t>(count)) & 3u)
        return sf_fail(h, SF_ERR_ARG, "sf_list_finished: env_ids and count must be 4-byte aligned");
    SfDeviceGuard guard(h);
    return sf_launch_list(h, env_ids, count, static_cast<cudaStream_t>(stream));
}

int sf_reset_finished(sf_handle *h, void *stream)
{
    if (!h) return SF_ERR_ARG;
    if (h->between_halves) return sf_fail(h, SF_ERR_ARG, "sf_reset_finished: the step opened by sf_step_a is still waiting for sf_step_b");
    SfDeviceGuard guard(h);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int rc = sf_launch_list(h, h->d_fin_ids, h->d_fin_n, s);
    if (rc) return rc;
    /* one-warp CTAs, four per SM (see sf_reset_finished_kernel for how the list is spread over them) */
    int grid = (h->d.n_envs + SF_FIN_CTA - 1) / SF_FIN_CTA;
    if (grid > 4 * h->n_sm) grid = 4 * h->n_sm;
    sf_reset_finished_kernel<<<grid, SF_FIN_CTA, 0, s>>>(h->d, h->k, h->d_fin_ids, h->d_fin_n);
    h->launches += 1;
    SF_CUDA(h, cudaGetLastError());
    return SF_OK;
}

int sf_get(sf_handle *h, int32_t field, void *dev_out, void *stream)
{
    if (!h || !dev_out) return h ? sf_fail(h, SF_ERR_ARG, "sf_get: null buffer") : SF_ERR_ARG;
    SfDeviceGuard guard(h);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int n = h->d.n_envs, grid = (n + 127) / 128;
    switch (field) {
    case SF_FIELD_STEP_OUT:
        SF_CUDA(h, cudaMemcpyAsync(dev_out, h->d.out, (size_t)n * sizeof(sf_step_out), cudaMemcpyDeviceToDevice, s));
        return SF_OK;
    case SF_FIELD_STATS:
        SF_CUDA(h, cudaMemcpyAsync(dev_out, h->d.stats, SF_STAT_COUNT * 8, cudaMemcpyDeviceToDevice, s));
        return SF_OK;
    case SF_FIELD_STATE_HASH:
        sf_hash_kernel<<<grid, 128, 0, s>>>(h->d, h->k, static_cast<uint64_t *>(dev_out));
        break;
    case SF_FIELD_COUNTERS:
        sf_counters_kernel<<<grid, 128, 0, s>>>(h->d, h->k, static_cast<int32_t *>(dev_out));
        break;
    case SF_FIELD_POPULATION:
        sf_population_kernel<<<grid, 128, 0, s>>>(h->d, h->k, static_cast<int32_t *>(dev_out));
        break;
    default:
        return sf_fail(h, SF_ERR_ARG, "sf_get: unknown field");
    }
    h->launches += 1;
    SF_CUDA(h, cudaGetLastError());
    return SF_OK;
}

int sf_export_env(sf_handle *h, int32_t env, int32_t *host_buf, int64_t *n_inout)
{
    if (!h || !host_buf || !n_inout) return h ? sf_fail(h, SF_ERR_ARG, "sf_export_env: null argument") : SF_ERR_ARG;
    if (env < 0 || env >= h->d.n_envs) return sf_fail(h, SF_ERR_ARG, "sf_export_env: arena id out of range");
    SfDeviceGuard guard(h);
    SF_CUDA(h, cudaDeviceSynchronize());
    sf_export_kernel<<<1, 1>>>(h->d, h->k, env, h->d_export, (long)SF_EXPORT_CAP, h->d_export_n);
    h->launches += 1;
    SF_CUDA(h, cudaGetLastError());
    long long n = 0;
    SF_CUDA(h, cudaMemcpy(&n, h->d_export_n, sizeof n, cudaMemcpyDeviceToHost));
    if (n < 0 || n > *n_inout) return sf_fail(h, SF_ERR_ARG, "sf_export_env: buffer too small");
    SF_CUDA(h, cudaMemcpy(host_buf, h->d_export, (size_t)n * 4, cudaMemcpyDeviceToHost));
    *n_inout = n;
    return SF_OK;
}

int sf_rng_stream(sf_handle *h, const int64_t *tb, const int64_t *serial, int32_t n_streams, int32_t n_draws,
                  int32_t *out_host)
{
    if (!h || !tb || !serial || !out_host || n_streams <= 0 || n_draws <= 0)
        return h ? sf_fail(h, SF_ERR_ARG, "sf_rng_stream: bad argument") : SF_ERR_ARG;
    for (int32_t i = 0; i < n_streams; ++i)
        if (tb[i] < 0 || serial[i] < 0) return sf_fail(h, SF_ERR_ARG, "sf_rng_stream: seeds must be non-negative");
    SfDeviceGuard guard(h);
    /* one allocation for the three buffers, released on every path */
    const size_t n_out = (size_t)n_streams * (size_t)n_draws, seeds = (size_t)n_streams * 8;
    struct Scratch {
        void *p = nullptr;
        ~Scratch() { cudaFree(p); }
    } scratch;
    SF_CUDA(h, cudaMalloc(&scratch.p, 2 * seeds + n_out * 4));
    int64_t *d_tb = static_cast<int64_t *>(scratch.p), *d_serial = d_tb + n_streams;
    int32_t *d_out = reinterpret_cast<int32_t *>(d_serial + n_streams);
    SF_CUDA(h, cudaMemcpy(d_tb, tb, seeds, cudaMemcpyHostToDevice));
    SF_CUDA(h, cudaMemcpy(d_serial, serial, seeds, cudaMemcpyHostToDevice));
    int grid = (n_streams + SF_CTA - 1) / SF_CTA;
    if (grid > h->n_sm) grid = h->n_sm;
    sf_rng_kernel<<<grid, SF_CTA, SF_SMEM_BYTES>>>(h->d, d_tb, d_serial, n_streams, n_draws, d_out);
    h->launches += 1;
    SF_CUDA(h, cudaGetLastError());
    SF_CUDA(h, cudaMemcpy(out_host, d_out, n_out * 4, cudaMemcpyDeviceToHost));
    return SF_OK;
}

int64_t sf_snapshot_bytes(const sf_handle *h) { return h ? (int64_t)h->snap.bytes : 0; }

/* the checks sf_save and sf_load share; stages the arena ids in d_ids */
static int sf_snap_args(sf_handle *h, const char *fn, const int32_t *env_ids, int32_t &n, const void *records,
                        bool distinct, cudaStream_t s)
{
    if (!records) return sf_fail(h, SF_ERR_ARG, std::string(fn) + ": null record buffer");
    if (h->between_halves) return sf_fail(h, SF_ERR_ARG, std::string(fn) + ": the step opened by sf_step_a is still waiting for sf_step_b");
    if (reinterpret_cast<uintptr_t>(records) & 15u) return sf_fail(h, SF_ERR_ARG, std::string(fn) + ": records must be 16-byte aligned");
    if (!env_ids) n = h->d.n_envs;
    if (n <= 0 || n > h->d.n_envs) return sf_fail(h, SF_ERR_ARG, std::string(fn) + ": bad arena count");
    if (env_ids) {
        std::vector<uint8_t> seen(distinct ? (size_t)h->d.n_envs : 0, 0);
        for (int i = 0; i < n; ++i) {
            if (env_ids[i] < 0 || env_ids[i] >= h->d.n_envs) return sf_fail(h, SF_ERR_ARG, std::string(fn) + ": arena id out of range");
            if (distinct && seen[env_ids[i]]++) return sf_fail(h, SF_ERR_ARG, std::string(fn) + ": duplicate destination arena");
        }
        SF_CUDA(h, cudaMemcpyAsync(h->d_ids, env_ids, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    }
    return SF_OK;
}

static int sf_snap_grid(const sf_handle *h, int n)
{
    const long work = (long)((n + SF_SNAP_TILE - 1) / SF_SNAP_TILE) * h->snap.n_item;
    const long cap = (long)h->n_sm * SF_SNAP_CTAS_PER_SM;
    return (int)(work < cap ? work : cap);
}

int sf_save(sf_handle *h, const int32_t *env_ids, int32_t n, void *records, void *stream)
{
    if (!h) return SF_ERR_ARG;
    SfDeviceGuard guard(h);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int rc = sf_snap_args(h, "sf_save", env_ids, n, records, false, s);
    if (rc) return rc;
    sf_snap_kernel<true><<<sf_snap_grid(h, n), SF_SNAP_CTA, 0, s>>>(h->snap, h->k.env_id_base, env_ids ? h->d_ids : nullptr, n,
                                                                   static_cast<uint8_t *>(records), nullptr, nullptr);
    h->launches += 1;
    SF_CUDA(h, cudaGetLastError());
    SF_CUDA(h, cudaStreamSynchronize(s)); /* the staging buffers are reused by the next call */
    return SF_OK;
}

int sf_load(sf_handle *h, const int32_t *env_ids, int32_t n, const void *records, int32_t n_records, const int32_t *rows,
            void *stream)
{
    if (!h) return SF_ERR_ARG;
    SfDeviceGuard guard(h);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    int rc = sf_snap_args(h, "sf_load", env_ids, n, records, true, s);
    if (rc) return rc;
    if (rows) {
        for (int i = 0; i < n; ++i)
            if (rows[i] < 0 || rows[i] >= n_records) return sf_fail(h, SF_ERR_ARG, "sf_load: record row out of range");
        SF_CUDA(h, cudaMemcpyAsync(h->d_rows, rows, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    } else if (n_records < n) {
        return sf_fail(h, SF_ERR_ARG, "sf_load: fewer records than arenas");
    }
    const uint8_t *rec = static_cast<const uint8_t *>(records);
    const int32_t *d_ids = env_ids ? h->d_ids : nullptr, *d_rows = rows ? h->d_rows : nullptr;
    SF_CUDA(h, cudaMemsetAsync(h->d_refused, 0, sizeof(int), s));
    sf_snap_check_kernel<<<(n + 255) / 256, 256, 0, s>>>(h->snap, rec, d_rows, n, h->d_refused);
    sf_snap_kernel<false><<<sf_snap_grid(h, n), SF_SNAP_CTA, 0, s>>>(h->snap, h->k.env_id_base, d_ids, n, const_cast<uint8_t *>(rec),
                                                                    d_rows, h->d_refused);
    sf_snap_reseed_kernel<<<(n + 255) / 256, 256, 0, s>>>(h->d, h->k, rec, h->snap.bytes, d_ids, d_rows, n, h->d_refused);
    h->launches += 3;
    SF_CUDA(h, cudaGetLastError());
    int refused = 0;
    SF_CUDA(h, cudaMemcpyAsync(&refused, h->d_refused, sizeof refused, cudaMemcpyDeviceToHost, s));
    SF_CUDA(h, cudaStreamSynchronize(s));
    if (refused) return sf_fail(h, SF_ERR_ARG, "sf_load: a record is not one of this configuration (magic, version, size or fingerprint)");
    return SF_OK;
}

int32_t sf_agents_per_env(const sf_handle *h) { return h ? h->k.n_agents : 0; }
int32_t sf_num_envs(const sf_handle *h) { return h ? h->d.n_envs : 0; }
int64_t sf_launch_count(const sf_handle *h) { return h ? h->launches : 0; }
int64_t sf_device_bytes(const sf_handle *h) { return h ? (int64_t)h->arena_bytes : 0; }

} /* extern "C" */
