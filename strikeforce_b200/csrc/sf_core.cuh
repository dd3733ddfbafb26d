/*
 * sf_core.cuh -- the per-arena tick of the batched simulator (device code).
 *
 * One CUDA thread advances one arena; the 32 lanes of a warp walk the slot arrays of 32
 * neighbouring arenas in lock step (state layout: sf_state.h).  Everything here is a
 * from-scratch formulation of the loop body of gameplay::play()
 * (reference StrikeForce-client/gameplay.hpp:1443-1472) on that layout; each function names
 * the reference code whose observable behaviour it reproduces bit for bit.
 *
 * The file is plain C++ under SF_FN so that tests/hostcheck can compile the very same
 * functions with g++ and diff them against the CPU models without a GPU.  That build is
 * a debugging aid for tests only; the product library contains the CUDA build alone.
 */
#ifndef SF_CORE_CUH
#define SF_CORE_CUH

#include "sf_state.h"
#include "sf_synth.h"

#ifdef __CUDACC__
#define SF_FN __device__ __forceinline__
#define SF_COLD __device__ __noinline__ /* rare paths stay out of the step kernel's hot code */
#define SF_MFN __device__ __forceinline__
#define SF_UNROLL _Pragma("unroll")
#define SF_NO_UNROLL _Pragma("unroll 1") /* cold loops: the step kernel is instruction-fetch sensitive */
/* the per-entity rules of a round are unrolled like its loads.  A/B build -DSF_SINGLE_COPY_RULES: one copy
 * of the rules per phase (select chains over the round's registers) makes the kernel 15% smaller
 * (13,976 -> 11,840 SASS instructions) and 6.7% SLOWER (1.237 -> 1.320 ms): the selects and the loop
 * cost more than the instruction cache gives back. */
#ifdef SF_SINGLE_COPY_RULES
#define SF_RULES_UNROLL _Pragma("unroll 1")
#else
#define SF_RULES_UNROLL _Pragma("unroll")
#endif
#else
#define SF_FN static inline
#define SF_COLD static
#define SF_MFN inline
#define SF_UNROLL
#define SF_NO_UNROLL
#define SF_RULES_UNROLL
#endif

/* Warp-lockstep helpers.  The device runs one arena per lane; every loop of the tick has a
 * warp-uniform trip count (the maximum over the 32 lanes) and ends each iteration with
 * SF_SYNCWARP(), and no lane leaves a phase early (a failed arena just turns `e.on` off), so
 * the 32 lanes re-converge after every divergent branch instead of drifting apart. */
#ifdef __CUDA_ARCH__
#define SF_SYNCWARP() __syncwarp()
#define SF_WARP_MAX(x) __reduce_max_sync(0xffffffffu, (int)(x))
#else
#define SF_SYNCWARP() ((void)0)
#define SF_WARP_MAX(x) ((int)(x))
#endif

/* A CTA barrier between the phases of a step keeps the 28 warps of an SM inside the same stretch of
 * code: the step kernel is ~210 KB of SASS and 13% of its stall samples were instruction fetch;
 * with the barriers a step is 3% shorter (callers: only the step kernels, whose warps all make the
 * same number of passes). */
#ifndef SF_BARRIER_MASK
#define SF_BARRIER_MASK 0x1F
#endif
#if defined(__CUDA_ARCH__) && !defined(SF_NO_PHASE_BARRIERS)
#define SF_PHASE_SYNC(n) do { if ((SF_BARRIER_MASK >> (n)) & 1) __syncthreads(); } while (0)
#else
#define SF_PHASE_SYNC(n) ((void)0)
#endif

#ifdef SF_DEBUG_HIST
static unsigned long long sf_dbg_hist[256]; /* host-check builds only: flagged cells per arena when the bullets are resolved */
#endif
#define SF_RNG_ZERO 0x10000u /* log-domain marker of the value 0 (only during the warm-up) */

/* tables every lane reads: shared memory on the device, plain arrays in the host check */
struct SfTabs {
    const uint8_t *smap;     /* static map bytes [SF_TCELLS], tiled cell ids */
    const uint16_t *exp_tab; /* [32768]: the first half of 3^k - 1; the rest follows from 3^32768 = -1 (sf_exp_m1) */
    const uint16_t *log_tab; /* [65536] */
    const uint32_t *rng_cst; /* [2][18][E] per-arena term constants (terms 10..17 are read on demand) */
    int32_t E;
    uint16_t *bt;            /* this arena's table of flagged cells: entry i at bt[i * bt_stride] (sf_bt_*) */
    int32_t bt_stride;
};

/* register-resident part of one arena while a kernel works on it */
struct SfEnv {
    uint32_t frame, steps, episode, jomle, ntemp;
    int32_t kills, tkills, loot, chest;
    int32_t level, status, hw_h;
    uint64_t mh, mz[2], mb[2], mp[2];
    uint64_t quit;       /* humans whose Hp was zeroed by '_' (gameplay.hpp:696-699) */
    bool on;             /* this lane holds an arena that is still running this step */
    int env;             /* arena index of this lane */
    uint32_t Lp[9];      /* log_3 of random[0..17] (random.hpp:31), two 16-bit logs per word */
    uint32_t cst[10];    /* terms 0..9: 2*seed[i] | 2*log_3(us[i]) << 8 */
    uint32_t W;          /* sum of the values random[10..17] (see sf_rand) */
    bool fast;           /* both seeds below 10^10: terms 10..17 are the plain window W */
    bool bank;           /* which half of rng_cst holds this stream's term constants */
    bool watch;          /* a human may stand on a portal exit (sf_portal_damage); false = provably none */
};

/* ------------------------------------------------------------------ small helpers */

SF_FN int sf_ffs64(uint64_t x)
{
#ifdef __CUDA_ARCH__
    return __ffsll((long long)x) - 1;
#else
    return x ? __builtin_ctzll(x) : -1;
#endif
}
SF_FN int sf_fls64(uint64_t x)
{
#ifdef __CUDA_ARCH__
    return 63 - __clzll((long long)x);
#else
    return x ? 63 - __builtin_clzll(x) : -1;
#endif
}
SF_FN int sf_popc64(uint64_t x)
{
#ifdef __CUDA_ARCH__
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}

/* 128-bit slot masks as two words */
SF_FN bool m2_test(const uint64_t m[2], int i) { return (m[i >> 6] >> (i & 63)) & 1; }
SF_FN void m2_set(uint64_t m[2], int i) { m[i >> 6] |= 1ull << (i & 63); }
SF_FN void m2_clear(uint64_t m[2], int i) { m[i >> 6] &= ~(1ull << (i & 63)); }
SF_FN int m2_lowest_free(const uint64_t m[2])
{
    if (~m[0]) return sf_ffs64(~m[0]);
    if (~m[1]) return 64 + sf_ffs64(~m[1]);
    return 128;
}
SF_FN int m2_highest(const uint64_t m[2])
{
    if (m[1]) return 64 + sf_fls64(m[1]);
    return sf_fls64(m[0]);
}
SF_FN int m2_count(const uint64_t m[2]) { return sf_popc64(m[0]) + sf_popc64(m[1]); }
/* next set bit at or above i (ascending walk), -1 if none */
SF_FN int m2_next(const uint64_t m[2], int i)
{
    if (i < 64) {
        uint64_t w = m[0] >> i;
        if (w) return i + sf_ffs64(w);
        i = 64;
    }
    if (i < 128) {
        uint64_t w = m[1] >> (i - 64);
        if (w) return i + sf_ffs64(w);
    }
    return -1;
}
/* next set bit at or below i (descending walk), -1 if none */
SF_FN int m2_prev(const uint64_t m[2], int i)
{
    if (i >= 64) {
        uint64_t w = m[1] << (127 - i);
        if (w) return i - (63 - sf_fls64(w));
        i = 63;
    }
    if (i >= 0) {
        uint64_t w = m[0] << (63 - i);
        if (w) return i - (63 - sf_fls64(w));
    }
    return -1;
}

/* ------------------------------------------------------------------ addressing */

#define SF_AT(arr, slot) (arr)[(size_t)(slot) * (size_t)d.E + (size_t)env]
/* player-built records are contiguous per arena (they are searched by cell, not walked) */
#define SF_T(arr, q) (arr)[(size_t)env * (size_t)d.cap_t + (size_t)(q)]
#define SF_G(cell) d.grid[(size_t)env * SF_GRID_STRIDE + (size_t)(cell)]

SF_FN int sf_cell_of(int f, int r, int c) { return sf_tcell(f, r, c); }
/* the neighbour of a (tiled) cell id, no bounds test; wdx / wdy, gameplay.hpp:459:
 * way-1 = 0 down(+row) 1 right(+col) 2 up 3 left.  Inside a tile rows are 8 ids apart and
 * columns 1; the next tile to the right starts 32 ids later, the one below 13 * 32 later. */
SF_FN int sf_step_cell(int t, int d)
{
    const int inr = (t >> 3) & 3, inc = t & 7;
    if (d == 0) return inr != 3 ? t + 8 : t + SF_TILES_X * 32 - 24;
    if (d == 1) return inc != 7 ? t + 1 : t + 32 - 7;
    if (d == 2) return inr != 0 ? t - 8 : t - SF_TILES_X * 32 + 24;
    return inc != 0 ? t - 1 : t - 32 + 7;
}
/* neighbour in direction d with the bounds test obey() makes (gameplay.hpp:704, 747, 801) */
SF_FN bool sf_neighbour(int cell, int d, int *out)
{
    int f, r, c;
    sf_tcell_decode(cell, &f, &r, &c);
    r += (d == 0) - (d == 2);
    c += (d == 1) - (d == 3);
    *out = sf_step_cell(cell, d);
    return !(r >= SF_ROWS || r < 0 || c >= SF_COLS || c < 0);
}

/* node::showit(), gameplay.hpp:321-341, from the static byte, the overlay word and the cell's
 * bullet flag s[2] (which is not stored in the overlay: sf_owner_at).  s[8] (death mark) is
 * render-only: updmap() clears it before any rule reads a cell (:489-495). */
SF_FN int sf_showit(uint32_t st, uint32_t g, bool s2)
{
    uint32_t kind = (g >> C_KIND_SHIFT) & 7u;
    if ((st & M_WALL) || kind == K_BLOCK) return SH_WALL;
    if (g & C_S0) return SH_HUMAN;
    if (g & C_S1) return SH_ZOMBIE;
    if ((st & M_UP) || kind == K_ENTRANCE) return SH_UP;
    if (st & M_DOWN) return SH_DOWN;
    if (s2) return SH_BULLET;
    if (kind >= K_CHEST0 && kind < K_BLOCK) return SH_CHEST;
    if ((st & M_EXIT) || kind == K_EXIT) return SH_EXIT;
    return SH_DOT;
}

/* a portal exit, static ('O' of the map) or player-built */
SF_FN bool sf_is_exit(const SfTabs &t, int cell, uint32_t g)
{
    return (t.smap[cell] & M_EXIT) || ((g >> C_KIND_SHIFT) & 7u) == K_EXIT;
}

/* ------------------------------------------------------------------ random.hpp */

/* _rand(), random.hpp:54-62, in the discrete-log domain of the cyclic group mod 65537
 * (generator 3): random[i]^seed[i] * us[i] = 3^(L[i]*seed[i] + log us[i]) and the new element
 * (sum)^jomle = 3^(log(sum) * jomle).  exp_tab holds 3^k - 1, so a term is "entry + 1".
 *
 * Seeds below 10^10 (a unix time, a 30-bit serial: gameplay.hpp:1745-1747) have digits 10..17
 * equal to 0, i.e. seed[i] = us[i] = 1 there, so those eight terms are the plain values
 * random[10..17] -- a window that slides by one element per draw.  Arenas flagged `fast` keep
 * that window sum in W (minus the element leaving, plus the new one) and look up only the ten
 * leading terms; a lane with longer seeds takes the eight extra look-ups itself. */
SF_FN uint32_t sf_rng_log(const SfEnv &e, int i) { return (e.Lp[i >> 1] >> (16 * (i & 1))) & 0xFFFFu; }

/* 3^k mod 65537, minus one, for k2 = 2 * k (k < 65536).  Only the first half of the table is kept
 * (64 KB of shared memory instead of 128 KB -- the other half holds the bullet-flag tables of the
 * CTA's arenas): 3^32768 = -1 (mod 65537), so 3^(k + 32768) - 1 = 65536 - 3^k = 65535 - (3^k - 1),
 * the 16-bit complement of the entry. */
SF_FN uint32_t sf_exp_m1(const SfTabs &t, uint32_t k2)
{
#ifdef SF_FULL_EXP /* A/B build: the whole table in shared memory (a 228 KB carve-out, 28 KB of L1) */
    return *(const uint16_t *)((const uint8_t *)t.exp_tab + k2);
#else
    const uint32_t v = *(const uint16_t *)((const uint8_t *)t.exp_tab + (k2 & 0xFFFEu));
    return (k2 & 0x10000u) ? (v ^ 0xFFFFu) : v;
#endif
}

SF_FN uint32_t sf_rng_term(const SfTabs &t, uint32_t L, uint32_t c)
{
    return sf_exp_m1(t, (L * (c & 0xFFu) + (c >> 8)) & 0x1FFFEu);
}

SF_FN int sf_rand(SfEnv &e, const SfTabs &t)
{
    uint32_t S = 11u; /* 1 + ten terms of "entry + 1" */
    SF_UNROLL
    for (int i = 0; i < 10; ++i) S += sf_rng_term(t, sf_rng_log(e, i), e.cst[i]);
    if (e.fast) {
        S += e.W;
    } else { /* a plain per-lane branch: draws happen in divergent code, no warp vote here */
        S += 8u;
        SF_UNROLL
        for (int i = 10; i < 18; ++i) S += sf_rng_term(t, sf_rng_log(e, i), t.rng_cst[((size_t)(e.bank ? 18 : 0) + (size_t)i) * (size_t)t.E + (size_t)e.env]);
    }
    /* S < 2^21: fold with 65536 == -1 (mod 65537) */
    int32_t r = (int32_t)(S & 0xFFFFu) - (int32_t)(S >> 16);
    if (r < 0) r += 65537;
    if (r == 0) r = 1;                                        /* sum + (sum == 0) */
    uint32_t lg = t.log_tab[r - 1];
    e.jomle += 1;
    uint32_t ln = (lg * (e.jomle & 0xFFFFu)) & 0xFFFFu;       /* binpow(sum, jomle), :42-52 */
    uint32_t val = sf_exp_m1(t, 2u * ln) + 1u;
    e.W += val - (sf_exp_m1(t, 2u * sf_rng_log(e, 10)) + 1u); /* element 10 leaves the window */
    SF_UNROLL
    for (int j = 0; j < 8; ++j) e.Lp[j] = (e.Lp[j] >> 16) | (e.Lp[j + 1] << 16);
    e.Lp[8] = (e.Lp[8] >> 16) | (ln << 16);
    return (int)(val & 1023u);
}

/* ---- _srand(tb, u_s), random.hpp:64-76 -------------------------------------------------
 * Seeding digit-splits both seeds, starts from eighteen zeros and discards 1024 draws.  The
 * draws are strictly serial (about 0.2 ms of dependent work), far longer than a whole step of
 * the batch, so an episode's stream is never warmed up on the step path: every arena carries
 * a PENDING stream -- the one its next episode will use -- which each step advances by
 * SF_WARM_PER_STEP draws with all lanes in lock step.  When the episode ends the pending stream
 * is installed (any draws still missing are made then) and the stream after it is seeded.
 *
 * During the warm-up zero has no logarithm; but after n draws the zeros are exactly the
 * elements 0 .. 17-n, so term i simply counts only when i + n >= 18. */
#define SF_WARM_DRAWS 1024u
#define SF_WARM_PER_STEP 8

SF_FN size_t sf_cst_index(const SfDev &d, int bank, int i, int env)
{
    return ((size_t)bank * 18 + (size_t)i) * (size_t)d.E + (size_t)env;
}

/* one warm-up draw of a stream held as packed logs Lp[9] with term constants c[18];
 * n = draws made so far (jomle = 18 + n) */
SF_FN void sf_warm_draw(const SfTabs &t, uint32_t Lp[9], const uint32_t c[18], uint32_t n)
{
    uint32_t S = 1u;
    SF_UNROLL
    for (int i = 0; i < 18; ++i) {
        uint32_t L = (Lp[i >> 1] >> (16 * (i & 1))) & 0xFFFFu;
        uint32_t term = sf_rng_term(t, L, c[i]) + 1u;
        if ((uint32_t)i + n >= 18u) S += term;
    }
    int32_t r = (int32_t)(S & 0xFFFFu) - (int32_t)(S >> 16);
    if (r < 0) r += 65537;
    if (r == 0) r = 1;
    uint32_t jomle = 18u + n + 1u;
    uint32_t ln = ((uint32_t)t.log_tab[r - 1] * (jomle & 0xFFFFu)) & 0xFFFFu;
    SF_UNROLL
    for (int j = 0; j < 8; ++j) Lp[j] = (Lp[j] >> 16) | (Lp[j + 1] << 16);
    Lp[8] = (Lp[8] >> 16) | (ln << 16);
}

/* digit-split the seeds of a stream into term constants of `bank` and mark it un-warmed */
SF_FN void sf_seed_pending(const SfDev &d, const SfTabs &t, int env, int bank, int64_t tb, int64_t u_s)
{
    uint32_t fast = (tb < 10000000000ll && u_s < 10000000000ll) ? 1u : 0u;
    SF_NO_UNROLL
    for (int i = 0; i < 18; ++i) {
        uint32_t us = (uint32_t)(u_s % 10 + 1), sd = (uint32_t)(tb % 10 + 1);
        u_s /= 10;
        tb /= 10;
        d.rng_cst[sf_cst_index(d, bank, i, env)] = (2u * sd) | ((2u * (uint32_t)t.log_tab[us - 1]) << 8);
    }
    SF_UNROLL
    for (int j = 0; j < 9; ++j) SF_AT(d.pend_log, j) = 0u;
    d.pend_n[env] = fast << 16;
}

/* advance the pending stream of arena `env` by up to `budget` draws */
SF_FN void sf_advance_pending(const SfDev &d, const SfTabs &t, int env, bool valid, int budget)
{
    uint32_t pn = valid ? d.pend_n[env] : SF_WARM_DRAWS;
    uint32_t n = pn & 0xFFFFu;
    if (n < SF_WARM_DRAWS) {
        const int bank = (int)((d.misc[env] >> 25) & 1u) ^ 1;
        uint32_t Lp[9], c[18];
        SF_UNROLL
        for (int j = 0; j < 9; ++j) Lp[j] = SF_AT(d.pend_log, j);
        SF_UNROLL
        for (int i = 0; i < 18; ++i) c[i] = d.rng_cst[sf_cst_index(d, bank, i, env)];
        SF_NO_UNROLL
        for (int j = 0; j < budget; ++j) {
            if (n < SF_WARM_DRAWS) {
                sf_warm_draw(t, Lp, c, n);
                n += 1;
            }
        }
        SF_UNROLL
        for (int j = 0; j < 9; ++j) SF_AT(d.pend_log, j) = Lp[j];
        d.pend_n[env] = (pn & ~0xFFFFu) | n;
    }
    /* no warp barrier here: sf_install_stream calls this from a single lane */
}

/* make the pending stream the arena's stream (finishing its warm-up if need be) and seed the
 * stream of the episode after it */
SF_FN void sf_install_stream(const SfDev &d, const SfTabs &t, int env, SfEnv &e, int64_t next_tb, int64_t next_serial)
{
    sf_advance_pending(d, t, env, true, (int)SF_WARM_DRAWS);
    e.bank = !e.bank;
    e.fast = (d.pend_n[env] >> 16) & 1u;
    SF_UNROLL
    for (int j = 0; j < 9; ++j) e.Lp[j] = SF_AT(d.pend_log, j);
    SF_UNROLL
    for (int i = 0; i < 10; ++i) e.cst[i] = d.rng_cst[sf_cst_index(d, e.bank ? 1 : 0, i, env)];
    e.jomle = 18u + SF_WARM_DRAWS;
    e.W = 0;
    for (int i = 10; i < 18; ++i) e.W += sf_exp_m1(t, 2u * sf_rng_log(e, i)) + 1u;
    /* the header must carry the new bank before the next pending stream is addressed */
    d.misc[env] = (d.misc[env] & ~(1u << 25)) | (e.bank ? 1u << 25 : 0u);
    sf_seed_pending(d, t, env, e.bank ? 0 : 1, next_tb, next_serial);
}

/* ------------------------------------------------------------------ entities */

SF_FN const SfTemplate &sf_tmpl(const SfConst &k, int h) { return h < k.n_players ? k.players[h] : k.npc; }
SF_FN int sf_punch_base(const SfConst &k, const SfEnv &e, int h)
{
    return h < k.n_players ? k.player_punch_base[h] : k.npc_punch_base[e.level];
}

/* an arena that needs a slot beyond its configured capacity stops (harness: SF_OVERFLOW) */
SF_FN void sf_fail_env(SfEnv &e, int status)
{
    e.status = status;
    e.on = false;
}

/* write every field of human slot h: Human::build + gen_human (Character.hpp:650-709, 873-888)
 * or the `hum[ind] = me` copy of load_data (gameplay.hpp:1864, 1909) */
SF_FN void sf_init_human(const SfDev &d, int env, const SfTemplate &tp, int h, int cell, bool rnpc, int team,
                         bool agent)
{
    SF_AT(d.h_pw, h) = (uint16_t)cell; /* way = 1 */
    SF_AT(d.h_sel, h) = (uint16_t)(sf_team_bits(team) | (rnpc ? HS_RNPC : 0u) | (agent ? HS_AGENT : 0u));
    SF_AT(d.h_bp, h) = (uint32_t)tp.blocks | ((uint32_t)tp.portals << 8);
    SF_AT(d.h_hp, h) = tp.hp;
    SF_AT(d.h_mind, h) = tp.mindamage;
    SF_AT(d.h_stam, h) = tp.stamina;
    SF_AT(d.h_kills, h) = 0;
    SF_AT(d.h_dmg, h) = 0;
    SF_AT(d.h_eff, h) = 0;
    SF_AT(d.h_cons, h) = tp.cons_packed;
    SF_AT(d.h_thr, h) = tp.thr_packed;
}

/* lowest free bullet slot (b_ind, gameplay.hpp:230-235); -1 and the arena fails when it lies
 * at or beyond the configured capacity */
SF_FN int sf_alloc_bullet(const SfConst &k, SfEnv &e)
{
    int b = m2_lowest_free(e.mb);
    if (b >= k.cap_b) {
        sf_fail_env(e, SF_OVERFLOW);
        return -1;
    }
    m2_set(e.mb, b);
    return b;
}

/* ---- the bullet flag s[2] ------------------------------------------------------------------
 * node::s[2] ("a bullet is here") and node::bullet (its last writer, gameplay.hpp:237-243) are not
 * stored per cell: s[2] of a cell is set exactly while one live bullet standing in it carries
 * BF_OWNS -- that bullet is the last writer -- so both are a property of the bullet list.  Moving
 * bullets are the bulk of all cell updates of a step (set at the new cell, cleared at the old one,
 * every half-tick), and on this layout a cell update is a scattered 2-byte write into a 2.6 GB
 * overlay; deriving the flag instead removes those writes and the look-ahead read of update_bull.
 *
 * "Is there a bullet flag on this cell?" is answered by a per-arena TABLE in shared memory: an
 * open-addressing hash set (linear probing) of the flagged cells, SF_BT_SLOTS 16-bit entries
 * (cell + 1, 0 = empty) plus a count.  One lane's rare event is its whole warp's wait -- and, with
 * the phase barriers, its whole CTA's -- so nothing on this path may be slow, not even the
 * overflow: an arena with more than SF_BT_FULL flagged cells (1% of the arenas of the benchmark
 * at any time) SPILLS the next flags into the overlay word of their cell (C_S2, the bit the
 * reference keeps there), marks their bullets BF_SPILL and raises SF_BT_SPILL in its count; while
 * that is up a look-up that misses the table also reads the cell.  sf_resolve_bullets, which
 * consumes every flag, clears the spilled bits through their bullets and wipes the table.  The
 * table is rebuilt from the bullet rows when a kernel picks an arena up. */
#ifndef SF_BT_SLOTS
#define SF_BT_SLOTS 47
#define SF_BT_FULL 40
#endif
#define SF_BT_ENTRIES (SF_BT_SLOTS + 1) /* 48 x uint16 = 24 words per arena */
#define SF_BT_SPILL 0x8000u
SF_FN uint16_t &sf_bt_at(const SfTabs &t, int i) { return t.bt[i * t.bt_stride]; }
SF_FN void sf_bt_wipe(const SfTabs &t)
{
    SF_UNROLL
    for (int i = 0; i < SF_BT_ENTRIES; ++i) sf_bt_at(t, i) = 0;
}
/* the slot that holds `cell`, or -1 - (the empty slot where it would go) */
SF_FN int sf_bt_find(const SfTabs &t, int cell)
{
    const uint32_t key = (uint32_t)cell + 1u;
    int i = (int)(((((uint32_t)cell * 40503u) >> 3) & 0xFFFFu) * SF_BT_SLOTS >> 16);
    SF_NO_UNROLL
    for (;;) {
        const uint32_t v = sf_bt_at(t, i);
        if (v == key) return i;
        if (v == 0u) return -1 - i;
        i = i + 1 == SF_BT_SLOTS ? 0 : i + 1;
    }
}
/* node::s[2] of `cell` */
SF_FN bool sf_flagged(const SfDev &d, const SfTabs &t, int env, int cell)
{
    if (sf_bt_find(t, cell) >= 0) return true;
    return (sf_bt_at(t, SF_BT_SLOTS) & SF_BT_SPILL) && (SF_G(cell) & C_S2);
}
/* raise the flag of `cell`: 0 = it was up already (in the table), SF_FLAG_NEW = raised in the
 * table, and with BF_SPILL or'ed in: ... in the overlay (the bullet that owns the flag carries
 * that bit: it is the one that takes the flag down again) */
#define SF_FLAG_NEW 1u
SF_FN uint32_t sf_flag_cell(const SfDev &d, const SfTabs &t, int env, int cell)
{
    const int i = sf_bt_find(t, cell);
    if (i >= 0) return 0u;
    const uint32_t n = sf_bt_at(t, SF_BT_SLOTS);
    if (n & SF_BT_SPILL) { /* some flags of this arena live in the overlay: this one? */
        const uint32_t g = SF_G(cell);
        if (g & C_S2) return BF_SPILL;
        if ((n & ~SF_BT_SPILL) >= SF_BT_FULL) {
            SF_G(cell) = (uint16_t)(g | C_S2);
            return SF_FLAG_NEW | BF_SPILL;
        }
    } else if (n >= SF_BT_FULL) {
        SF_G(cell) = (uint16_t)(SF_G(cell) | C_S2);
        sf_bt_at(t, SF_BT_SLOTS) = (uint16_t)(n | SF_BT_SPILL);
        return SF_FLAG_NEW | BF_SPILL;
    }
    sf_bt_at(t, -1 - i) = (uint16_t)(cell + 1);
    sf_bt_at(t, SF_BT_SLOTS) = (uint16_t)(n + 1u);
    return SF_FLAG_NEW;
}

/* the live bullet that owns `cell` (slot `skip` left out), -1 if none: a walk over the bullet
 * rows, eight positions in flight at a time.  Needed only when a bullet is put on a cell that is
 * flagged already (the old last writer loses BF_OWNS) and by the kernels outside the tick; one
 * out-of-line copy that takes plain values, so the arena's registers stay where they are. */
SF_COLD int sf_owner_walk(const uint16_t *pw, const uint32_t *meta, size_t stride, uint64_t m0, uint64_t m1, int cell,
                          int skip)
{
    SF_NO_UNROLL
    for (int half = 0; half < 2; ++half) {
        uint64_t m = half ? m1 : m0;
        SF_NO_UNROLL
        while (m) {
            int o[8];
            uint32_t p[8];
            SF_UNROLL
            for (int j = 0; j < 8; ++j) {
                o[j] = m ? half * 64 + sf_ffs64(m) : -1;
                m &= m - 1; /* 0 stays 0 */
                p[j] = o[j] >= 0 ? (uint32_t)pw[(size_t)o[j] * stride] : 0xFFFFu;
            }
            SF_UNROLL
            for (int j = 0; j < 8; ++j)
                if ((int)(p[j] & POS_CELL) == cell && o[j] >= 0 && o[j] != skip && (meta[(size_t)o[j] * stride] & BF_OWNS))
                    return o[j];
        }
    }
    return -1;
}
SF_FN int sf_owner_scan(const SfDev &d, int env, const SfEnv &e, int cell, int skip)
{
    return sf_owner_walk(d.b_pw + env, d.b_meta + env, (size_t)d.E, e.mb[0], e.mb[1], cell, skip);
}

/* rebuild the table from the bullet rows (the owning bullets of a resting arena are exact; the
 * spilled flags are in the overlay already) */
SF_FN void sf_bt_rebuild(const SfDev &d, const SfTabs &t, int env, const SfEnv &e)
{
    sf_bt_wipe(t);
    const int hi = SF_WARP_MAX(e.on ? m2_highest(e.mb) : -1);
    const uint64_t live0 = e.on ? e.mb[0] : 0ull, live1 = e.on ? e.mb[1] : 0ull;
    for (int b0 = 0; b0 <= hi; b0 += 4) {
        uint32_t pw[4], meta[4];
        SF_UNROLL
        for (int j = 0; j < 4; ++j) {
            const int b = b0 + j;
            const bool lv = b <= hi && (((b < 64 ? live0 : live1) >> (b & 63)) & 1);
            pw[j] = lv ? (uint32_t)SF_AT(d.b_pw, b) : 0u;
            meta[j] = lv ? SF_AT(d.b_meta, b) : 0u;
        }
        SF_NO_UNROLL
        for (int j = 0; j < 4; ++j) {
            const uint32_t mj = j == 0 ? meta[0] : j == 1 ? meta[1] : j == 2 ? meta[2] : meta[3];
            const uint32_t pj = j == 0 ? pw[0] : j == 1 ? pw[1] : j == 2 ? pw[2] : pw[3];
            if (mj & BF_SPILL) sf_bt_at(t, SF_BT_SLOTS) = (uint16_t)(sf_bt_at(t, SF_BT_SLOTS) | SF_BT_SPILL);
            else if (mj & BF_OWNS) {
                const uint32_t fl = sf_flag_cell(d, t, env, (int)(pj & POS_CELL));
                if (fl & BF_SPILL) SF_AT(d.b_meta, b0 + j) = mj | BF_SPILL; /* never: the table held them before */
            }
        }
        SF_SYNCWARP();
    }
}

/* a new bullet becomes the cell's last writer (node::bullet under s[2]); any older owner of
 * the same cell keeps flying but loses the flag */
SF_FN void sf_write_bullet(const SfDev &d, int env, int b, int cell, int way0, int range, int owner, int dmg, int eff,
                           uint32_t fl)
{
    SF_AT(d.b_pw, b) = (uint16_t)(cell | (way0 << POS_HI_SHIFT));
    SF_AT(d.b_meta, b) = (uint32_t)range | ((uint32_t)(owner + 1) << 16) | BF_OWNS | (fl & BF_SPILL);
    SF_AT(d.b_dmg, b) = dmg;
    SF_AT(d.b_eff, b) = eff;
}
SF_FN void sf_place_bullet(const SfDev &d, const SfTabs &t, int env, SfEnv &e, int b, int cell, int way0, int range,
                           int owner, int dmg, int eff)
{
    const uint32_t fl = sf_flag_cell(d, t, env, cell);
    if (!(fl & SF_FLAG_NEW)) { /* rare, and always inside divergent code */
        int o = sf_owner_scan(d, env, e, cell, b);
        if (o >= 0) SF_AT(d.b_meta, o) = SF_AT(d.b_meta, o) & ~(BF_OWNS | BF_SPILL);
    }
    sf_write_bullet(d, env, b, cell, way0, range, owner, dmg, eff, fl);
}

/* slot of the player-built record of `cell` in the temp list (gameplay.hpp:469), -1 if none.
 * A rare event (a stale or missing hint, sf_built_slot), called from several places: one
 * out-of-line copy that takes plain values, so the arena's registers stay where they are. */
SF_FN int sf_find_built_in(const uint16_t *tc, uint32_t ntemp, int cell)
{
    int found = -1;
#ifdef __CUDA_ARCH__
    /* the per-arena record block is 16-byte aligned (cap_t is a multiple of 8) */
    const uint4 *tv = reinterpret_cast<const uint4 *>(tc);
    const uint32_t want = (uint32_t)cell;
    /* callers are inside divergent code, so the walk may stop at the first hit */
    for (uint32_t q0 = 0; q0 < ntemp && found < 0; q0 += 8) {
        uint4 v = tv[q0 >> 3];
        uint32_t w[4] = {v.x, v.y, v.z, v.w};
        SF_UNROLL
        for (int j = 3; j >= 0; --j) {
            if ((w[j] >> 16) == want && q0 + 2 * j + 1 < ntemp) found = (int)(q0 + 2 * j + 1);
            if ((w[j] & 0xFFFFu) == want && q0 + 2 * j < ntemp) found = (int)(q0 + 2 * j);
        }
    }
#else
    for (uint32_t q = 0; q < ntemp && found < 0; ++q)
        if (tc[q] == cell) found = (int)q;
#endif
    return found;
}
SF_FN int sf_find_built(const SfDev &d, int env, const SfEnv &e, int cell)
{
    return sf_find_built_in(&SF_T(d.t_cell, 0), e.ntemp, cell);
}
/* A player-built cell that nobody stands on carries a HINT of its record's slot in the bits the
 * occupant does not need (0-7 and 14-15, ten bits).  The hint is always validated against the
 * record, so a stale one (after a human stood there, or after a swap-remove) only costs the
 * search; whoever searched writes the fresh hint back. */
#define C_HINT 0xC0FFu
SF_FN uint32_t sf_hint_bits(int q) { return ((uint32_t)q & 0xFFu) | (((uint32_t)q >> 8) & 3u) << 14; }
SF_FN int sf_built_slot(const SfDev &d, int env, const SfEnv &e, int cell, uint32_t g)
{
    if (!(g & (C_S0 | C_S1))) {
        uint32_t hq = (g & 0xFFu) | ((g >> 14) & 3u) << 8;
        if (hq < e.ntemp && SF_T(d.t_cell, hq) == cell) return (int)hq;
    }
    int q = sf_find_built(d, env, e, cell);
    if (q >= 0 && q < 1024 && !(g & (C_S0 | C_S1))) SF_G(cell) = (uint16_t)((g & ~C_HINT) | sf_hint_bits(q));
    return q;
}
SF_FN void sf_remove_built(const SfDev &d, int env, SfEnv &e, int q)
{
    uint32_t last = e.ntemp - 1;
    if ((uint32_t)q != last) {
        SF_T(d.t_cell, q) = SF_T(d.t_cell, last);
        SF_T(d.t_dmg, q) = SF_T(d.t_dmg, last);
        SF_T(d.t_pidx, q) = SF_T(d.t_pidx, last);
    }
    e.ntemp = last;
}
SF_FN bool sf_push_built(const SfDev &d, const SfConst &k, int env, SfEnv &e, int cell, int pidx)
{
    if ((int)e.ntemp >= k.cap_t) { /* harness: temp.size() > cap is SF_OVERFLOW */
        sf_fail_env(e, SF_OVERFLOW);
        return false;
    }
    SF_T(d.t_cell, e.ntemp) = (uint16_t)cell;
    SF_T(d.t_dmg, e.ntemp) = 0;
    SF_T(d.t_pidx, e.ntemp) = (uint8_t)pidx;
    e.ntemp += 1;
    return true;
}

SF_FN int sf_exit_cell(const SfDev &d, const SfConst &k, int env, int idx)
{
    return idx < k.n_static_exits ? (int)k.static_exit_cell[idx] : (int)SF_AT(d.p_cell, idx);
}

/* ------------------------------------------------------------------ spawns */

/* spawn_chest / spawn_zombie_npc / spawn_human_npc, gameplay.hpp:532-572 (Zombie::gen_npc
 * Character.hpp:850-857).  The three share their first three draws (floor, row, col) and the
 * "cell prints '.'" test, so they run as three rounds of one code path. */
SF_FN void sf_spawns(const SfDev &d, const SfConst &k, const SfTabs &t, int env, SfEnv &e)
{
#pragma unroll 1
    for (int kind = 0; kind < 3; ++kind) {
        uint32_t period = kind == 0 ? 30u : kind == 1 ? 40u : 50u; /* pc, pz, ph: gameplay.hpp:459 */
        bool due = e.on && (e.frame % period <= 1u);
        if (kind == 0 && 9000 <= e.chest) due = false; /* C, gameplay.hpp:37 */
        int i = 0, j = 0, c = 0;
#pragma unroll 1
        for (int q = 0; q < 3; ++q) { /* one draw site for floor, row, col */
            if (due) {
                int r = sf_rand(e, t);
                if (q == 0) i = r % SF_FLOORS;
                else if (q == 1) j = r % SF_ROWS;
                else c = r % SF_COLS;
            }
        }
        int cell = sf_cell_of(i, j, c);
        bool dot = false;
        if (due) dot = sf_showit(t.smap[cell], SF_G(cell), false) == SH_DOT && !sf_flagged(d, t, env, cell);
        int z = 0;
        if (dot && kind == 1) {
            z = m2_lowest_free(e.mz);
            if (z >= k.cap_z) {
                sf_fail_env(e, SF_OVERFLOW);
                dot = false;
            }
        }
        int extra = 0;
        if (dot && kind < 2) extra = sf_rand(e, t) % 4; /* chest type / "is it a super zombie" */
        if (dot) {
            if (kind == 0) {
                SF_G(cell) = (uint16_t)((K_CHEST0 + extra) << C_KIND_SHIFT);
                e.chest += 1;
                if (e.chest > k.cap_chest) sf_fail_env(e, SF_OVERFLOW);
            } else if (kind == 1) {
                int super_ = (extra == 0);
                SF_AT(d.z_pos, z) = (uint16_t)(cell | (super_ << POS_HI_SHIFT));
                SF_AT(d.z_hp, z) = (super_ + 1) * 400;
                SF_AT(d.z_mind, z) = (super_ + 1) * 100;
                SF_G(cell) = (uint16_t)(C_S1 | (uint32_t)z);
                m2_set(e.mz, z);
            } else {
                /* h_ind skips ind and the slots of the other players (remote[]), gameplay.hpp:216-221 */
                int h = sf_ffs64(~(e.mh | ((1ull << k.n_players) - 1ull)));
                if (h < 0 || h >= k.cap_h) sf_fail_env(e, SF_OVERFLOW);
                else {
                    sf_init_human(d, env, k.npc, h, cell, true, 0, false);
                    SF_G(cell) = (uint16_t)(C_S0 | (uint32_t)h);
                    e.mh |= 1ull << h;
                    if (h + 1 > e.hw_h) e.hw_h = h + 1;
                }
            }
        }
        SF_SYNCWARP();
    }
}

/* ------------------------------------------------------------------ half-tick pieces */

/* zombie_action, gameplay.hpp:654-693.  Two zombies per round: their positions, then their four
 * neighbours, are loaded back to back (eight independent loads in flight) before the rules run in
 * slot order; what the first zombie writes is forwarded into the second zombie's loaded copy so
 * that it sees exactly what a sequential walk would.  A zombie's own cell is never read: it holds
 * the zombie and nothing else (zombies only enter cells that print '.', and nothing is built or
 * dropped on an occupied cell), and its bullet flag comes from the table. */
SF_FN void sf_zombie_action(const SfDev &d, const SfConst &k, const SfTabs &t, int env, SfEnv &e)
{
    const int hi = SF_WARP_MAX(e.on ? m2_highest(e.mz) : -1);
    /* zombies neither appear nor vanish here: liveness comes from a snapshot of the mask, and the
     * positions of a round are loaded one round ahead */
    const uint64_t live0 = e.on ? e.mz[0] : 0ull, live1 = e.on ? e.mz[1] : 0ull;
    uint32_t pw_n[2];
    SF_UNROLL
    for (int j = 0; j < 2; ++j) {
        bool ln = j <= hi && (((j < 64 ? live0 : live1) >> (j & 63)) & 1);
        pw_n[j] = ln ? (uint32_t)SF_AT(d.z_pos, j) : 0u;
    }
    for (int z0 = 0; z0 <= hi; z0 += 2) {
        bool act[2];
        uint32_t pw[2];
        int cell[2];
        uint32_t gv[2][4];
        SF_UNROLL
        for (int j = 0; j < 2; ++j) {
            const int z = z0 + j;
            act[j] = e.on && z <= hi && (((z < 64 ? live0 : live1) >> (z & 63)) & 1);
            pw[j] = pw_n[j];
            cell[j] = (int)(pw[j] & POS_CELL);
        }
        SF_UNROLL
        for (int j = 0; j < 2; ++j) {
            const int z = z0 + 2 + j;
            bool ln = z <= hi && (((z < 64 ? live0 : live1) >> (z & 63)) & 1);
            pw_n[j] = ln ? (uint32_t)SF_AT(d.z_pos, z) : 0u;
        }
        SF_UNROLL
        for (int j = 0; j < 2; ++j) {
            SF_UNROLL
            for (int i1 = 0; i1 < 4; ++i1) gv[j][i1] = act[j] ? (uint32_t)SF_G(sf_step_cell(cell[j], i1)) : 0u;
        }
        SF_RULES_UNROLL
        for (int j = 0; j < 2; ++j) { /* the rules, in slot order */
            const int z = z0 + j;
            const bool actj = j ? act[1] : act[0];
            const int cellj = j ? cell[1] : cell[0];
            const uint32_t pwj = j ? pw[1] : pw[0];
            const uint32_t g0 = j ? gv[1][0] : gv[0][0], g1 = j ? gv[1][1] : gv[0][1];
            const uint32_t g2 = j ? gv[1][2] : gv[0][2], g3 = j ? gv[1][3] : gv[0][3];
            bool go = actj && e.on && !sf_flagged(d, t, env, cellj);
            bool wander = false;
            if (go) {
                /* directions in which a human stands */
                const uint32_t humans = ((g0 & C_S0) ? 1u : 0u) | ((g1 & C_S0) ? 2u : 0u) | ((g2 & C_S0) ? 4u : 0u) | ((g3 & C_S0) ? 8u : 0u);
                wander = humans == 0u;
                SF_NO_UNROLL
                for (int i1 = 0; i1 < 4; ++i1) { /* rare: one copy of the punch, not four */
                    if (!((humans >> i1) & 1u)) continue;
                    const int nc = sf_step_cell(cellj, i1);
                    /* only a human that carries no bullet flag yet is punched: raising the flag tells */
                    const uint32_t fl = e.on ? sf_flag_cell(d, t, env, nc) : 0u;
                    if (fl & SF_FLAG_NEW) {
                        int b = sf_alloc_bullet(k, e);
                        if (b >= 0) {
                            int md = SF_AT(d.z_mind, z); /* Zombie::punch, Character.hpp:838-844 */
                            sf_write_bullet(d, env, b, nc, i1, 1, -1, md > 0 ? md : 0, 0, fl);
                        }
                    }
                }
                wander = wander && e.on;
            }
            /* one draw site: stage 0 = "stay put?" (rand()%5 < 2), stages 1, 2 = the two tries */
            int stage = wander ? 0 : 3;
#pragma unroll 1
            for (int it = 0; it < 3; ++it) {
                if (stage < 3) {
                    int r = sf_rand(e, t);
                    if (stage == 0) {
                        stage = (r % 5 < 2) ? 3 : 1;
                    } else {
                        int i2 = r % 4;
                        int nc = sf_step_cell(cellj, i2);
                        uint32_t gn = i2 == 0 ? g0 : i2 == 1 ? g1 : i2 == 2 ? g2 : g3;
                        stage = stage == 1 ? 2 : 3;
                        if (sf_showit(t.smap[nc], gn, false) == SH_DOT && !sf_flagged(d, t, env, nc)) {
                            uint32_t vnew = C_S1 | (uint32_t)z;
                            SF_G(nc) = (uint16_t)vnew;
                            SF_G(cellj) = (uint16_t)0u;
                            SF_AT(d.z_pos, z) = (uint16_t)((pwj & ~POS_CELL) | (uint32_t)nc);
                            if (j == 0) { /* what the second zombie of the round has loaded already */
                                SF_UNROLL
                                for (int c = 0; c < 4; ++c) {
                                    if (sf_step_cell(cell[1], c) == nc) gv[1][c] = vnew;
                                    if (sf_step_cell(cell[1], c) == cell[0]) gv[1][c] = 0u;
                                }
                            }
                            stage = 3;
                        }
                    }
                }
            }
        }
        SF_SYNCWARP();
    }
}

/* portal_damage, gameplay.hpp:1279-1297: an exit that does not print 'O' radiates -- one that
 * carries a bullet flag (the table), or on which somebody stands (the overlay).  Four exits per
 * round so that their cells load together; exits are distinct cells, so the rounds need no
 * forwarding. */
SF_FN void sf_portal_damage(const SfDev &d, const SfConst &k, const SfTabs &t, int env, SfEnv &e)
{
    /* e.watch: whoever puts a human on an exit cell raises it (zombies never enter one); an arena
     * whose flag is down reads none of its exits' cells, and the flag comes down again when a
     * pass finds nobody on any exit */
    const bool look = e.on && e.watch;
    const int hi = SF_WARP_MAX(e.on ? m2_highest(e.mp) : -1);
    bool any = false;
    for (int i0 = 0; i0 <= hi; i0 += 4) {
        bool lv[4];
        int cell[4];
        uint32_t g[4];
        SF_UNROLL
        for (int j = 0; j < 4; ++j) {
            lv[j] = e.on && i0 + j <= hi && m2_test(e.mp, i0 + j);
            cell[j] = lv[j] ? sf_exit_cell(d, k, env, i0 + j) : 0;
        }
        SF_UNROLL
        for (int j = 0; j < 4; ++j) g[j] = (lv[j] && look) ? (uint32_t)SF_G(cell[j]) : 0u;
        SF_NO_UNROLL
        for (int j = 0; j < 4; ++j) { /* one copy of the look-up and the placement, not four */
            const bool lvj = j == 0 ? lv[0] : j == 1 ? lv[1] : j == 2 ? lv[2] : lv[3];
            const int cj = j == 0 ? cell[0] : j == 1 ? cell[1] : j == 2 ? cell[2] : cell[3];
            const uint32_t gj = j == 0 ? g[0] : j == 1 ? g[1] : j == 2 ? g[2] : g[3];
            if (lvj) {
                const bool stood_on = gj & (C_S0 | C_S1);
                any = any || stood_on;
                if (e.on && (stood_on || sf_flagged(d, t, env, cj))) {
                    int b = sf_alloc_bullet(k, e);
                    if (b >= 0) sf_place_bullet(d, t, env, e, b, cj, 2, 1, -1, 20, -10);
                }
            }
        }
        SF_SYNCWARP();
    }
    if (look) e.watch = any;
}

/* destroy test of one player-built cell, second loop of update_tmp, gameplay.hpp:1356-1373 */
SF_FN void sf_check_built(const SfDev &d, const SfConst &k, int env, SfEnv &e, int cell)
{
    uint32_t g = SF_G(cell);
    int q = sf_built_slot(d, env, e, cell, g);
    if (q >= 0) {
        g = SF_G(cell);
        uint32_t kind = (g >> C_KIND_SHIFT) & 7u;
        int dmg = SF_T(d.t_dmg, q);
        /* destroying a record frees the hint bits too (the occupant byte only if nobody is there) */
        if (kind == K_ENTRANCE && !(g & (C_S0 | C_S1)) && dmg >= 1000) { /* lim_portal */
            int pi = SF_T(d.t_pidx, q);
            int ecell = sf_exit_cell(d, k, env, pi);
            uint32_t ge = SF_G(ecell);
            SF_G(cell) = (uint16_t)(g & ~(C_KIND | C_HINT));
            m2_clear(e.mp, pi);
            sf_remove_built(d, env, e, q);
            int q1 = sf_built_slot(d, env, e, ecell, ge);
            ge = SF_G(ecell);
            SF_G(ecell) = (uint16_t)((ge & (C_S0 | C_S1)) ? (ge & ~(C_KIND | 0xC000u)) : (ge & ~(C_KIND | C_HINT)));
            if (q1 >= 0) sf_remove_built(d, env, e, q1);
        } else if (kind == K_BLOCK && dmg >= 1100) { /* lim_block */
            SF_G(cell) = (uint16_t)(g & ~(C_KIND | C_HINT));
            sf_remove_built(d, env, e, q);
        }
    }
}

/* human_damage, gameplay.hpp:611-634 */
SF_FN void sf_human_damage(const SfDev &d, const SfConst &k, int env, SfEnv &e, int h, int b, int cell, uint32_t g,
                           uint32_t meta)
{
    int dmg = SF_AT(d.b_dmg, b), eff = SF_AT(d.b_eff, b);
    int owner = (int)((meta >> 16) & 0xFFu) - 1;
    int hp = SF_AT(d.h_hp, h) - dmg; /* Character::hit, Character.hpp:242-246 */
    SF_AT(d.h_hp, h) = hp;
    SF_AT(d.h_mind, h) += eff;
    m2_clear(e.mb, b); /* with its owner the cell's bullet flag is gone */
    uint32_t team_h = SF_AT(d.h_sel, h) & HS_TEAM;
    uint32_t team_o = owner >= 0 ? (SF_AT(d.h_sel, owner) & HS_TEAM) : 0u;
    uint32_t team_me = SF_AT(d.h_sel, k.ind) & HS_TEAM;
    if (owner >= 0 && team_h != team_o) {
        SF_AT(d.h_dmg, owner) += dmg;
        SF_AT(d.h_eff, owner) += eff;
    }
    if (hp <= 0) {
        e.mh &= ~(1ull << h);
        if (h != k.ind) { /* the own corpse keeps its cell, gameplay.hpp:642-645 */
            SF_G(cell) = (uint16_t)(g & ~(C_S0 | C_OCC));
            SF_AT(d.h_sel, h) = (uint16_t)(SF_AT(d.h_sel, h) & ~HS_AGENT); /* deleteAgent, :648-649 */
        }
        if (owner >= 0 && team_o == team_me && team_h != team_me) {
            e.tkills += 1, e.loot += 100;
            if (owner == k.ind) e.loot += 900, e.kills += 1;
        }
        if (owner >= 0 && team_h != team_o) SF_AT(d.h_kills, owner) += 1;
    }
}

/* zombie_damage, gameplay.hpp:574-598 */
SF_FN void sf_zombie_damage(const SfDev &d, const SfConst &k, int env, SfEnv &e, int z, int b, int cell, uint32_t g,
                            uint32_t meta)
{
    int dmg = SF_AT(d.b_dmg, b), eff = SF_AT(d.b_eff, b);
    int owner = (int)((meta >> 16) & 0xFFu) - 1;
    int hp = SF_AT(d.z_hp, z) - dmg;
    SF_AT(d.z_hp, z) = hp;
    SF_AT(d.z_mind, z) += eff;
    m2_clear(e.mb, b);
    if (owner >= 0) {
        SF_AT(d.h_dmg, owner) += dmg;
        SF_AT(d.h_eff, owner) += eff;
    }
    if (hp <= 0) {
        m2_clear(e.mz, z);
        SF_G(cell) = (uint16_t)(g & ~(C_S1 | C_OCC));
        if (owner >= 0 && (SF_AT(d.h_sel, owner) & HS_TEAM) == (SF_AT(d.h_sel, k.ind) & HS_TEAM)) {
            int pts = 500 + 250 * (int)(SF_AT(d.z_pos, z) >> POS_HI_SHIFT);
            e.tkills += 1, e.loot += pts / 10;
            if (owner == k.ind) e.loot += pts * 9 / 10, e.kills += 1;
        }
        if (owner >= 0) SF_AT(d.h_kills, owner) += 1;
    }
}

/* update_tmp + hit_human + hit_zombie, gameplay.hpp:1343-1381, 600-609, 636-652, in ONE walk over
 * the bullets (four per round: flags and positions, then cells, load together).
 *
 * update_tmp: a bullet standing on a player-built block, or on a player-built entrance that no
 * human hides, is absorbed (the cell's dmg grows); then the touched cells are tested against
 * lim_block / lim_portal.  Absorbing cells hold no human or zombie, so this never interferes
 * with the hits.
 * hit_human / hit_zombie: the reference walks every live human / zombie and tests s[2] of its
 * cell; a set s[2] always has exactly one owning bullet, so walking the owning bullets and
 * looking at who stands in their cell visits the same (victim, bullet) pairs, which are
 * independent of each other (distinct victims, distinct bullets, credits are sums).
 * Finally the bullet flags of all cells are dropped (the table is wiped; the BF_OWNS bits go as
 * the bullets move on): that is the themap1 snapshot of update_bull (:1061-1072, "s[2] = 0 on the
 * current cell of every live bullet"), which nothing reads in between.  After this walk no cell
 * has s[2] set. */
SF_FN void sf_resolve_bullets(const SfDev &d, const SfConst &k, const SfTabs &t, int env, SfEnv &e)
{
#ifdef SF_DEBUG_HIST
    if (e.on) sf_dbg_hist[sf_bt_at(t, SF_BT_SLOTS) < 255 ? sf_bt_at(t, SF_BT_SLOTS) : 255] += 1;
#endif
    const uint64_t quitters = e.on ? (e.quit & e.mh) : 0ull; /* Hp <= 0 by '_': removed, never hit (:640-645) */
    e.quit = 0;
    const bool built_any = e.ntemp != 0;
    int hc0 = 0, hc1 = 0, hc2 = 0, hc3 = 0; /* cells that absorbed a bullet in this call */
    int n_hit = 0;
    const int hi = SF_WARP_MAX(e.on ? m2_highest(e.mb) : -1);
    /* liveness is tested against a snapshot of the mask (every slot is visited once), and the
     * flags / positions of a round are loaded one round ahead, so that they are in flight
     * together with the cell loads of the round before */
    const uint64_t live0 = e.on ? e.mb[0] : 0ull, live1 = e.on ? e.mb[1] : 0ull;
    uint32_t meta_n[4], pw_n[4];
    SF_UNROLL
    for (int j = 0; j < 4; ++j) {
        bool ln = j <= hi && (((j < 64 ? live0 : live1) >> (j & 63)) & 1);
        meta_n[j] = ln ? SF_AT(d.b_meta, j) : 0u;
        pw_n[j] = ln ? (uint32_t)SF_AT(d.b_pw, j) : 0u;
    }
    for (int b0 = 0; b0 <= hi; b0 += 4) {
        bool lv[4];
        uint32_t meta[4], g[4];
        int cell[4];
        SF_UNROLL
        for (int j = 0; j < 4; ++j) {
            const int b = b0 + j;
            lv[j] = b <= hi && (((b < 64 ? live0 : live1) >> (b & 63)) & 1);
            meta[j] = meta_n[j];
            cell[j] = (int)(pw_n[j] & POS_CELL);
        }
        SF_UNROLL
        for (int j = 0; j < 4; ++j) {
            const int b = b0 + 4 + j;
            bool ln = b <= hi && (((b < 64 ? live0 : live1) >> (b & 63)) & 1);
            meta_n[j] = ln ? SF_AT(d.b_meta, b) : 0u;
            pw_n[j] = ln ? (uint32_t)SF_AT(d.b_pw, b) : 0u;
        }
        SF_UNROLL
        for (int j = 0; j < 4; ++j) {
            bool need = lv[j] && (built_any || (meta[j] & BF_OWNS));
            g[j] = need ? (uint32_t)SF_G(cell[j]) : 0u;
        }
        SF_RULES_UNROLL
        for (int j = 0; j < 4; ++j) { /* the rules, in slot order */
            const bool lvj = j == 0 ? lv[0] : j == 1 ? lv[1] : j == 2 ? lv[2] : lv[3];
            if (lvj) {
                const int b = b0 + j;
                const uint32_t mj = j == 0 ? meta[0] : j == 1 ? meta[1] : j == 2 ? meta[2] : meta[3];
                const int cj = j == 0 ? cell[0] : j == 1 ? cell[1] : j == 2 ? cell[2] : cell[3];
                uint32_t gj = j == 0 ? g[0] : j == 1 ? g[1] : j == 2 ? g[2] : g[3];
                if ((mj & (BF_OWNS | BF_SPILL)) == (BF_OWNS | BF_SPILL)) { /* its flag is in the overlay: take it down */
                    gj &= ~C_S2;
                    SF_G(cj) = (uint16_t)gj;
                }
                uint32_t kind = (gj >> C_KIND_SHIFT) & 7u;
                if (built_any && (kind == K_BLOCK || (kind == K_ENTRANCE && !(gj & (C_S0 | C_S1))))) {
                    int q = sf_built_slot(d, env, e, cj, gj);
                    SF_T(d.t_dmg, q) += SF_AT(d.b_dmg, b);
                    m2_clear(e.mb, b);
                    if (n_hit == 0) hc0 = cj;
                    else if (n_hit == 1) hc1 = cj;
                    else if (n_hit == 2) hc2 = cj;
                    else if (n_hit == 3) hc3 = cj;
                    n_hit += 1;
                } else if (mj & BF_OWNS) {
                    int occ = (int)(gj & C_OCC);
                    if ((gj & C_S0) && ((e.mh >> occ) & 1) && !((quitters >> occ) & 1)) {
                        sf_human_damage(d, k, env, e, occ, b, cj, gj, mj);
                    } else if (gj & C_S1) {
                        sf_zombie_damage(d, k, env, e, occ, b, cj, gj, mj);
                    }
                }
            }
        }
        SF_SYNCWARP();
    }
    sf_bt_wipe(t);
    /* a limit can only be crossed by an absorption of this very call (while a human hides an
     * entrance nothing is absorbed, :1349), so only the cells touched above need the test */
    if (n_hit > 4) {
        for (int q = (int)e.ntemp - 1; q >= 0; --q)
            if (q < (int)e.ntemp) sf_check_built(d, k, env, e, SF_T(d.t_cell, q));
    } else {
#pragma unroll 1
        for (int i = 0; i < 4; ++i)
            if (i < n_hit) sf_check_built(d, k, env, e, i == 0 ? hc0 : i == 1 ? hc1 : i == 2 ? hc2 : hc3);
    }
    SF_SYNCWARP();
    uint64_t q = quitters;
    const int nq = SF_WARP_MAX(sf_popc64(q));
    for (int i = 0; i < nq; ++i) {
        if (q) {
            int h = sf_ffs64(q);
            q &= q - 1;
            e.mh &= ~(1ull << h);
            if (h != k.ind) {
                int cell = (int)(SF_AT(d.h_pw, h) & POS_CELL);
                SF_G(cell) = (uint16_t)(SF_G(cell) & ~(C_S0 | C_OCC));
                SF_AT(d.h_sel, h) = (uint16_t)(SF_AT(d.h_sel, h) & ~HS_AGENT);
            }
        }
        SF_SYNCWARP();
    }
}

/* update_bull, gameplay.hpp:1059-1100, plus the harness's out-of-bounds guard.  The snapshot
 * half (s[2] cleared under every live bullet) was done by sf_resolve_bullets; here the bullets
 * move, walked in the REVERSE of the reference's order so that the first bullet to reach a cell
 * is the reference's last writer of it.  Whether a bullet may enter the cell ahead is decided by
 * the static map alone, except on a staircase (which lets a bullet in only while somebody stands
 * on it): a player-built block or entrance prints '#' / '^' but is "built" and takes the bullet,
 * so the cell itself is read for staircases only.  The flag raised at the new cell goes into the
 * table (empty since sf_resolve_bullets): a cell found there already has its last writer. */
SF_FN void sf_update_bull(const SfDev &d, const SfTabs &t, int env, SfEnv &e)
{
    const int hi = SF_WARP_MAX(e.on ? m2_highest(e.mb) : -1);
    int r = 0;
    if (e.on) r = sf_rand(e, t) & 1;
    SF_SYNCWARP();
    bool oob = false;
    /* reference order: r == 1 ascending, r == 0 descending (:1073-1076); walk the opposite way */
    const uint64_t live0 = e.on ? e.mb[0] : 0ull, live1 = e.on ? e.mb[1] : 0ull; /* snapshot: each slot is visited once */
    uint32_t pw_n[4], meta_n[4]; /* loaded one round ahead */
    SF_UNROLL
    for (int j = 0; j < 4; ++j) {
        const int bn = r ? hi - j : j;
        bool ln = j <= hi && (((bn < 64 ? live0 : live1) >> (bn & 63)) & 1);
        pw_n[j] = ln ? (uint32_t)SF_AT(d.b_pw, bn) : 0u;
        meta_n[j] = ln ? SF_AT(d.b_meta, bn) : 0u;
    }
    for (int i0 = 0; i0 <= hi; i0 += 4) {
        bool lv[4];
        int b[4], nc[4];
        uint32_t pw[4], meta[4], gn[4], st[4];
        SF_UNROLL
        for (int j = 0; j < 4; ++j) {
            b[j] = r ? hi - (i0 + j) : i0 + j;
            lv[j] = i0 + j <= hi && (((b[j] < 64 ? live0 : live1) >> (b[j] & 63)) & 1);
            pw[j] = pw_n[j];
            meta[j] = meta_n[j] & ~(BF_OWNS | BF_SPILL);
        }
        SF_UNROLL
        for (int j = 0; j < 4; ++j) {
            const int bn = r ? hi - (i0 + 4 + j) : i0 + 4 + j;
            bool ln = i0 + 4 + j <= hi && (((bn < 64 ? live0 : live1) >> (bn & 63)) & 1);
            pw_n[j] = ln ? (uint32_t)SF_AT(d.b_pw, bn) : 0u;
            meta_n[j] = ln ? SF_AT(d.b_meta, bn) : 0u;
        }
        SF_UNROLL
        for (int j = 0; j < 4; ++j) {
            nc[j] = 0;
            if (lv[j] && !sf_neighbour((int)(pw[j] & POS_CELL), (int)(pw[j] >> POS_HI_SHIFT), &nc[j])) {
                oob = true; /* the reference would read themap[i][-1][k], :1069 */
                lv[j] = false;
            }
            bool expired = ((meta[j] >> 8) & 0xFFu) + 1 >= (meta[j] & 0xFFu); /* Bullet::expire, Item.hpp:165-168 */
            if (lv[j] && expired) {
                m2_clear(e.mb, b[j]);
                lv[j] = false;
            }
            st[j] = lv[j] ? (uint32_t)t.smap[nc[j]] : 0u;
            gn[j] = (st[j] & (M_UP | M_DOWN)) ? (uint32_t)SF_G(nc[j]) : 0u;
        }
        SF_RULES_UNROLL
        for (int j = 0; j < 4; ++j) { /* the moves, in walk order */
            const bool lvj = j == 0 ? lv[0] : j == 1 ? lv[1] : j == 2 ? lv[2] : lv[3];
            if (lvj) {
                const uint32_t stj = j == 0 ? st[0] : j == 1 ? st[1] : j == 2 ? st[2] : st[3];
                const uint32_t gj = j == 0 ? gn[0] : j == 1 ? gn[1] : j == 2 ? gn[2] : gn[3];
                const int bj = j == 0 ? b[0] : j == 1 ? b[1] : j == 2 ? b[2] : b[3];
                /* showit() is neither '#' nor '^' / 'v', or the cell is player-built (:1080-1083) */
                if (!(stj & M_WALL) && (!(stj & (M_UP | M_DOWN)) || (gj & (C_S0 | C_S1)))) {
                    const int ncj = j == 0 ? nc[0] : j == 1 ? nc[1] : j == 2 ? nc[2] : nc[3];
                    const uint32_t pwj = j == 0 ? pw[0] : j == 1 ? pw[1] : j == 2 ? pw[2] : pw[3];
                    uint32_t m = j == 0 ? meta[0] : j == 1 ? meta[1] : j == 2 ? meta[2] : meta[3];
                    const uint32_t fl = sf_flag_cell(d, t, env, ncj);
                    if (fl & SF_FLAG_NEW) m |= BF_OWNS | (fl & BF_SPILL);
                    SF_AT(d.b_pw, bj) = (uint16_t)((pwj & ~POS_CELL) | (uint32_t)ncj);
                    SF_AT(d.b_meta, bj) = m + 0x100u;
                } else {
                    m2_clear(e.mb, bj);
                }
            }
        }
        SF_SYNCWARP();
    }
    if (oob) sf_fail_env(e, SF_UB_GUARD);
}

/* human_rnpc_bot, gameplay.hpp:1927-1940; returns the command symbol.  Written as a chain of
 * "does this lane still need a draw" steps so that the lanes of a warp stay together. */
SF_FN int sf_rnpc_bot(const SfTabs &t, SfEnv &e, bool want)
{
    /* the key rows of the reference, eight symbols to a 64-bit constant */
    const uint64_t weapons = 0x2f2e2c6d6e627663ull; /* "cvbnm,./" */
    const uint64_t moves = 0x0070647377613231ull;   /* "12awsdp"  */
    const uint64_t others = 0x5d5b6a686766752bull;  /* "+ufghj[]" */
    int c = '+';
    /* stage 0: rand()%5 < 3 -> 'x'; 1: rand()%5 < 3 -> moves; 2: pick from a row; 3: weapon key; 4: done */
    int stage = want ? ((e.frame % 50 <= 1) ? 3 : 0) : 4;
    bool second = false;
#pragma unroll 1
    for (int it = 0; it < 3; ++it) {
        if (stage < 4) {
            int r = sf_rand(e, t);
            if (stage == 3) {
                c = (int)((weapons >> (8 * (r % 8))) & 0xFFu);
                stage = 4;
            } else if (stage == 0) {
                if (r % 5 < 3) c = 'x', stage = 4;
                else stage = 1;
            } else if (stage == 1) {
                second = r % 5 < 3;
                stage = 2;
            } else {
                c = second ? (int)((moves >> (8 * (r % 7))) & 0xFFu) : (int)((others >> (8 * (r % 8))) & 0xFFu);
                stage = 4;
            }
        }
    }
    return c;
}

/* index of a selection key in its row, -1 if c is not in it (obey, gameplay.hpp:759-791) */
SF_FN int sf_key_index(int c, int group)
{
    if (group == 0) return c == 'f' ? 0 : c == 'g' ? 1 : c == 'h' ? 2 : c == 'j' ? 3 : -1;
    if (group == 1) return c == 'k' ? 0 : c == 'l' ? 1 : c == ';' ? 2 : c == '\'' ? 3 : -1;
    return c == 'c' ? 0 : c == 'v' ? 1 : c == 'b' ? 2 : c == 'n' ? 3 : c == 'm' ? 4 : c == ',' ? 5
         : c == '.' ? 6 : c == '/' ? 7 : -1;
}

/* obey + teleport + claim_chest for one human, gameplay.hpp:695-821, 517-530, 507-515.
 * Everything a command can need -- the human's own cell, the one cell it can act on (ahead
 * for '[' ']' 'z' 'x', in the walking direction for 'a' 's' 'd' 'w'), and its selection, stamina
 * and mindamage when it fires or consumes -- is loaded up front in one round of independent
 * loads; the rules then run on registers. */
SF_FN void sf_obey(const SfDev &d, const SfConst &k, const SfTabs &t, int env, SfEnv &e, int h, int c, uint32_t pw,
                   uint32_t sel)
{
    int cell = (int)(pw & POS_CELL);
    int way0 = (int)(pw >> POS_HI_SHIFT);
    const bool acts_ahead = c == '[' || c == ']' || c == 'z' || c == 'x';
    const bool walks = c == 'a' || c == 's' || c == 'd' || c == 'w';
    const int dir = acts_ahead ? way0 : c == 's' ? 0 : c == 'd' ? 1 : c == 'w' ? 2 : 3;
    int nc = cell;
    const bool inb = (acts_ahead || walks) && sf_neighbour(cell, dir, &nc);
    const bool uses_kit = c == 'x' || c == 'z' || c == 'u';
    /* the human's own cell matters only if it leaves it, or waits on a player-built entrance
       (HS_ON_ENT); a human that stays put stands on nothing it could claim or enter */
    bool have_g = walks || (sel & HS_ON_ENT);
    uint32_t g = have_g ? (uint32_t)SF_G(cell) : 0u;
    /* the cell acted on: a punch / shot / throw is stopped by the static map alone, except on a
       staircase (free only while somebody stands on it; see sf_update_bull) */
    const uint32_t stn = inb ? (uint32_t)t.smap[nc] : 0u;
    const bool fires = c == 'z' || c == 'x';
    uint32_t gn = (inb && (!fires || (stn & (M_UP | M_DOWN)))) ? (uint32_t)SF_G(nc) : 0u;
    int st = uses_kit ? SF_AT(d.h_stam, h) : 0;
    int md = uses_kit ? SF_AT(d.h_mind, h) : 0;
    const int vec = (int)((sel >> HS_VEC_SHIFT) & 3u) - 1, ind = (int)((sel >> HS_IND_SHIFT) & 15u) - 1;
    if (c == '_') {
        SF_AT(d.h_hp, h) = 0;
        e.quit |= 1ull << h;
    } else if (c == '[' || c == ']') {
        if (inb && sf_showit(stn, gn, false) == SH_DOT && !sf_flagged(d, t, env, nc)) {
            uint32_t bp = SF_AT(d.h_bp, h);
            uint32_t blocks = bp & 0xFFu, portals = (bp >> 8) & 0xFFu, pend = (bp >> 16) & 0xFFu;
            if (c == '[') {
                if (blocks && sf_push_built(d, k, env, e, nc, 0)) {
                    SF_G(nc) = (uint16_t)((K_BLOCK << C_KIND_SHIFT) | sf_hint_bits((int)e.ntemp - 1));
                    SF_AT(d.h_bp, h) = bp - 1u;
                }
            } else if (pend) { /* second press: the entrance bound to the pending exit */
                if (sf_push_built(d, k, env, e, nc, (int)pend - 1)) {
                    SF_G(nc) = (uint16_t)((K_ENTRANCE << C_KIND_SHIFT) | sf_hint_bits((int)e.ntemp - 1));
                    SF_AT(d.h_bp, h) = bp & ~0xFF0000u;
                }
            } else if (portals) { /* first press: the exit, lowest free portal slot (p_ind) */
                int pi = m2_lowest_free(e.mp);
                if (pi >= k.cap_p) sf_fail_env(e, SF_OVERFLOW);
                else if (sf_push_built(d, k, env, e, nc, 0)) {
                    SF_G(nc) = (uint16_t)((K_EXIT << C_KIND_SHIFT) | sf_hint_bits((int)e.ntemp - 1));
                    SF_AT(d.p_cell, pi) = (uint16_t)nc;
                    m2_set(e.mp, pi);
                    SF_AT(d.h_bp, h) = (bp - 0x100u) | ((uint32_t)(pi + 1) << 16);
                }
            }
        }
    } else if (c == 'q' || c == 'e') { /* turn_l: way+1, turn_r: way-1, Character.hpp:745-759 */
        way0 = (c == 'e') ? ((way0 + 3) & 3) : ((way0 + 1) & 3);
        SF_AT(d.h_pw, h) = (uint16_t)((uint32_t)cell | ((uint32_t)way0 << POS_HI_SHIFT));
    } else if (walks) {
        if (inb) {
            /* '*' hides a chest, an exit or the floor: only for the exit does the flag matter */
            int sit = sf_showit(stn, gn, false);
            if (sit == SH_CHEST || sit == SH_UP || sit == SH_DOWN || sit == SH_DOT ||
                (sit == SH_EXIT && sf_flagged(d, t, env, nc))) {
                gn = (gn & ~C_OCC) | C_S0 | (uint32_t)h;
                SF_G(nc) = (uint16_t)gn;
                if (sf_is_exit(t, nc, gn)) e.watch = true; /* an exit under a bullet prints '*' */
                SF_G(cell) = (uint16_t)(g & ~(C_S0 | C_OCC));
                cell = nc;
                g = gn;
                SF_AT(d.h_pw, h) = (uint16_t)((uint32_t)cell | ((uint32_t)way0 << POS_HI_SHIFT));
            }
        }
    } else if (c == 'u') { /* Human::use, Character.hpp:379-389 */
        if (vec == 0) {
            uint32_t cp = SF_AT(d.h_cons, h);
            uint32_t cnt = (cp >> (8 * ind)) & 0xFFu;
            if (cnt >= 1) {
                SF_AT(d.h_stam, h) = st + k.cons[ind].stamina;
                SF_AT(d.h_hp, h) += k.cons[ind].hp;
                SF_AT(d.h_mind, h) = md + k.cons[ind].effect;
                SF_AT(d.h_cons, h) = cp - (1u << (8 * ind));
                if (cnt - 1 < 1) SF_AT(d.h_sel, h) = (uint16_t)(sel &= ~(3u << HS_VEC_SHIFT)); /* vec = -1 */
            }
        }
    } else if (c == 'z' || c == 'x') {
        int b = m2_lowest_free(e.mb); /* b_ind() comes first, :800 */
        if (inb) {
            bool can = false;
            int dmg = 0, eff = 0, range = 1;
            if (c == 'z') { /* Human::punch, Character.hpp:391-397 */
                int pb = sf_punch_base(k, e, h);
                dmg = pb > md ? pb : md;
                can = true;
            } else if (vec == 1) { /* Human::throw_it, Character.hpp:410-427 */
                const SfWpn w = sf_tmpl(k, h).thr[ind];
                dmg = w.damage > w.damage + md ? w.damage : w.damage + md;
                eff = w.effect, range = w.range;
                if (st + w.stamina >= 0) {
                    uint32_t tp = SF_AT(d.h_thr, h);
                    uint32_t cnt = (tp >> (8 * ind)) & 0xFFu;
                    if (cnt < 1) {
                        SF_AT(d.h_sel, h) = (uint16_t)(sel &= ~(3u << HS_VEC_SHIFT));
                    } else {
                        SF_AT(d.h_stam, h) = st + w.stamina;
                        SF_AT(d.h_thr, h) = tp - (1u << (8 * ind));
                        if (cnt - 1 < 1) SF_AT(d.h_sel, h) = (uint16_t)(sel &= ~(3u << HS_VEC_SHIFT));
                        can = true;
                    }
                }
            } else if (vec == 2) { /* Human::shot_it, Character.hpp:399-408 */
                const SfTemplate &tp = sf_tmpl(k, h);
                const SfWpn w = tp.wpn[ind];
                if (st + w.stamina >= 0) {
                    int sb = tp.shot_base[ind];
                    SF_AT(d.h_stam, h) = st + w.stamina;
                    dmg = sb > w.damage + md ? sb : w.damage + md;
                    eff = w.effect, range = w.range;
                    can = true;
                }
            }
            if (can) {
                if (!(stn & M_WALL) && (!(stn & (M_UP | M_DOWN)) || (gn & (C_S0 | C_S1)))) {
                    if (b >= k.cap_b) sf_fail_env(e, SF_OVERFLOW);
                    else {
                        m2_set(e.mb, b);
                        sf_place_bullet(d, t, env, e, b, nc, way0, range, h, dmg, eff);
                    }
                }
            }
        }
    } else {
        int i;
        if ((i = sf_key_index(c, 0)) >= 0) {
            if ((SF_AT(d.h_cons, h) >> (8 * i)) & 0xFFu) {
                uint32_t s4 = sel & HS_KEEP;
                SF_AT(d.h_sel, h) = (uint16_t)(sel = s4 | (1u << HS_VEC_SHIFT) | ((uint32_t)(i + 1) << HS_IND_SHIFT));
            }
        } else if ((i = sf_key_index(c, 1)) >= 0) {
            if ((SF_AT(d.h_thr, h) >> (8 * i)) & 0xFFu) {
                uint32_t s4 = sel & HS_KEEP;
                SF_AT(d.h_sel, h) = (uint16_t)(sel = s4 | (2u << HS_VEC_SHIFT) | ((uint32_t)(i + 1) << HS_IND_SHIFT));
            }
        } else if ((i = sf_key_index(c, 2)) >= 0) {
            if ((sf_tmpl(k, h).w_owned >> i) & 1u) {
                uint32_t s4 = sel & HS_KEEP;
                SF_AT(d.h_sel, h) = (uint16_t)(sel = s4 | (3u << HS_VEC_SHIFT) | ((uint32_t)(i + 1) << HS_IND_SHIFT));
            }
        }
    }
    if (e.on) {
        /* teleport, gameplay.hpp:517-530 (g is the current content of the human's cell) */
        uint32_t stc = t.smap[cell];
        int pidx = -1;
        if (stc & (M_UP | M_DOWN)) pidx = (int)(stc >> M_TARGET_SHIFT);
        else if (((g >> C_KIND_SHIFT) & 7u) == K_ENTRANCE) pidx = SF_T(d.t_pidx, sf_find_built(d, env, e, cell));
        if (pidx >= 0) {
            int dc = sf_exit_cell(d, k, env, pidx);
            uint32_t gd = SF_G(dc);
            if (sf_showit(t.smap[dc], gd, false) == SH_EXIT && !sf_flagged(d, t, env, dc)) {
                if (!have_g) g = SF_G(cell), have_g = true;
                gd = (gd & ~C_OCC) | C_S0 | (uint32_t)h;
                e.watch = true;
                SF_G(dc) = (uint16_t)gd;
                SF_G(cell) = (uint16_t)(g & ~(C_S0 | C_OCC));
                cell = dc;
                g = gd;
                SF_AT(d.h_pw, h) = (uint16_t)((uint32_t)cell | ((uint32_t)way0 << POS_HI_SHIFT));
            }
        }
        /* claim_chest, gameplay.hpp:507-515, Human::claim_chest Character.hpp:372-377 */
        uint32_t kind = (g >> C_KIND_SHIFT) & 7u;
        if (kind >= K_CHEST0 && kind < K_BLOCK) {
            int ty = (int)kind - K_CHEST0;
            SF_AT(d.h_stam, h) += k.cons[ty].stamina;
            SF_AT(d.h_hp, h) += k.cons[ty].hp;
            SF_AT(d.h_mind, h) += k.cons[ty].effect;
            SF_G(cell) = (uint16_t)(g & ~C_KIND);
            e.chest -= 1;
        }
        if (have_g) { /* still on a player-built entrance: its exit was taken, try again next step */
            const uint32_t ent = kind == K_ENTRANCE ? HS_ON_ENT : 0u;
            if (ent != (sel & HS_ON_ENT)) SF_AT(d.h_sel, h) = (uint16_t)(sel ^ HS_ON_ENT);
        }
    }
}

/* human_action, gameplay.hpp:965-1012.  actions = this arena's row of the action buffer:
 * [ind] the player's command (get_my_action, :939-963; ind = 0 outside Battle Royale), the other
 * entries what bot() returns for the agent-driven squad humans (bots/bot-0.5/Custom.hpp:137-158, one
 * of "+xzqeawsd") or, in Battle Royale, what the other players sent. */
SF_FN void sf_human_action(const SfDev &d, const SfConst &k, const SfTabs &t, int env, SfEnv &e,
                           const uint8_t *actions)
{
    /* commands wait in h_cmd between the two loops (command[], gameplay.hpp:43) */
    const uint64_t live = e.on ? e.mh : 0ull;
    const int hi = SF_WARP_MAX(live ? sf_fls64(live) : -1);
    const int ind = k.ind;
    const int cmd0 = (actions && e.on) ? actions[ind] : '+';
    for (int h = 0; h <= hi; ++h) {
        if (h == ind) continue; /* command[ind] is the player's own, set before human_action (:956-961) */
        bool is_live = (live >> h) & 1;
        uint32_t sel = is_live ? SF_AT(d.h_sel, h) : 0u;
        int c = sf_rnpc_bot(t, e, is_live && (sel & HS_RNPC));
        if (is_live && !(sel & HS_RNPC)) {
            c = '+';
            if (k.mode == SF_MODE_ROYALE && h < k.n_players && actions) {
                c = actions[h]; /* a remote player's command arrives as sent (recieve(), gameplay.hpp:977-986) */
            } else if ((sel & HS_AGENT) && h < k.n_agents && actions) {
                c = actions[h];
                bool ok = c == '+' || c == 'x' || c == 'z' || c == 'q' || c == 'e' || c == 'a' || c == 'w' ||
                          c == 's' || c == 'd';
                if (!ok) c = '+';
            }
        }
        if (is_live) SF_AT(d.h_cmd, h) = (uint8_t)c;
        SF_SYNCWARP();
    }
    int r = 0;
    if (e.on) r = sf_rand(e, t) & 1;
    SF_SYNCWARP();
    /* a human's position and command are loaded one iteration ahead (nobody else writes them) */
    uint32_t pw_n = 0, sel_n = 0;
    int c_n = '+';
    {
        int h = r ? 0 : hi;
        if (hi >= 0 && ((live >> h) & 1))
            pw_n = SF_AT(d.h_pw, h), sel_n = SF_AT(d.h_sel, h), c_n = h == ind ? cmd0 : (int)SF_AT(d.h_cmd, h);
    }
    for (int i = 0; i <= hi; ++i) {
        const int h = r ? i : hi - i;
        const uint32_t pw = pw_n, sel = sel_n;
        const int c = c_n;
        if (i < hi) {
            int hn = r ? i + 1 : hi - i - 1;
            if ((live >> hn) & 1)
                pw_n = SF_AT(d.h_pw, hn), sel_n = SF_AT(d.h_sel, hn), c_n = hn == ind ? cmd0 : (int)SF_AT(d.h_cmd, hn);
        }
        if (e.on && ((live >> h) & 1)) sf_obey(d, k, t, env, e, h, c, pw, sel);
        SF_SYNCWARP();
    }
}

/* ------------------------------------------------------------------ reset */

/* one arena's overlay is 19,968 bytes, a multiple of 64 and 64-byte aligned */
SF_FN void sf_clear_grid(uint16_t *g)
{
#ifdef __CUDA_ARCH__
    uint4 *p = reinterpret_cast<uint4 *>(g);
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    for (int i = 0; i < SF_GRID_STRIDE / 8; ++i) p[i] = zero;
#else
    for (int i = 0; i < SF_GRID_STRIDE; ++i) g[i] = 0;
#endif
}

/* load_data(), online branch (gameplay.hpp:1847-1859): in index order every player draws
 * way = rand() % 4 + 1, then cells until one prints '.' */
SF_FN void sf_royale_place(const SfDev &d, const SfConst &k, const SfTabs &t, int env, SfEnv &e)
{
    /* one draw site: stage 0 = way, 1..3 = floor, row, column of the next try */
    int i = 0, stage = 0, way0 = 0, f = 0, r = 0;
#pragma unroll 1
    while (i < k.n_players) {
        const int v = sf_rand(e, t);
        if (stage == 0) way0 = v % 4, stage = 1;
        else if (stage == 1) f = v % SF_FLOORS, stage = 2;
        else if (stage == 2) r = v % SF_ROWS, stage = 3;
        else {
            const int cell = sf_cell_of(f, r, v % SF_COLS);
            stage = 1;
            if (sf_showit(t.smap[cell], SF_G(cell), false) == SH_DOT) { /* no bullets yet */
                sf_init_human(d, env, k.players[i], i, cell, false, k.teams[i], true);
                SF_AT(d.h_pw, i) = (uint16_t)((uint32_t)cell | ((uint32_t)way0 << POS_HI_SHIFT));
                SF_G(cell) = (uint16_t)(C_S0 | (uint32_t)i);
                ++i, stage = 0;
            }
        }
    }
}

/* setup() + load_data() + _srand, gameplay.hpp:1231-1277, 1741-1747, 1861-1920; the harness
 * then does "++frame" (play(), :1441) */
SF_FN void sf_reset_env(const SfDev &d, const SfConst &k, const SfTabs &t, int env, SfEnv &e)
{
    sf_clear_grid(d.grid + (size_t)env * SF_GRID_STRIDE);
    int64_t ge = k.env_id_base + env;
    e.level = k.level_min + (int)(ge % k.level_span);
    e.frame = 1;
    e.steps = 0;
    e.kills = e.tkills = e.loot = e.chest = 0;
    e.ntemp = 0;
    e.status = SF_RUNNING;
    e.on = true;
    e.watch = true; /* until the first look */
    e.quit = 0;
    e.mz[0] = e.mz[1] = e.mb[0] = e.mb[1] = 0;
    e.mp[0] = (1ull << k.n_static_exits) - 1ull;
    e.mp[1] = 0;
    if (k.mode == SF_MODE_SQUAD) {
        int c0 = sf_cell_of(0, 3, 1);
        sf_init_human(d, env, k.players[0], 0, c0, false, 1, true);
        SF_G(c0) = (uint16_t)(C_S0 | 0u);
        for (int i = 1; i < 10; ++i) {
            int c = i < 5 ? sf_cell_of(0, 1, i + 1) : sf_cell_of(2, 1, i + 1);
            sf_init_human(d, env, k.npc, i, c, false, i < 5 ? 1 : 2, k.squad_agents != 0);
            SF_G(c) = (uint16_t)(C_S0 | (uint32_t)i);
        }
        e.mh = 0x3FFull;
        e.hw_h = 10;
    } else if (k.mode == SF_MODE_ROYALE) {
        e.level = 1; /* gameplay.hpp:1641, 1659 */
        e.mh = (1ull << k.n_players) - 1ull;
        e.hw_h = k.n_players;
    } else {
        int c0 = sf_cell_of(0, 1, 1);
        sf_init_human(d, env, k.players[0], 0, c0, false, 1, true);
        SF_G(c0) = (uint16_t)(C_S0 | 0u);
        e.mh = 1ull;
        e.hw_h = 1;
    }
    /* the stream of this episode was seeded as the pending one; the next episode's follows */
    sf_install_stream(d, t, env, e, sf_synth_tb(ge), sf_synth_serial(ge, (int64_t)e.episode + 1));
    if (k.mode == SF_MODE_ROYALE) sf_royale_place(d, k, t, env, e);
}

/* ------------------------------------------------------------------ the step */

/* check_end(), gameplay.hpp:1102-1229, as restated by the harness (eval_end): evaluated at the
 * end of the step, wall clock replaced by the frame clock (level * 300 s = level * 7500 frames) */
SF_FN void sf_eval_end(const SfDev &d, const SfConst &k, int env, SfEnv &e)
{
    if (e.on) {
        bool rivals = false; /* rivals_are_dead, gameplay.hpp:497-505 */
        if (k.mode == SF_MODE_ROYALE) {
            uint32_t me = SF_AT(d.h_sel, k.ind) & HS_TEAM;
            for (uint64_t m = e.mh; m; m &= m - 1) {
                uint32_t tm = SF_AT(d.h_sel, sf_ffs64(m)) & HS_TEAM;
                if (tm && tm != me) rivals = true;
            }
        }
        if (k.mode == SF_MODE_ROYALE && !rivals) {
            e.status = SF_WIN; /* "online && rivals_are_dead()" is the first test of check_end(), :1103 */
        } else if (SF_AT(d.h_hp, k.ind) <= 0) {
            e.status = SF_DEAD;
        } else if (k.mode == SF_MODE_ROYALE) {
            /* an online match ends in no other way */
        } else if (k.mode == SF_MODE_TIMER) {
            if ((int64_t)e.frame >= (int64_t)e.level * 7500) e.status = (e.kills < e.level * 5) ? SF_TIMEOUT : SF_WIN;
        } else if (k.mode == SF_MODE_SOLO) {
            if (e.level * 5 <= e.kills) e.status = SF_WIN;
        } else if (e.level * 10 <= e.tkills) {
            /* rivals_are_dead, gameplay.hpp:497-505 */
            uint32_t me = SF_AT(d.h_sel, k.ind) & HS_TEAM;
            bool alive = false;
            for (uint64_t m = e.mh; m; m &= m - 1) {
                uint32_t tm = SF_AT(d.h_sel, sf_ffs64(m)) & HS_TEAM;
                if (tm && tm != me) alive = true;
            }
            if (!alive) e.status = SF_WIN;
        }
        if (e.status == SF_RUNNING && k.max_steps > 0 && (int)e.steps >= k.max_steps) e.status = SF_TRUNCATED;
        e.on = e.status == SF_RUNNING;
    }
    SF_SYNCWARP();
}

/* The loop body of gameplay::play(), gameplay.hpp:1444-1471, then the victory test.  Both
 * half-ticks end with the same three calls (update_tmp, hit_human / hit_zombie, ++frame,
 * update_bull), so they run as two rounds of one loop: round 0 = spawns + zombie_action +
 * portal_damage (:1444-1456), round 1 = human_action (:1464). */
SF_FN void sf_step_halves(const SfDev &d, const SfConst &k, const SfTabs &t, int env, SfEnv &e,
                          const uint8_t *actions, int first, int last)
{
#pragma unroll 1
    for (int ph = first; ph <= last; ++ph) {
        SF_PHASE_SYNC(0);
        if (ph == 0) {
            sf_spawns(d, k, t, env, e);
            SF_PHASE_SYNC(1);
            sf_zombie_action(d, k, t, env, e);
            SF_PHASE_SYNC(2);
            sf_portal_damage(d, k, t, env, e);
        } else {
            sf_human_action(d, k, t, env, e, actions);
        }
        SF_PHASE_SYNC(3);
        sf_resolve_bullets(d, k, t, env, e);
        if (e.on) e.frame += 1;
        SF_PHASE_SYNC(4);
        sf_update_bull(d, t, env, e);
    }
    if (last == 1) {
        if (e.on) e.steps += 1;
        sf_eval_end(d, k, env, e);
    }
}

/* ------------------------------------------------------------------ header load / store */

SF_FN void sf_load_env(const SfDev &d, int env, SfEnv &e)
{
    e.frame = d.frame[env];
    e.kills = d.kills[env], e.tkills = d.tkills[env], e.loot = d.loot[env], e.chest = d.chest[env];
    uint32_t misc = d.misc[env];
    e.level = (int)(misc & 0xFFu), e.status = (int)((misc >> 8) & 0xFFu), e.hw_h = (int)((misc >> 16) & 0xFFu);
    e.steps = d.steps[env], e.episode = d.episode[env], e.ntemp = d.ntemp[env];
    e.mh = d.mh[env];
    e.mz[0] = SF_AT(d.mz, 0), e.mz[1] = SF_AT(d.mz, 1);
    e.mb[0] = SF_AT(d.mb, 0), e.mb[1] = SF_AT(d.mb, 1);
    e.mp[0] = SF_AT(d.mp, 0), e.mp[1] = SF_AT(d.mp, 1);
    e.quit = 0;
    e.env = env;
    e.fast = (misc >> 24) & 1u;
    e.bank = (misc >> 25) & 1u;
    e.watch = (misc >> 26) & 1u;
    SF_UNROLL
    for (int j = 0; j < 9; ++j) e.Lp[j] = SF_AT(d.rng_log, j);
    SF_UNROLL
    for (int i = 0; i < 10; ++i) e.cst[i] = d.rng_cst[sf_cst_index(d, e.bank ? 1 : 0, i, env)];
    e.W = d.rng_w[env];
    e.jomle = d.jomle[env];
    e.on = e.status == SF_RUNNING;
}

SF_FN void sf_store_env(const SfDev &d, int env, const SfEnv &e)
{
    d.frame[env] = e.frame;
    d.kills[env] = e.kills, d.tkills[env] = e.tkills, d.loot[env] = e.loot, d.chest[env] = e.chest;
    d.misc[env] = (uint32_t)e.level | ((uint32_t)e.status << 8) | ((uint32_t)e.hw_h << 16) | (e.fast ? 1u << 24 : 0u) |
                  (e.bank ? 1u << 25 : 0u) | (e.watch ? 1u << 26 : 0u);
    d.steps[env] = e.steps, d.episode[env] = e.episode, d.ntemp[env] = e.ntemp;
    d.mh[env] = e.mh;
    SF_AT(d.mz, 0) = e.mz[0], SF_AT(d.mz, 1) = e.mz[1];
    SF_AT(d.mb, 0) = e.mb[0], SF_AT(d.mb, 1) = e.mb[1];
    SF_AT(d.mp, 0) = e.mp[0], SF_AT(d.mp, 1) = e.mp[1];
    SF_UNROLL
    for (int j = 0; j < 9; ++j) SF_AT(d.rng_log, j) = e.Lp[j];
    d.rng_w[env] = e.W;
    d.jomle[env] = e.jomle;
}

/* algorithmic bytes of one step from the live populations (SURVEY.md 8d, DESIGN.md):
 * 2 * (140 + 64 n_h + 12 n_z + 28 n_b + 4 n_c + 8 n_t + 4 n_p) + A_act + 32 */
SF_FN uint32_t sf_algo_bytes(const SfConst &k, const SfEnv &e)
{
    uint32_t nh = (uint32_t)sf_popc64(e.mh), nz = (uint32_t)m2_count(e.mz), nb = (uint32_t)m2_count(e.mb);
    uint32_t np = (uint32_t)m2_count(e.mp) - (uint32_t)k.n_static_exits;
    return 2u * (140u + 64u * nh + 12u * nz + 28u * nb + 4u * (uint32_t)e.chest + 8u * e.ntemp + 4u * np) +
           (uint32_t)k.n_agents + 32u;
}

/* ------------------------------------------------------------------ kernel bodies */

enum { SF_HALF_BOTH = 0, SF_HALF_A = 1, SF_HALF_B = 2 };

/* per-lane contribution to the handle's running statistics (SF_STAT_*) */
struct SfStatDelta {
    uint32_t steps, episodes, wins, deaths, timeouts, truncated, overflows, ub_guards, draws, algo_bytes;
    int32_t kills, tkills, loot;
};

/* reset one arena for episode `episode` with explicit seeds */
SF_FN void sf_reset_body(const SfDev &d, const SfConst &k, const SfTabs &t, int env, int64_t tb, int64_t serial,
                         uint32_t episode)
{
    SfEnv e;
    e.episode = episode;
    e.env = env;
    e.bank = (d.misc[env] >> 25) & 1u;
    sf_seed_pending(d, t, env, e.bank ? 0 : 1, tb, serial);
    sf_reset_env(d, k, t, env, e);
    sf_store_env(d, env, e);
    sf_step_out o;
    o.status = SF_RUNNING, o.d_kills = o.d_teams_kills = o.d_loot = o.d_hp = o.d_damage = o.d_effect = 0;
    o.episode_steps = 0;
    d.out[env] = o;
}

/* an arena whose episode has ended and that has not been reset since, from its header word */
SF_FN bool sf_misc_finished(uint32_t misc) { return ((misc >> 8) & 0xFFu) != SF_RUNNING; }

/* sf_reset_finished for arena `env`: what auto-reset does at the end of the step in which the episode
 * ended (the tail of sf_step_body), on the state that step stored -- next episode of the arena's own
 * synthetic seed chain, the pending stream installed.  d.out and the statistics are not touched. */
SF_FN void sf_reset_finished_body(const SfDev &d, const SfConst &k, const SfTabs &t, int env)
{
    SfEnv e;
    sf_load_env(d, env, e);
    if (e.status != SF_RUNNING) {
        e.episode += 1;
        sf_reset_env(d, k, t, env, e);
        sf_store_env(d, env, e);
    }
}

/* one env-step (or one half of it) for arena `env`; `actions` is the arena's row of the
 * action buffer (NULL for SF_HALF_A).  `valid` is false for the padding lanes of the last
 * warp: they walk through the same code with nothing to do, so that every lane of a warp
 * reaches every SF_SYNCWARP().
 *
 * Nothing but `e` stays in registers across the tick: the step output starts as "minus the
 * values at entry" in d.out and gets the values at exit added, and the statistics read the
 * entry values back from the header arrays, which are only overwritten by sf_store_env. */
SF_FN void sf_step_body(const SfDev &d, const SfConst &k, const SfTabs &t, int env, bool valid,
                        const uint8_t *actions, int half, SfStatDelta &sd)
{
    if (half != SF_HALF_B) {
        sf_advance_pending(d, t, env, valid, SF_WARM_PER_STEP);
        SF_SYNCWARP();
    }
    SfEnv e;
    sf_load_env(d, env, e);
    if (!valid) e.on = false;
    const bool was_on = e.on;
    if (valid) {
        sf_step_out o;
        if (half == SF_HALF_B) o = d.out[env];
        else o.status = 0, o.d_kills = o.d_teams_kills = o.d_loot = o.d_hp = o.d_damage = o.d_effect = 0, o.episode_steps = 0;
        o.d_kills -= e.kills, o.d_teams_kills -= e.tkills, o.d_loot -= e.loot;
        o.d_hp -= SF_AT(d.h_hp, k.ind), o.d_damage -= SF_AT(d.h_dmg, k.ind), o.d_effect -= SF_AT(d.h_eff, k.ind);
        d.out[env] = o;
    }
    if (half != SF_HALF_B && e.on) sd.algo_bytes += sf_algo_bytes(k, e);
    sf_bt_rebuild(d, t, env, e);
    sf_step_halves(d, k, t, env, e, actions, half == SF_HALF_B ? 1 : 0, half == SF_HALF_A ? 0 : 1);
    if (valid) {
        /* a terminal arena that is not auto-reset waits for sf_reset: report, change nothing */
        sf_step_out o = d.out[env];
        o.d_kills += e.kills, o.d_teams_kills += e.tkills, o.d_loot += e.loot;
        o.d_hp += SF_AT(d.h_hp, k.ind), o.d_damage += SF_AT(d.h_dmg, k.ind), o.d_effect += SF_AT(d.h_eff, k.ind);
        o.status = e.status;
        o.episode_steps = (int32_t)e.steps;
        d.out[env] = o;
        if (d.out_mirror) d.out_mirror[env] = o; /* straight into the caller's host buffer, no copy afterwards */
    }
    /* Auto-reset happens at the end of the whole step: an episode that ends in half A (an overflow or
       guard abort) is stored as it ended, half B runs on it with nothing to do, keeps its terminal status
       in d.out and resets it.  With auto-reset no arena waits for sf_reset, so an arena that is terminal
       when half B starts ended in this step's half A. */
    bool reset = false;
    if (was_on) {
        sd.kills += e.kills - d.kills[env], sd.tkills += e.tkills - d.tkills[env], sd.loot += e.loot - d.loot[env];
        sd.draws += e.jomle - d.jomle[env];
        if (half != SF_HALF_A && (e.status == SF_RUNNING || e.status == SF_WIN || e.status == SF_DEAD ||
                                  e.status == SF_TIMEOUT || e.status == SF_TRUNCATED))
            sd.steps += 1; /* a step that ran to its end (overflow / guard abort it midway) */
        if (e.status != SF_RUNNING) {
            sd.episodes += 1;
            sd.wins += e.status == SF_WIN, sd.deaths += e.status == SF_DEAD, sd.timeouts += e.status == SF_TIMEOUT;
            sd.truncated += e.status == SF_TRUNCATED, sd.overflows += e.status == SF_OVERFLOW;
            sd.ub_guards += e.status == SF_UB_GUARD;
            reset = k.auto_reset != 0 && half != SF_HALF_A;
        }
        if (!reset) sf_store_env(d, env, e);
    } else if (half == SF_HALF_B && valid && k.auto_reset != 0 && e.status != SF_RUNNING) {
        reset = true;
    }
    if (reset) { /* new behaviour (SURVEY 7.4#10): next episode of the synthetic seed chain */
        e.episode += 1;
        sf_reset_env(d, k, t, env, e);
        sf_store_env(d, env, e);
    }
    SF_SYNCWARP();
}

#endif /* SF_CORE_CUH */
