/*
 * sf_snapshot.cuh -- the arena record of sf_save / sf_load: its layout and the per-arena pack and
 * unpack helpers.  This file is the only place that knows where a field lies in a record; the
 * kernels of sf_lib.cu and the host-check build of tests/ both walk the table it builds.
 *
 * A record is every per-arena word of SfDev (sf_state.h) at the handle's full capacities, dead
 * slots included, so that loading it puts the arena back exactly as it was:
 *
 *   header (64 B)   magic, SF_SNAPSHOT_VERSION, record bytes, configuration fingerprint, global id
 *                   (env_id_base + env) of the arena it was saved from, zeros
 *   SoA sections    one per [rows][E] array of SfDev: the arena's column of that array, rows in
 *                   slot order (header arrays, live masks, rng_log, both banks of rng_cst, pend_log,
 *                   pend_n, rng_w, jomle, the human rows including h_cmd, zombie, bullet and portal rows)
 *   block sections  the per-arena contiguous arrays: the built list t_cell / t_dmg / t_pidx, the whole
 *                   overlay (SF_GRID_STRIDE cells, spill and hint bits included), the arena's sf_step_out
 *
 * Every section starts on a 16-byte boundary; padding bytes are zero.  The record size is a multiple
 * of 128.  Not in a record: the handle's statistics, out_mirror, and the tables shared by all arenas.
 * The bullet-flag table is not state: every kernel rebuilds it from the bullet rows (sf_bt_rebuild).
 */
#ifndef SF_SNAPSHOT_CUH
#define SF_SNAPSHOT_CUH

#include <string.h>

#include "sf_core.cuh"

#define SF_SNAPSHOT_MAGIC 0x4E534653u /* "SFSN" */
#define SF_SNAPSHOT_VERSION 1u
#define SF_SNAP_HEADER 64
#define SF_SNAP_MAX_SEGS 48
#define SF_SNAP_MAX_ITEMS 64
#define SF_SNAP_TILE 32           /* list entries per work item */
#define SF_SNAP_STAGE_RUN 512     /* bytes per arena of one SoA work item (16 KB of shared memory per tile) */
#define SF_SNAP_BLOCK_PIECE 4096  /* bytes per arena of one block work item */

/* one section: a [rows][E] array of `elem`-byte words (rows > 0) or a per-arena block of `elem` bytes
 * (rows == 0) at dev + env * elem */
struct SfSnapSeg {
    uint8_t *dev;
    uint32_t off;  /* byte offset in the record */
    uint32_t rows;
    uint32_t elem;
};

/* a unit of work for one tile of 32 list entries: the SoA sections [first, last), which are contiguous in
 * the record, or the bytes [lo, hi) of block section `first` */
struct SfSnapItem {
    uint16_t first, last;
    uint32_t lo, hi;
};

struct SfSnapLayout {
    uint32_t bytes;          /* record size */
    int32_t n_seg, n_soa, n_item, E;
    uint64_t fingerprint;
    SfSnapSeg seg[SF_SNAP_MAX_SEGS]; /* SoA sections first, then the blocks */
    SfSnapItem item[SF_SNAP_MAX_ITEMS];
};

SF_HDI uint32_t sf_snap_pad16(uint32_t n) { return (n + 15u) & ~15u; }
/* bytes one section occupies in the record */
SF_HDI uint32_t sf_snap_seg_bytes(const SfSnapSeg &s) { return sf_snap_pad16(s.rows ? s.rows * s.elem : s.elem); }

/* where section s ends in the record: the next section's offset, or the record size after the last one (so that
 * a save writes the zero tail of the record too) */
SF_HDI uint32_t sf_snap_end(const SfSnapLayout &L, int s) { return s + 1 < L.n_seg ? L.seg[s + 1].off : L.bytes; }

/* the layout of a handle's records (dev pointers from d) */
static inline void sf_snap_layout(const SfDev &d, const SfConst &k, uint64_t fingerprint, SfSnapLayout &L)
{
    memset(&L, 0, sizeof L);
    L.E = d.E;
    L.fingerprint = fingerprint;
    uint32_t off = SF_SNAP_HEADER;
    auto soa = [&](void *p, uint32_t rows, uint32_t elem) {
        SfSnapSeg &s = L.seg[L.n_seg++];
        s.dev = static_cast<uint8_t *>(p), s.off = off, s.rows = rows, s.elem = elem;
        off += sf_snap_seg_bytes(s);
    };
    const uint32_t H = (uint32_t)k.cap_h, Z = (uint32_t)k.cap_z, B = (uint32_t)k.cap_b, P = (uint32_t)k.cap_p;
    soa(d.frame, 1, 4), soa(d.kills, 1, 4), soa(d.tkills, 1, 4), soa(d.loot, 1, 4), soa(d.chest, 1, 4);
    soa(d.misc, 1, 4), soa(d.steps, 1, 4), soa(d.episode, 1, 4), soa(d.ntemp, 1, 4);
    soa(d.mh, 1, 8), soa(d.mz, 2, 8), soa(d.mb, 2, 8), soa(d.mp, 2, 8);
    soa(d.rng_log, 9, 4), soa(d.rng_cst, 36, 4), soa(d.pend_log, 9, 4), soa(d.pend_n, 1, 4);
    soa(d.rng_w, 1, 4), soa(d.jomle, 1, 4);
    soa(d.h_pw, H, 2), soa(d.h_sel, H, 2), soa(d.h_bp, H, 4), soa(d.h_hp, H, 4), soa(d.h_mind, H, 4);
    soa(d.h_stam, H, 4), soa(d.h_kills, H, 4), soa(d.h_dmg, H, 4), soa(d.h_eff, H, 4), soa(d.h_cons, H, 4);
    soa(d.h_thr, H, 4), soa(d.h_cmd, H, 1);
    soa(d.z_pos, Z, 2), soa(d.z_hp, Z, 4), soa(d.z_mind, Z, 4);
    soa(d.b_pw, B, 2), soa(d.b_meta, B, 4), soa(d.b_dmg, B, 4), soa(d.b_eff, B, 4);
    soa(d.p_cell, P, 2);
    L.n_soa = L.n_seg;
    const uint32_t T = (uint32_t)d.cap_t; /* a multiple of 8: every block is a multiple of 8 bytes */
    soa(d.t_cell, 0, 2 * T), soa(d.t_dmg, 0, 4 * T), soa(d.t_pidx, 0, T);
    soa(d.grid, 0, 2u * SF_GRID_STRIDE), soa(d.out, 0, (uint32_t)sizeof(sf_step_out));
    L.bytes = (off + 127u) & ~127u;
    /* work items: runs of SoA sections up to SF_SNAP_STAGE_RUN bytes per arena, blocks in pieces */
    for (int s = 0; s < L.n_soa;) {
        SfSnapItem &it = L.item[L.n_item++];
        it.first = (uint16_t)s;
        uint32_t run = 0;
        while (s < L.n_soa && (run == 0 || run + sf_snap_seg_bytes(L.seg[s]) <= SF_SNAP_STAGE_RUN))
            run += sf_snap_seg_bytes(L.seg[s++]);
        it.last = (uint16_t)s;
    }
    for (int s = L.n_soa; s < L.n_seg; ++s)
        for (uint32_t lo = 0; lo < L.seg[s].elem; lo += SF_SNAP_BLOCK_PIECE) {
            SfSnapItem &it = L.item[L.n_item++];
            it.first = it.last = (uint16_t)s;
            it.lo = lo;
            it.hi = lo + SF_SNAP_BLOCK_PIECE < L.seg[s].elem ? lo + SF_SNAP_BLOCK_PIECE : L.seg[s].elem;
        }
}

/* 64-bit FNV-1a over the words that give the state words their meaning: geometry, capacities, mode and
 * players, templates, item tables, the static map, and the build options that change what a state
 * word says (the bullet-flag table size decides which flags spill into the overlay).  Built field by
 * field, so struct padding never enters it.  Left out: n_envs, env_id_base, auto_reset, max_steps and
 * the level range, which decide what happens next, not what a record means. */
struct SfFnv {
    uint64_t h = 1469598103934665603ull;
    void add(int64_t v)
    {
        for (int i = 0; i < 8; ++i) h = (h ^ (uint64_t)((v >> (8 * i)) & 0xFF)) * 1099511628211ull;
    }
    void wpn(const SfWpn &w) { add(w.stamina), add(w.damage), add(w.effect), add(w.range); }
    void tmpl(const SfTemplate &t)
    {
        add(t.hp), add(t.mindamage), add(t.stamina), add(t.blocks), add(t.portals), add(t.cons_packed), add(t.thr_packed);
        for (int i = 0; i < 4; ++i) wpn(t.thr[i]);
        for (int i = 0; i < 8; ++i) wpn(t.wpn[i]), add(t.shot_base[i]);
        add(t.w_owned), add(t.mindamage_def);
    }
};

static inline uint64_t sf_snap_fingerprint(const SfConst &k, const uint8_t *smap, int32_t cap_t_rounded)
{
    SfFnv f;
    f.add(SF_SNAPSHOT_VERSION), f.add(SF_ROWS), f.add(SF_COLS), f.add(SF_BT_SLOTS), f.add(SF_BT_FULL);
    f.add(k.cap_h), f.add(k.cap_z), f.add(k.cap_b), f.add(k.cap_chest), f.add(k.cap_t), f.add(cap_t_rounded), f.add(k.cap_p);
    f.add(k.mode), f.add(k.squad_agents), f.add(k.n_agents), f.add(k.n_players), f.add(k.ind);
    for (int i = 0; i < SF_MAX_PLAYERS; ++i) f.add(k.teams[i]);
    for (int i = 0; i < 4; ++i) f.add(k.cons[i].stamina), f.add(k.cons[i].hp), f.add(k.cons[i].effect);
    for (int i = 0; i < SF_MAX_PLAYERS; ++i) f.tmpl(k.players[i]), f.add(k.player_punch_base[i]);
    f.tmpl(k.npc);
    for (int i = 0; i <= SF_MAX_LEVEL; ++i) f.add(k.npc_punch_base[i]), f.add(k.npc_mindamage_def[i]);
    f.add(k.n_static_exits);
    for (int i = 0; i < SF_MAX_STATIC_EXITS; ++i) f.add(k.static_exit_cell[i]);
    for (int i = 0; i < SF_TCELLS; ++i) f.add(smap[i]);
    return f.h;
}

/* ------------------------------------------------------------------ header */

/* word i of the 16 header words: magic, version, bytes, 0, fingerprint (lo, hi), global id (lo, hi), zeros */
SF_HDI uint32_t sf_snap_header_word(const SfSnapLayout &L, int64_t global_id, int i)
{
    switch (i) {
    case 0: return SF_SNAPSHOT_MAGIC;
    case 1: return SF_SNAPSHOT_VERSION;
    case 2: return L.bytes;
    case 4: return (uint32_t)L.fingerprint;
    case 5: return (uint32_t)(L.fingerprint >> 32);
    case 6: return (uint32_t)(uint64_t)global_id;
    case 7: return (uint32_t)((uint64_t)global_id >> 32);
    default: return 0u;
    }
}
/* a record of this layout's handle configuration? */
SF_HDI bool sf_snap_compatible(const uint32_t *w, const SfSnapLayout &L)
{
    return w[0] == SF_SNAPSHOT_MAGIC && w[1] == SF_SNAPSHOT_VERSION && w[2] == L.bytes &&
           w[4] == (uint32_t)L.fingerprint && w[5] == (uint32_t)(L.fingerprint >> 32);
}
SF_HDI int64_t sf_snap_global_id(const uint32_t *w) { return (int64_t)((uint64_t)w[6] | ((uint64_t)w[7] << 32)); }

/* ------------------------------------------------------------------ per-arena helpers */

/* the record of arena env (the host-check build's sf_save; the device kernels produce the same bytes) */
SF_FN void sf_snap_pack(const SfSnapLayout &L, int64_t env_id_base, int env, uint8_t *rec)
{
    for (uint32_t i = 0; i < L.bytes; ++i) rec[i] = 0;
    for (int i = 0; i < 16; ++i) reinterpret_cast<uint32_t *>(rec)[i] = sf_snap_header_word(L, env_id_base + env, i);
    for (int s = 0; s < L.n_seg; ++s) {
        const SfSnapSeg &g = L.seg[s];
        if (g.rows)
            for (uint32_t r = 0; r < g.rows; ++r)
                memcpy(rec + g.off + r * g.elem, g.dev + ((size_t)r * (size_t)L.E + (size_t)env) * g.elem, g.elem);
        else
            memcpy(rec + g.off, g.dev + (size_t)env * g.elem, g.elem);
    }
}

SF_FN void sf_snap_unpack(const SfSnapLayout &L, int env, const uint8_t *rec)
{
    for (int s = 0; s < L.n_seg; ++s) {
        const SfSnapSeg &g = L.seg[s];
        if (g.rows)
            for (uint32_t r = 0; r < g.rows; ++r)
                memcpy(g.dev + ((size_t)r * (size_t)L.E + (size_t)env) * g.elem, rec + g.off + r * g.elem, g.elem);
        else
            memcpy(g.dev + (size_t)env * g.elem, rec + g.off, g.elem);
    }
}

/* After a record saved from global id src_id was loaded into arena env: if env has another global id, the
 * current episode goes on as saved, but the seed chain stays with the slot -- the pending stream (the next
 * episode's) is seeded again as sf_reset_env of this slot would have seeded it, sf_synth(ge, episode + 1),
 * and starts its warm-up from the beginning. */
SF_FN void sf_snap_reseed(const SfDev &d, const SfConst &k, const SfTabs &t, int env, int64_t src_id)
{
    const int64_t ge = k.env_id_base + env;
    if (ge == src_id) return;
    const int bank = (int)((d.misc[env] >> 25) & 1u);
    sf_seed_pending(d, t, env, bank ^ 1, sf_synth_tb(ge), sf_synth_serial(ge, (int64_t)d.episode[env] + 1));
}

#endif /* SF_SNAPSHOT_CUH */
