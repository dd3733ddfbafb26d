// Host build of the bullet-flag table (strikeforce_b200/csrc/sf_core.cuh, sf_bt_*) on top of the host-check build
// with arena records.
//
// TEST INFRASTRUCTURE ONLY, like hostcheck.cpp and snapcheck.cpp, which this file compiles as they are: the entry
// points below call the table functions of the tick directly on the table of the handle (contiguous, bt_stride = 1),
// so the tests can drive inserts, look-ups, wipes and the rebuild from the bullet rows one at a time.
#include "snapcheck.cpp"

extern "C" {

// empty the table and take every spilled flag of arena `env` down, as sf_resolve_bullets does through the bullets
void hc_bt_wipe(HcHandle *h, int env)
{
    const SfDev &d = h->d;
    sf_bt_wipe(h->t);
    for (int c = 0; c < SF_TCELLS; ++c) SF_G(c) = (uint16_t)(SF_G(c) & ~C_S2);
}

// sf_flag_cell: 0, SF_FLAG_NEW and / or BF_SPILL
unsigned hc_bt_flag(HcHandle *h, int env, int cell) { return sf_flag_cell(h->d, h->t, env, cell); }

// sf_flagged
int hc_bt_flagged(HcHandle *h, int env, int cell) { return sf_flagged(h->d, h->t, env, cell); }

// the count word: flags in the table | SF_BT_SPILL
unsigned hc_bt_count(HcHandle *h) { return sf_bt_count(h->t); }

// sf_bt_rebuild of arena `env`, as a kernel does when it picks the arena up
void hc_bt_rebuild(HcHandle *h, int env)
{
    SfEnv e;
    sf_load_env(h->d, env, e);
    sf_bt_rebuild(h->d, h->t, env, e);
}

// the cells of the live bullets of arena `env` that own a flag, and which of those flags are kept in the overlay
// (BF_SPILL); returns their number
int hc_bt_owners(HcHandle *h, int env, int32_t *cells, int32_t *spilled)
{
    const SfDev &d = h->d;
    SfEnv e;
    sf_load_env(d, env, e);
    int n = 0;
    for (int b = 0; b < 128; ++b) {
        if (!m2_test(e.mb, b) || !(SF_AT(d.b_meta, b) & BF_OWNS)) continue;
        cells[n] = (int32_t)(SF_AT(d.b_pw, b) & POS_CELL);
        spilled[n] = (SF_AT(d.b_meta, b) & BF_SPILL) != 0;
        n += 1;
    }
    return n;
}

// the number of buckets; SF_BT_FULL and the number of cell ids into *full and *cells
int hc_bt_geometry(int *full, int *cells)
{
    *full = SF_BT_FULL, *cells = SF_TCELLS;
    return SF_BT_BUCKETS;
}

} // extern "C"
