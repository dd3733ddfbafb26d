// Host build of the arena records (strikeforce_b200/csrc/sf_snapshot.cuh) on top of the host-check build.
//
// TEST INFRASTRUCTURE ONLY, like hostcheck.cpp, which this file compiles as it is: hc_save / hc_load are
// plain per-arena loops over the same layout table and pack / unpack helpers the CUDA kernels follow, so the
// GPU tests can compare device records with these byte for byte.
#include "hostcheck.cpp"
#include "sf_snapshot.cuh"

// the record layout of a handle (cheap enough to build per call: a table of ~45 sections and one hash)
static SfSnapLayout snap_layout(const HcHandle *h)
{
    SfSnapLayout L;
    sf_snap_layout(h->d, h->k, sf_snap_fingerprint(h->k, h->tabs.smap.data(), h->d.cap_t), L);
    return L;
}

extern "C" {

long hc_snapshot_bytes(HcHandle *h) { return (long)snap_layout(h).bytes; }

void hc_save(HcHandle *h, int env, uint8_t *rec) { sf_snap_pack(snap_layout(h), h->k.env_id_base, env, rec); }

// sf_load of one record: -1 (nothing changed) when it is not a record of this configuration
int hc_load(HcHandle *h, int env, const uint8_t *rec)
{
    const SfSnapLayout L = snap_layout(h);
    const uint32_t *w = reinterpret_cast<const uint32_t *>(rec);
    if (!sf_snap_compatible(w, L)) return -1;
    sf_snap_unpack(L, env, rec);
    sf_snap_reseed(h->d, h->k, h->t, env, sf_snap_global_id(w));
    return 0;
}

} // extern "C"
