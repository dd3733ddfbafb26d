// Host build of sf_save_list / sf_load_list on top of the host-check build with arena records, finished-arena calls
// and sf_step_list.
//
// TEST INFRASTRUCTURE ONLY, like hostcheck.cpp, snapcheck.cpp, finishcheck.cpp and listcheck.cpp, which this file
// compiles as they are: hc_save_list and hc_load_list are per-entry loops over the same sf_snap_pack /
// sf_snap_unpack / sf_snap_reseed the CUDA kernels follow, with the list rules of the CUDA path (an out-of-range id
// saves an all-zero row and is skipped by a load, the lowest live index of an id loads it, a load is all or
// nothing), so the tests can compare them with loops of hc_save / hc_load record for record.
#include "listcheck.cpp"

extern "C" {

// sf_save_list: record row i ([n][snapshot_bytes]) of entry i < n is the record of arena ids[i], or all zeros
// when the id is out of range; rows at and beyond n are not written
void hc_save_list(HcHandle *h, const int32_t *ids, int n, uint8_t *records)
{
    const SfSnapLayout L = snap_layout(h);
    for (int i = 0; i < n; ++i) {
        uint8_t *rec = records + (size_t)i * L.bytes;
        if (ids[i] >= 0 && ids[i] < h->d.n_envs) sf_snap_pack(L, h->k.env_id_base, ids[i], rec);
        else memset(rec, 0, L.bytes);
    }
}

// sf_load_list: entry i < n loads record rows[i] (rows NULL: row i) of records[n_records] into arena ids[i] if the
// id is in range and no entry below i lists it.  Returns the number of refused owning entries (a row outside
// [0, n_records) or an incompatible record); nothing changes unless it is 0.
int hc_load_list(HcHandle *h, const uint8_t *records, int n_records, const int32_t *rows, const int32_t *ids, int n)
{
    const SfSnapLayout L = snap_layout(h);
    std::vector<int32_t> claim((size_t)h->d.n_envs, INT32_MAX);
    for (int i = n - 1; i >= 0; --i)
        if (ids[i] >= 0 && ids[i] < h->d.n_envs) claim[ids[i]] = i;
    auto owns = [&](int i) { return ids[i] >= 0 && ids[i] < h->d.n_envs && claim[ids[i]] == i; };
    auto row = [&](int i) { return rows ? rows[i] : i; };
    int refused = 0;
    for (int i = 0; i < n; ++i)
        if (owns(i))
            refused += row(i) < 0 || row(i) >= n_records ||
                       !sf_snap_compatible(reinterpret_cast<const uint32_t *>(records + (size_t)row(i) * L.bytes), L);
    if (refused) return refused;
    for (int i = 0; i < n; ++i)
        if (owns(i)) {
            const uint8_t *rec = records + (size_t)row(i) * L.bytes;
            sf_snap_unpack(L, ids[i], rec);
            sf_snap_reseed(h->d, h->k, h->t, ids[i], sf_snap_global_id(reinterpret_cast<const uint32_t *>(rec)));
        }
    return 0;
}

} // extern "C"
