"""sf_save_list / sf_load_list on the host-check build of the device code: a saved row must be byte for byte the
hc_save record of its id (all zeros for an out-of-range id), a device-list load must leave every arena as a loop of
hc_load over the owning entries does (the lowest live index of an id), also after 300 further steps with auto-reset
and with records loaded under other global ids (clones), and a load with a refused owning entry must change
nothing and report how many were refused.  The configurations and small capacities are those of
test_split_step.py, so that many episodes end after a load.  The GPU tests (test_gpu_record_list.py) repeat this
through the real kernels."""
import numpy as np
import pytest

import common
import reclistcheck
from strikeforce_b200 import config as sfcfg
from test_split_step import BASE, CONFIGS, MAX_STEPS, N

T1, T2, FOLLOW = 60, 40, 300
SENTINEL = 0xA5


def _sims(arena_data, name, n=2):
    kw, extra = CONFIGS[name]
    cfg = sfcfg.make_config(arena_data, n_envs=N, auto_reset=True, max_steps=MAX_STEPS, env_id_base=BASE, **kw)
    return [reclistcheck.RecListSim(cfg, extra=extra) for _ in range(n)]


def _step(sims, t0, steps):
    for t in range(t0, t0 + steps):
        act = common.synth_actions(range(BASE, BASE + N), sims[0].n_agents, t, sfcfg.ACTIONS28).tobytes()
        for s in sims:
            s.step(act)


def _records(sim):
    return [sim.save(e) for e in range(N)]


def _assert_same_records(a, b, what):
    for e, (x, y) in enumerate(zip(_records(a), _records(b))):
        assert (x == y).all(), "%s: arena %d differs at bytes %s" % (what, e, np.nonzero(x != y)[0][:16])


def _owners(ids, n):
    """the live entries that own their id: in range, lowest index"""
    seen, out = set(), []
    for i, e in enumerate(ids[:n]):
        if 0 <= e < N and e not in seen:
            seen.add(int(e))
            out.append(i)
    return out


@pytest.mark.parametrize("name", list(CONFIGS))
def test_save_list_rows(arena_data, name):
    """Rows of hc_save_list equal hc_save of their id, repeated ids included; an id outside [0, n_envs) gives an
    all-zero row; rows at and beyond the count keep the sentinel the buffer held."""
    (sim,) = _sims(arena_data, name, 1)
    _step([sim], 0, T1)
    rng = np.random.default_rng(sum(map(ord, name)))
    zero = np.zeros(sim.snapshot_bytes, np.uint8)
    for rep in range(4):
        ids = np.concatenate([rng.permutation(N), rng.integers(0, N, 5), [-1, N, 1 << 30, -(1 << 31)]])
        ids = rng.permutation(ids).astype(np.int32)
        count = [None, len(ids) - 7, 0, 1][rep]
        out = np.full((len(ids), sim.snapshot_bytes), SENTINEL, np.uint8)
        sim.save_list(ids, out, count)
        live = len(ids) if count is None else count
        for i, e in enumerate(ids):
            if i >= live:
                assert (out[i] == SENTINEL).all(), "row %d beyond the count %d was written" % (i, live)
            elif 0 <= e < N:
                assert (out[i] == sim.save(e)).all(), "row %d (arena %d) differs from hc_save" % (i, e)
            else:
                assert (out[i] == zero).all(), "row %d (id %d) is not all zeros" % (i, e)
        _step([sim], T1 + rep, 1)


def _load_plan(rng, recs_n):
    """ids with repeats and out-of-range ids, rows into recs_n records (records of other arenas: clones), and a count
    below the list length; returns ids, rows, count"""
    ids = np.concatenate([rng.permutation(N)[:rng.integers(N // 2, N + 1)], rng.integers(0, N, 4), [-1, N, 7 << 20]])
    ids = rng.permutation(ids).astype(np.int32)
    rows = rng.integers(0, recs_n, len(ids)).astype(np.int32)
    return ids, rows, len(ids) - int(rng.integers(0, 4))


@pytest.mark.parametrize("name", list(CONFIGS))
def test_load_list_equals_load_loop(arena_data, name):
    """Two simulators on the same seeds and actions.  After T1 steps the records of all arenas are kept and both step
    on T2.  One loads a device-style list (repeats, out-of-range ids, rows that clone records into other global
    ids, a count below the list length; the repeated entries and the entries beyond the count name bad rows and
    zero records, which must not be checked); the other runs hc_load of each owning entry.  The records of every
    arena are equal after the load, and every step of the next 300, across auto-resets, leaves equal hashes and
    sf_step_out; at the end the records are equal again."""
    a, b = _sims(arena_data, name)
    _step([a, b], 0, T1)
    recs = np.stack(_records(a) + [np.zeros(a.snapshot_bytes, np.uint8)])  # the last row: a zero record
    _step([a, b], T1, T2)
    rng = np.random.default_rng(sum(map(ord, name)) + 1)
    clones = 0
    for rep in range(3):
        ids, rows, count = _load_plan(rng, N)
        owners = _owners(ids, count)
        for i in range(len(ids)):
            if i not in owners:
                rows[i] = [N, len(recs), -5][i % 3]  # the zero record, or rows out of range: not checked
        assert a.load_list(recs, ids, rows, count) == 0
        for i in owners:
            assert b.load(int(ids[i]), recs[rows[i]])
            clones += int(rows[i]) != int(ids[i])
        _assert_same_records(a, b, "after load %d" % rep)
        _step([a, b], T1 + T2 + rep, 1)
    assert clones >= 5
    ends = 0
    for t in range(T1 + T2 + 3, T1 + T2 + 3 + FOLLOW):
        _step([a, b], t, 1)
        for e in range(N):
            assert a.state_hash(e) == b.state_hash(e), "state: step %d arena %d" % (t, e)
            assert a.step_out(e) == b.step_out(e), "step_out: step %d arena %d" % (t, e)
            ends += a.step_out(e)["status"] != sfcfg.RUNNING
    _assert_same_records(a, b, "after %d steps" % FOLLOW)
    assert ends >= N, "only %d episodes ended" % ends


@pytest.mark.parametrize("name", list(CONFIGS))
def test_refused_load_changes_nothing(arena_data, name):
    """A bad owning entry anywhere in the list (a record with a broken magic, of another fingerprint, the zero row,
    a row out of range) refuses the whole load: no arena changes and the count of refused owners is returned.  The
    same list with the bad rows moved to ignored repeats, or beyond the count, loads."""
    a, b = _sims(arena_data, name)
    _step([a, b], 0, T1)
    good = np.stack(_records(a))
    _step([a, b], T1, T2)
    before = _records(a)
    bad_magic = good[3].copy()
    bad_magic[0] ^= 1
    bad_print = good[4].copy()
    bad_print[16] ^= 0x40  # the fingerprint's low word
    recs = np.concatenate([good, [bad_magic, bad_print, np.zeros_like(good[0])]])
    bad_rows = [N, N + 1, N + 2, len(recs), -1]
    rng = np.random.default_rng(sum(map(ord, name)) + 2)
    for k in range(1, len(bad_rows) + 1):
        ids = rng.permutation(N).astype(np.int32)
        rows = ids.copy()
        where = rng.choice(N, k, replace=False)
        rows[where] = rng.choice(bad_rows, k, replace=False)
        assert a.load_list(recs, ids, rows) == k
        assert a.load_list(recs, ids, rows, count=int(where.max()) + 1) == k
        for e, rec in enumerate(_records(a)):
            assert (rec == before[e]).all(), "arena %d changed by a refused load" % e
        # the same bad rows on ignored repeats and beyond the count: not checked
        ids2 = np.concatenate([ids, ids[where], ids[:3]]).astype(np.int32)
        rows2 = np.concatenate([ids, rows[where], [N, N + 2, -1]]).astype(np.int32)
        assert a.load_list(recs, ids2, rows2, count=N + k) == 0
        for e in range(N):
            assert b.load(e, good[e])
        _assert_same_records(a, b, "after the accepted load")
        _step([a, b], T1 + T2 + k, 1)
        before = _records(a)
    assert a.load_list(recs, [-1, N], [N, -1]) == 0
    assert a.load_list(recs, [2, 3], [N, N], count=0) == 0
    _assert_same_records(a, b, "after lists of nothing")
