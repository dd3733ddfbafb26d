"""GPU tests of sf_save_list / sf_load_list (BatchedArena.save / load / clone with device id lists): the record calls
of a device-side search loop.

- save_list rows equal sf_save rows and the host-check build's hc_save bytes, every GPU_CONFIGS entry at a sub-wave
  and a multi-pass batch: ids in order, a permutation, repeated ids, -1 and n_envs (all-zero rows), a device count
  below n_max (the rows beyond it keep a sentinel), a device count of 0 and count = NULL.
- load_list of a list with repeats, out-of-range ids, clone rows and a count below n_max leaves save() of all
  arenas equal to a twin loaded with the equivalent host list; both then step on with equal hashes and sf_step_out
  every step, across auto-resets.  Also across handles with another env_id_base.
- A refused load_list reports the number of refused owners in its status and changes no arena; neither call
  touches the statistics.
- A search loop (device clone of a root into K slots, observe_list / step_list for several steps, load_list
  restoring the slots) captured once in a CUDA graph and replayed equals the same calls run eagerly.
- The SF_ERR_ARG cases change nothing."""
import ctypes as C

import numpy as np
import pytest

import snapcheck
from strikeforce_b200 import config as sfcfg
from test_gpu_launch_paths import GPU_CONFIGS, _first_diff, _handle, _multi_pass_batch

pytestmark = pytest.mark.gpu

BASE, MAX_STEPS = 300, 150
SENTINEL = 0xA5
SYMBOLS = np.frombuffer(sfcfg.ACTIONS28, dtype=np.uint8)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _kw(name, **extra):
    return dict(dict(GPU_CONFIGS[name], auto_reset=True, max_steps=MAX_STEPS, env_id_base=BASE), **extra)


def _batch(torch, batch):
    return (200, None) if batch == "sub-wave" else (_multi_pass_batch(torch), 1)


def _step(sims, t0, steps):
    for t in range(t0, t0 + steps):
        act = sims[0].synth_actions(t, sfcfg.ACTIONS28)
        for s in sims:
            s.step(act)


def _dev(torch, sim, a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32), device=sim.device)


def _owners(ids, live, n):
    """indices of the live entries that own their id (in range, lowest index)"""
    seen, out = set(), []
    for i, e in enumerate(ids[:live]):
        if 0 <= e < n and int(e) not in seen:
            seen.add(int(e))
            out.append(i)
    return out


@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_save_list_rows(torch_cuda, monkeypatch, name, batch):
    """Rows of save_list equal the rows of sf_save of the same ids and, for a sample, hc_save of the host-check build
    after the same seeds and actions.  Out-of-range ids give all-zero rows; rows at and beyond a device count keep
    the sentinel; a device count of 0 writes nothing."""
    torch = torch_cuda
    n, lanes = _batch(torch, batch)
    kw = _kw(name)
    sim = _handle(monkeypatch, n, lanes, **kw)
    hkw = dict(mode=sfcfg.MODES[kw["mode"]], level_min=kw.get("level", 1), level_max=kw.get("level_max"),
               squad_agents=kw.get("squad_agents", False), caps=kw["caps"], player=kw.get("player", "account1"),
               teams=kw.get("teams"))
    hs = snapcheck.SnapSim(sfcfg.make_config(sim.arena, n_envs=n, auto_reset=True, max_steps=MAX_STEPS, env_id_base=BASE,
                                             **hkw))
    rng = np.random.default_rng(sum(map(ord, name + batch)))
    B = sim.snapshot_bytes
    try:
        for t in range(60):
            act = sim.synth_actions(t, sfcfg.ACTIONS28)
            sim.step(act)
            hs.step(act.cpu().numpy().tobytes())
        full = sim.save()
        perm = rng.permutation(n)
        rep = np.concatenate([rng.integers(0, n, 40), [-1, n, 7, 7, 7, -(1 << 31)]])
        cases = [(np.arange(n), None), (perm, None), (rng.permutation(rep), None), (perm, n // 3), (rep, 0),
                 (np.arange(n), n), (rng.permutation(rep)[:1], None)]
        for ids, count in cases:
            d_ids = _dev(torch, sim, ids)
            out = torch.full((len(ids), B), SENTINEL, dtype=torch.uint8, device=sim.device)
            d_count = None if count is None else _dev(torch, sim, [count])
            assert sim.save(d_ids, out=out, count=d_count) is out
            live = len(ids) if count is None else count
            ok = (ids >= 0) & (ids < n)
            okl = np.nonzero(ok[:live])[0]
            if len(okl):
                want = sim.save(ids[okl])
                got = out[torch.as_tensor(okl, device=sim.device)]
                assert torch.equal(got, want), "rows differ from sf_save: %s" % _first_diff(got, want)
                assert torch.equal(got, full[torch.as_tensor(ids[okl], device=sim.device)])
            bad = np.nonzero(~ok[:live])[0]
            if len(bad):
                assert not bool(out[torch.as_tensor(bad, device=sim.device)].any()), "an out-of-range id wrote a non-zero row"
            if live < len(ids):
                assert bool((out[live:] == SENTINEL).all()), "a row beyond the count was written"
        host = full.cpu().numpy()
        for e in rng.choice(n, min(n, 64), replace=False):
            ref = hs.save(int(e))
            assert (host[e] == ref).all(), "arena %d differs from hc_save at bytes %s" % (e, np.nonzero(host[e] != ref)[0][:16])
    finally:
        sim.close()


def _load_plan(rng, n):
    """ids with repeats and out-of-range ids, rows into n records (other arenas: clones), the live count; entries
    that own nothing name bad rows, which must not be checked"""
    ids = np.concatenate([rng.permutation(n)[:rng.integers(n // 2, n + 1)], rng.integers(0, n, 9), [-1, n, 1 << 30]])
    ids = rng.permutation(ids)
    rows = rng.integers(0, n, len(ids))
    live = len(ids) - int(rng.integers(0, 5))
    owners = _owners(ids, live, n)
    mask = np.ones(len(ids), bool)
    mask[owners] = False
    rows[mask] = rng.choice([-1, n + 3, 1 << 30], int(mask.sum()))
    return ids, rows, live, owners


@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_load_list_equals_host_load(torch_cuda, monkeypatch, name, batch):
    """Two handles on the same seeds and actions.  After T1 steps the records of all arenas are kept and both step on.
    Three times, one loads a device list (see _load_plan) and the other the owning entries with a host id list:
    status 0, save() of all arenas equal, statistics untouched.  Both then step 200 times with equal state hashes
    and sf_step_out every step, across auto-resets, and end with equal records."""
    torch = torch_cuda
    n, lanes = _batch(torch, batch)
    sim = _handle(monkeypatch, n, lanes, **_kw(name))
    twin = _handle(monkeypatch, n, lanes, **_kw(name))
    rng = np.random.default_rng(sum(map(ord, name + batch)) + 1)
    try:
        _step([sim, twin], 0, 40)
        rec = sim.save()
        _step([sim, twin], 40, 30)
        t = 70
        for rep in range(3):
            ids, rows, live, owners = _load_plan(rng, n)
            stats = sim.stats()
            status = sim.load(rec, _dev(torch, sim, ids), rows=_dev(torch, sim, rows), count=_dev(torch, sim, [live]))
            assert int(status) == 0
            assert sim.stats() == stats, "load_list touched the statistics"
            twin.load(rec, ids[owners], rows=rows[owners])
            a, b = sim.save(), twin.save()
            assert torch.equal(a, b), "load %d: records differ at arena %s" % (rep, _first_diff(a, b))
            _step([sim, twin], t, 5)
            t += 5
        ends = 0
        for t in range(t, t + 200):
            _step([sim, twin], t, 1)
            a, b = sim.state_hash(), twin.state_hash()
            assert torch.equal(a, b), "state: step %d arena %s" % (t, _first_diff(a, b))
            a, b = sim.step_out(), twin.step_out()
            assert torch.equal(a, b), "step_out: step %d arena %s" % (t, _first_diff(a, b))
            ends += int((a[:, 0] != sfcfg.RUNNING).sum())
        assert torch.equal(sim.save(), twin.save())
        assert ends >= n, "only %d episodes ended" % ends
    finally:
        sim.close(), twin.close()


def test_load_list_across_handles(torch_cuda):
    """Records of one handle loaded by device list into a handle with another env_id_base (every record a clone
    under another global id there) equal the same records loaded by host list into a twin of that handle, and
    both play on alike across auto-resets."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 200
    src = BatchedArena(n, **_kw("squad-agents"))
    dst = BatchedArena(n, **_kw("squad-agents", env_id_base=BASE + 1000))
    twin = BatchedArena(n, **_kw("squad-agents", env_id_base=BASE + 1000))
    rng = np.random.default_rng(11)
    try:
        _step([src], 0, 50)
        _step([dst, twin], 0, 20)
        rec = src.save()
        ids, rows, live, owners = _load_plan(rng, n)
        status = dst.load(rec, _dev(torch, dst, ids), rows=_dev(torch, dst, rows), count=_dev(torch, dst, [live]))
        twin.load(rec, ids[owners], rows=rows[owners])
        assert int(status) == 0
        assert torch.equal(dst.save(), twin.save())
        for t in range(50, 250):
            _step([dst, twin], t, 1)
            assert torch.equal(dst.state_hash(), twin.state_hash()), "step %d" % t
            assert torch.equal(dst.step_out(), twin.step_out()), "step %d" % t
    finally:
        src.close(), dst.close(), twin.close()


def test_refused_load_list(torch_cuda):
    """Owning entries with a record of another configuration, a broken magic, a zero row or a row out of range:
    status is their number and no arena hash changes.  The same bad rows on ignored repeats or beyond the count do
    not refuse the load.  The statistics are untouched throughout."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 200
    sim = BatchedArena(n, **_kw("squad-agents"))
    other = BatchedArena(n, **_kw("squad-agents", caps=dict(GPU_CONFIGS["squad-agents"]["caps"], cap_chests=77)))
    rng = np.random.default_rng(13)
    try:
        _step([sim], 0, 30)
        good = sim.save()
        _step([sim], 30, 10)
        assert other.snapshot_bytes == sim.snapshot_bytes
        broken = good[5:6].clone()
        broken[0, 0] ^= 1
        recs = torch.cat([good, other.save(torch.tensor([0], dtype=torch.int32, device=sim.device)), broken,
                          torch.zeros_like(good[:1])])
        bad_rows = [n, n + 1, n + 2, len(recs), -1]
        before = sim.state_hash()
        for k in range(1, len(bad_rows) + 1):
            stats = sim.stats()
            ids = rng.permutation(n)[:n - 8]  # room for the repeats below: n_max <= n_envs
            rows = ids.copy()
            where = rng.choice(len(ids), k, replace=False)
            rows[where] = rng.choice(bad_rows, k, replace=False)
            status = sim.load(recs, _dev(torch, sim, ids), rows=_dev(torch, sim, rows))
            assert int(status) == k
            assert torch.equal(sim.state_hash(), before), "a refused load changed an arena"
            status = sim.load(recs, _dev(torch, sim, ids), rows=_dev(torch, sim, rows), count=_dev(torch, sim, [where.max() + 1]))
            assert int(status) == k
            assert torch.equal(sim.state_hash(), before)
            ids2 = np.concatenate([ids, ids[where], ids[:3]])
            rows2 = np.concatenate([ids, rows[where], [n, n + 2, -1]])
            count = len(ids) + k
            assert int(sim.load(recs, _dev(torch, sim, ids2), rows=_dev(torch, sim, rows2), count=_dev(torch, sim, [count]))) == 0
            assert torch.equal(sim.save(ids), good[torch.as_tensor(ids, device=sim.device)]), "the accepted load"
            sim.load(recs[:n], _dev(torch, sim, np.arange(n)))  # the same again, rows = NULL
            assert torch.equal(sim.save(), good)
            assert sim.stats() == stats, "a load touched the statistics"
            _step([sim], 30, 10)
            before = sim.state_hash()
    finally:
        sim.close(), other.close()


def test_cuda_graph_search_loop(torch_cuda):
    """One search expansion per replay: device clone of the root into K slots (save_list + load_list), then S times
    observe_list and step_list of the slots, then load_list restoring every slot from the records of all arenas
    taken before the capture (rows = the slots).  The slots, their count and the actions are written into the
    graph's buffers before each replay; between replays the root moves on by one step_list.  Captured once and
    replayed 200 times, it equals the same calls run eagerly on a twin: statuses, observations, the trajectory
    checksum, the statistics and the records.  The capture enqueues 6 + 4 S + 5 launches and the replays none."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, k, S, reps, root, mask = 256, 64, 4, 200, 3, 0b11
    kw = _kw("squad-agents")
    eager, graphed = BatchedArena(n, **kw), BatchedArena(n, **kw)
    rng = np.random.default_rng(37)
    try:
        _step([eager, graphed], 0, 30)
        na = eager.n_agents

        def buffers(sim):
            z = dict(device=sim.device)
            return dict(src=torch.full((k,), root, dtype=torch.int32, **z), slots=torch.zeros(k, dtype=torch.int32, **z),
                        count=torch.zeros(1, dtype=torch.int32, **z), act=torch.zeros((S, k, na), dtype=torch.uint8, **z),
                        obs=torch.zeros((S, k, 2, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN), **z),
                        scratch=torch.zeros((k, sim.snapshot_bytes), dtype=torch.uint8, **z),
                        backup=sim.save(), st=torch.full((2,), -1, dtype=torch.int32, **z))

        def body(sim, g):
            sim.clone(g["src"], g["slots"], count=g["count"], scratch=g["scratch"], status=g["st"][0:1])
            for s in range(S):
                sim.observe(mask, out=g["obs"][s], env_ids=g["slots"], count=g["count"])
                sim.step_list(g["act"][s], g["slots"], g["count"])
            sim.load(g["backup"], g["slots"], rows=g["slots"], count=g["count"], status=g["st"][1:2])

        def inputs():
            slots = rng.permutation(np.setdiff1d(np.arange(n), [root]))[:k].astype(np.int32)
            return (torch.as_tensor(slots, device=eager.device),
                    torch.tensor([int(rng.integers(k // 2, k + 1))], dtype=torch.int32, device=eager.device),
                    torch.as_tensor(rng.choice(SYMBOLS, (S, k, na)), device=eager.device))

        def feed(g, inp):
            g["slots"].copy_(inp[0]), g["count"].copy_(inp[1]), g["act"].copy_(inp[2])

        def root_step(sim, t):
            row = sim.synth_actions(t, sfcfg.ACTIONS28)[root:root + 1].contiguous()
            sim.step_list(row, torch.tensor([root], dtype=torch.int32, device=sim.device))

        e_buf, g_buf = buffers(eager), buffers(graphed)
        inp = inputs()
        feed(e_buf, inp)
        body(eager, e_buf)  # every kernel is loaded before the capture starts
        stream = torch.cuda.Stream(device=graphed.device)
        stream.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        launches = graphed.launches
        with torch.cuda.graph(graph, stream=stream):
            body(graphed, g_buf)
        captured = graphed.launches - launches
        torch.cuda.current_stream().wait_stream(stream)
        e_check = torch.zeros((), dtype=torch.int64, device=eager.device)
        g_check = torch.zeros((), dtype=torch.int64, device=eager.device)
        for t in range(reps):
            if t:
                inp = inputs()
                feed(e_buf, inp)
                body(eager, e_buf)
            feed(g_buf, inp)
            graph.replay()
            live = int(inp[1])
            e_check = e_check * 1000003 + eager.state_hash().sum()
            g_check = g_check * 1000003 + graphed.state_hash().sum()
            assert g_buf["st"].tolist() == [0, 0] and e_buf["st"].tolist() == [0, 0], "statuses: replay %d" % t
            assert torch.equal(g_buf["obs"][:, :live].view(torch.int32), e_buf["obs"][:, :live].view(torch.int32)), \
                "observations: replay %d" % t
            root_step(eager, 30 + t)
            root_step(graphed, 30 + t)
            if t % 50 == 0:
                assert torch.equal(graphed.save(), eager.save()), "records: replay %d" % t
        assert int(g_check) == int(e_check), "trajectory checksum"
        assert graphed.stats() == eager.stats()
        assert torch.equal(graphed.save(), eager.save())
        assert captured == 6 + 4 * S + 5
        # the twin ran the body eagerly once before the capture and at every replay but the first, and the 30
        # synth_actions launches of the set-up; every other call was made on both
        assert eager.launches - graphed.launches == (reps - 1) * captured + 30
    finally:
        eager.close(), graphed.close()


def test_errors(torch_cuda):
    """sf_save_list and sf_load_list refuse, with SF_ERR_ARG and no change to any hash or record: a call between
    sf_step_a and sf_step_b, NULL records / env_ids / status, a misaligned records, env_ids, count, rows or status,
    n_max of 0 and n_envs + 1, n_records of 0, and rows NULL with fewer records than n_max."""
    from strikeforce_b200.lib import lib
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 64
    sim = BatchedArena(n, **_kw("squad-agents"))
    try:
        _step([sim], 0, 20)
        B = sim.snapshot_bytes
        rec = sim.save()
        raw = torch.zeros(n * B + 16, dtype=torch.uint8, device=sim.device)
        raw[8:8 + n * B].view(n, B).copy_(rec)
        ids = torch.arange(n, dtype=torch.int32, device=sim.device)
        count = torch.tensor([n], dtype=torch.int32, device=sim.device)
        rows = torch.arange(n, dtype=torch.int32, device=sim.device)
        status = torch.full((2,), 7, dtype=torch.int32, device=sim.device)
        h, stream = sim._h, sim._stream()
        p = lambda t, off=0: C.c_void_p(t.data_ptr() + off)  # noqa: E731
        out = torch.full((n, B), SENTINEL, dtype=torch.uint8, device=sim.device)
        raw_out = torch.full((n * B + 16,), SENTINEL, dtype=torch.uint8, device=sim.device)

        def save_list(r=None, i=None, c=None, n_max=n):
            return lib().sf_save_list(h, p(out) if r is None else r, p(ids) if i is None else i,
                                      p(count) if c is None else c, n_max, stream)

        def load_list(r=None, nr=n, rw=None, i=None, c=None, n_max=n, st=None):
            return lib().sf_load_list(h, p(rec) if r is None else r, nr, p(rows) if rw is None else rw,
                                      p(ids) if i is None else i, p(count) if c is None else c, n_max,
                                      p(status) if st is None else st, stream)

        def refused(rc):
            assert rc == -1, "expected SF_ERR_ARG, got %d" % rc
            assert torch.equal(sim.state_hash(), before)
            assert bool((out == SENTINEL).all()) and bool((raw_out == SENTINEL).all()), "a refused save wrote"
            assert status.tolist() == [7, 7], "a refused load wrote its status"

        sim.step_a()
        before = sim.state_hash()
        refused(save_list())
        refused(load_list())
        sim.step_b(sim.synth_actions(20, sfcfg.ACTIONS28))
        before = sim.state_hash()
        null = C.c_void_p(None)
        refused(save_list(r=null))
        refused(save_list(i=null))
        refused(save_list(r=p(raw_out, 8)))
        refused(save_list(i=p(ids, 2)))
        refused(save_list(c=p(count, 1)))
        refused(save_list(n_max=0))
        refused(save_list(n_max=n + 1))
        refused(load_list(r=null))
        refused(load_list(i=null))
        refused(load_list(st=null))
        refused(load_list(r=p(raw, 8)))
        refused(load_list(i=p(ids, 2)))
        refused(load_list(c=p(count, 1)))
        refused(load_list(rw=p(rows, 2)))
        refused(load_list(st=p(status, 2)))
        refused(load_list(n_max=0))
        refused(load_list(n_max=n + 1))
        refused(load_list(nr=0))
        refused(load_list(rw=null, nr=n - 1))
        assert load_list(rw=null, nr=n) == 0 and status.tolist() == [0, 7]
        assert save_list() == 0 and torch.equal(out, rec)
    finally:
        sim.close()
