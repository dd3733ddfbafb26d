"""GPU tests of sf_step_list (BatchedArena.step_list): stepping a device list of arenas and leaving the others
untouched.

- sf_step_list of a subset S and then of its complement equals one sf_step of a twin handle, every GPU_CONFIGS entry,
  at a sub-wave and a multi-pass batch, with auto-reset and with sf_reset_finished after every step: state hashes,
  sf_step_out and statistics every step, sf_save records at the end.  After S, the arenas in S equal the twin's and
  every other arena keeps its hash and sf_step_out row.  The lists rotate through an empty device count, all ids
  in order, a full permutation, repeated ids whose later rows are '_', the ids -1 and n_envs, a device count below
  n_max with in-range entries beyond it, and count = NULL.
- Arenas per warp chosen on the device from the count at a batch that needs more than one per warp.
- The search shape: one root cloned into K slots, the slots stepped with K different rows and observed with
  sf_observe_list; the root and every other arena stay bit-identical and every child equals the same clone stepped
  alone.
- observe_list -> step_list -> list_finished -> reset_finished captured in a CUDA graph and replayed equals the eager
  run.
- The SF_ERR_ARG cases, and a split step after sf_step_list."""
import ctypes as C

import numpy as np
import pytest

from strikeforce_b200 import config as sfcfg
from test_gpu_launch_paths import GPU_CONFIGS, _first_diff, _handle, _multi_pass_batch

pytestmark = pytest.mark.gpu

BASE, MAX_STEPS, STEPS = 300, 150, 200
IDLE = ord("_")
SYMBOLS = np.frombuffer(sfcfg.ACTIONS28, dtype=np.uint8)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _kw(name, auto_reset):
    return dict(GPU_CONFIGS[name], auto_reset=auto_reset, max_steps=MAX_STEPS, env_id_base=BASE)


def _entries(rng, part, act_h, n, room):
    """part in random order, then repeated ids with all-'_' rows and the ids -1 and n, at most `room` entries"""
    ids = rng.permutation(part)
    rows = act_h[ids]
    if len(ids):
        dup = rng.choice(ids, size=3)
        ids = np.concatenate([ids, dup, [-1, n]])
        rows = np.concatenate([rows, np.full((3, act_h.shape[1]), IDLE, np.uint8), rng.choice(SYMBOLS, (2, act_h.shape[1]))])
    return ids[:room], rows[:room]


def _step_list(torch, sim, rng, ids, rows, count=False, pad=0):
    """sf_step_list of (ids, rows); count=True passes a device count of len(ids), followed by `pad` in-range entries
    beyond it that must not be stepped (an empty list goes as a device count of 0: n_max is at least 1)"""
    if len(ids) + pad == 0:
        count, pad = True, 1
    ids = np.concatenate([ids, rng.integers(0, sim.n_envs, pad)]).astype(np.int32)
    rows = np.concatenate([rows.reshape(-1, sim.n_agents), rng.choice(SYMBOLS, (pad, sim.n_agents))]).astype(np.uint8)
    d_ids = torch.as_tensor(ids, device=sim.device)
    d_rows = torch.as_tensor(np.ascontiguousarray(rows), device=sim.device)
    d_count = torch.tensor([len(ids) - pad], dtype=torch.int32, device=sim.device) if count else None
    sim.step_list(d_rows, d_ids, d_count)


def _plan(rng, t, n, act_h):
    """(S, first call, second call) of step t; a call is (ids, rows, count, pad)"""
    every = np.arange(n)
    none = (np.zeros(0, np.int64), np.zeros((0, act_h.shape[1]), np.uint8))
    kind = t % 5
    if kind == 1:
        return every, (every, act_h, True, 0), none + (True, 3)
    if kind == 2:
        perm = rng.permutation(n)
        return every, (perm, act_h[perm], False, 0), none + (True, 1)
    if kind == 4:
        return every[:0], none + (True, 2), (every, act_h, False, 0)
    inside = rng.random(n) < 0.9 * rng.random()
    s, c = every[inside], every[~inside]
    pad = 5 if kind == 3 else 0
    return s, _entries(rng, s, act_h, n, n - pad) + (kind == 3, pad), _entries(rng, c, act_h, n, n) + (False, 0)


@pytest.mark.parametrize("auto_reset", [True, False], ids=["auto-reset", "reset-finished"])
@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_step_list_in_two_parts_equals_step(torch_cuda, monkeypatch, name, batch, auto_reset):
    """A twin takes one sf_step of all arenas per step; the handle under test takes sf_step_list of S and then of the
    complement (see _plan for the lists).  Without auto-reset both reset their finished arenas after every step."""
    torch = torch_cuda
    n, lanes = (200, None) if batch == "sub-wave" else (_multi_pass_batch(torch), 1)
    twin = _handle(monkeypatch, n, lanes, **_kw(name, auto_reset))
    sim = _handle(monkeypatch, n, lanes, **_kw(name, auto_reset))
    rng = np.random.default_rng(sum(map(ord, name + batch)) + auto_reset)
    ends = torch.zeros((), dtype=torch.int64, device=sim.device)
    try:
        for t in range(STEPS):
            act = twin.synth_actions(t, sfcfg.ACTIONS28)
            act_h = act.cpu().numpy()
            twin.step(act)
            s, first, second = _plan(rng, t, n, act_h)
            inside = torch.zeros(n, dtype=torch.bool, device=sim.device)
            inside[torch.as_tensor(s, device=sim.device)] = True
            h0, o0 = sim.state_hash(), sim.step_out()
            _step_list(torch, sim, rng, *first)
            h, o, th, to = sim.state_hash(), sim.step_out(), twin.state_hash(), twin.step_out()
            assert torch.equal(h[inside], th[inside]), "state in S: step %d" % t
            assert torch.equal(o[inside], to[inside]), "step_out in S: step %d" % t
            assert torch.equal(h[~inside], h0[~inside]), "state outside S changed: step %d" % t
            assert torch.equal(o[~inside], o0[~inside]), "step_out outside S changed: step %d" % t
            _step_list(torch, sim, rng, *second)
            a, b = sim.step_out(), twin.step_out()
            assert torch.equal(a, b), "step_out: step %d arena %s" % (t, _first_diff(a, b))
            a, b = sim.state_hash(), twin.state_hash()
            assert torch.equal(a, b), "state: step %d arena %s" % (t, _first_diff(a, b))
            assert sim.stats() == twin.stats(), "statistics: step %d" % t
            ends += (twin.step_out()[:, 0] != sfcfg.RUNNING).sum()
            if not auto_reset:
                twin.reset_finished()
                sim.reset_finished()
        a, b = sim.save(), twin.save()
        assert torch.equal(a, b), "records differ: arena %s" % _first_diff(a, b)
        assert int(ends) >= n, "only %d episodes ended" % int(ends)
    finally:
        twin.close(), sim.close()


def test_lanes_from_the_count(torch_cuda, monkeypatch):
    """At a batch of more arenas than warp slots, sf_step puts several arenas into each warp; sf_step_list picks the
    number on the device from the count: the same for all ids in order with count = n_envs, one for a short list.
    Both equal sf_step."""
    torch = torch_cuda
    n = _multi_pass_batch(torch)
    twin = _handle(monkeypatch, n, None, **_kw("squad-agents", True))
    sim = _handle(monkeypatch, n, None, **_kw("squad-agents", True))
    rng = np.random.default_rng(5)
    every = np.arange(n)
    try:
        for t in range(60):
            act = twin.synth_actions(t, sfcfg.ACTIONS28)
            act_h = act.cpu().numpy()
            twin.step(act)
            if t % 2:
                _step_list(torch, sim, rng, every, act_h, True, 0)
            else:
                short = rng.permutation(n)[:700]
                rest = np.setdiff1d(every, short)
                _step_list(torch, sim, rng, short, act_h[short], True, 0)
                _step_list(torch, sim, rng, rest, act_h[rest])
            a, b = sim.state_hash(), twin.state_hash()
            assert torch.equal(a, b), "state: step %d arena %s" % (t, _first_diff(a, b))
            assert torch.equal(sim.step_out(), twin.step_out()), "step_out: step %d" % t
        assert sim.stats() == twin.stats()
    finally:
        twin.close(), sim.close()


def test_search_expansion(torch_cuda):
    """Squad with agents, 64 arenas.  Three rounds: clone the root into K = 16 slots, step the slots with 16
    different rows in one sf_step_list and observe them with sf_observe_list.  The records of the root and of every
    arena outside the slots are unchanged; every child's state, sf_step_out row and observation equal those of the
    same clone in a second handle stepped alone (one sf_step_list of one entry per child).  Between rounds the root
    moves on by one sf_step_list of itself in both handles."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, k, root = 64, 16, 5
    kw = _kw("squad-agents", True)
    a, b = BatchedArena(n, **kw), BatchedArena(n, **kw)
    rng = np.random.default_rng(23)
    mask = (1 << a.n_agents) - 1
    children = set()
    try:
        for t in range(30):
            act = a.synth_actions(t, sfcfg.ACTIONS28)
            a.step(act)
            b.step(act)
        for r in range(3):
            slots = rng.choice(np.setdiff1d(np.arange(n), [root]), k, replace=False).astype(np.int32)
            others = np.setdiff1d(np.arange(n), slots)
            a.clone([root] * k, slots)
            b.clone([root] * k, slots)
            before = a.save(others)
            ids = torch.as_tensor(slots, device=a.device)
            rows = torch.as_tensor(rng.choice(SYMBOLS, (k, a.n_agents)), device=a.device)
            a.step_list(rows, ids)
            obs = a.observe(mask, env_ids=ids).clone()
            assert torch.equal(a.save(others), before), "round %d: an arena outside the slots changed" % r
            for j in range(k):
                b.step_list(rows[j:j + 1].contiguous(), ids[j:j + 1].contiguous())
            sel = ids.long()
            assert torch.equal(a.state_hash()[sel], b.state_hash()[sel]), "round %d: children differ" % r
            assert torch.equal(a.step_out()[sel], b.step_out()[sel]), "round %d: step_out rows differ" % r
            assert torch.equal(obs.view(torch.int32), b.observe(mask, env_ids=ids).view(torch.int32)), "round %d" % r
            children.update(a.state_hash()[sel].cpu().tolist())
            root_row = torch.as_tensor(rng.choice(SYMBOLS, (1, a.n_agents)), device=a.device)
            root_id = torch.tensor([root], dtype=torch.int32, device=a.device)
            a.step_list(root_row, root_id)
            b.step_list(root_row, root_id)
            assert torch.equal(a.save(), b.save()), "round %d" % r
        assert len(children) > 3, "the children did not take different rows"
    finally:
        a.close(), b.close()


def test_cuda_graph_step_list_loop(torch_cuda):
    """observe_list -> step_list -> list_finished -> reset_finished, with a device list and count written into the
    graph's buffers before every replay, captured once and replayed 200 times equals the same calls run eagerly on a
    second handle: the count, the observations, the finished list, the trajectory checksum (state hashes every
    step), the statistics and the records.  Squad with agents, small capacities, auto_reset = 0.  The capture
    enqueues 1 + 3 + 2 + 3 launches; the replays add none to sf_launch_count."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, steps, mask = 300, 200, 0b11
    kw = _kw("squad-agents", False)
    eager, graphed = BatchedArena(n, **kw), BatchedArena(n, **kw)
    rng = np.random.default_rng(31)
    try:
        def buffers(sim):
            return dict(ids=torch.zeros(n, dtype=torch.int32, device=sim.device),
                        count=torch.zeros(1, dtype=torch.int32, device=sim.device),
                        act=torch.zeros((n, sim.n_agents), dtype=torch.uint8, device=sim.device),
                        obs=torch.zeros((n, 2, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN), device=sim.device),
                        fin=torch.zeros(n, dtype=torch.int32, device=sim.device),
                        fin_n=torch.zeros(1, dtype=torch.int32, device=sim.device))

        def body(sim, g):
            sim.observe(mask, out=g["obs"], env_ids=g["ids"], count=g["count"])
            sim.step_list(g["act"], g["ids"], g["count"])
            sim.list_finished(g["fin"], g["fin_n"])
            sim.reset_finished()

        def inputs(t):
            ids = rng.permutation(n).astype(np.int32)
            k = int(rng.integers(0, n + 1))
            act = eager.synth_actions(t, sfcfg.ACTIONS28)
            ids_d = torch.as_tensor(ids, device=eager.device)
            return ids_d, torch.tensor([k], dtype=torch.int32, device=eager.device), act[ids_d.long()]

        def feed(g, inp):
            g["ids"].copy_(inp[0]), g["count"].copy_(inp[1]), g["act"].copy_(inp[2])

        e_buf, g_buf = buffers(eager), buffers(graphed)
        e_check = torch.zeros((), dtype=torch.int64, device=eager.device)
        g_check = torch.zeros((), dtype=torch.int64, device=eager.device)
        inp = inputs(0)
        feed(e_buf, inp)
        body(eager, e_buf)  # every kernel is loaded before the capture starts
        e_check = e_check * 1000003 + eager.state_hash().sum()
        stream = torch.cuda.Stream(device=graphed.device)
        stream.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        launches = graphed.launches
        with torch.cuda.graph(graph, stream=stream):
            body(graphed, g_buf)
        captured = graphed.launches - launches
        torch.cuda.current_stream().wait_stream(stream)
        ended = 0
        for t in range(steps):
            if t:
                inp = inputs(t)
            feed(g_buf, inp)
            graph.replay()
            g_check = g_check * 1000003 + graphed.state_hash().sum()
            if t:
                feed(e_buf, inp)
                body(eager, e_buf)
                e_check = e_check * 1000003 + eager.state_hash().sum()
            k = int(e_buf["fin_n"])
            assert torch.equal(g_buf["fin_n"], e_buf["fin_n"]), "finished count: step %d" % t
            assert torch.equal(g_buf["fin"][:k], e_buf["fin"][:k]), "finished ids: step %d" % t
            assert torch.equal(g_buf["obs"].view(torch.int32), e_buf["obs"].view(torch.int32)), "observations: step %d" % t
            ended += k
        assert int(g_check) == int(e_check), "trajectory checksum"
        assert graphed.stats() == eager.stats()
        assert torch.equal(graphed.save(), eager.save())
        assert ended >= n // 2, "only %d episodes ended" % ended
        assert captured == 9
        assert graphed.launches - launches == captured + steps + 1  # the hashes and the save, not the replays
    finally:
        eager.close(), graphed.close()


def test_errors(torch_cuda):
    """sf_step_list refuses, with SF_ERR_ARG and no change to any hash, sf_step_out row or statistic: a call between
    sf_step_a and sf_step_b, NULL actions, NULL env_ids, a misaligned env_ids or count, n_max of 0 and of
    n_envs + 1.  It neither opens nor closes a split step: a split step after it equals one of a twin handle."""
    from strikeforce_b200.lib import lib
    torch = torch_cuda
    n = 64
    sim = _handle_plain(n)
    twin = _handle_plain(n)
    try:
        for t in range(30):
            act = sim.synth_actions(t, sfcfg.ACTIONS28)
            sim.step(act)
            twin.step(act)
        ids = torch.arange(n, dtype=torch.int32, device=sim.device)
        count = torch.tensor([n], dtype=torch.int32, device=sim.device)
        act = sim.synth_actions(30, sfcfg.ACTIONS28).clone()
        h, stream = sim._h, sim._stream()

        def sl(a=None, i=None, c=None, n_max=n):
            return lib().sf_step_list(h, C.c_void_p(act.data_ptr()) if a is None else a,
                                      C.c_void_p(ids.data_ptr()) if i is None else i,
                                      C.c_void_p(count.data_ptr()) if c is None else c, n_max, stream)

        def refused(rc):
            assert rc == -1, "expected SF_ERR_ARG, got %d" % rc
            assert torch.equal(sim.state_hash(), before)
            assert torch.equal(sim.step_out(), out)
            assert sim.stats() == stats

        sim.step_a()
        before, out, stats = sim.state_hash(), sim.step_out(), sim.stats()
        refused(sl())
        sim.step_b(act)
        twin.step_a()
        twin.step_b(act)
        before, out, stats = sim.state_hash(), sim.step_out(), sim.stats()
        refused(sl(a=C.c_void_p(None)))
        refused(sl(i=C.c_void_p(None)))
        refused(sl(i=C.c_void_p(ids.data_ptr() + 2)))
        refused(sl(c=C.c_void_p(count.data_ptr() + 1)))
        refused(sl(n_max=0))
        refused(sl(n_max=n + 1))
        act = sim.synth_actions(31, sfcfg.ACTIONS28).clone()
        assert sl() == 0
        twin.step(act)
        act2 = sim.synth_actions(32, sfcfg.ACTIONS28).clone()
        for s in (sim, twin):
            s.step_a()
            s.step_b(act2)
        assert torch.equal(sim.state_hash(), twin.state_hash())
        assert torch.equal(sim.step_out(), twin.step_out())
        assert sim.stats() == twin.stats()
    finally:
        sim.close(), twin.close()


def _handle_plain(n):
    from strikeforce_b200.sim import BatchedArena
    return BatchedArena(n, **_kw("squad-agents", False))
