"""GPU tests of the per-agent step outputs (sf_enable_agent_out, DESIGN.md section 7g):
- For every GPU configuration at a sub-wave and a multi-pass batch, the CUDA handle and the host-check build run in
  lockstep, with the step taken in turn by sf_step, sf_step_a + sf_step_b, sf_step_host and sf_step_list (a
  permutation with repeated ids, -1 and n_envs, and a device count that sometimes leaves arenas out).  Every step
  the state hashes are equal, agent_out() equals hc_agent_out for every arena, and DRIVEN equals
  action_mask() != 0 taken before the step.  The multi-pass batch is checked on windows at both ends.
- Against the C oracle: rows built from the oracle's canonical records (and the device masks, which the lockstep
  test pins) for a few arenas per configuration.
- Agent outputs change nothing else: state hashes, sf_step_out, statistics, records and the launch count per step
  equal those of a twin handle without them; agent_out() adds one launch.
- step_list -> list_finished -> reset_finished -> agent_out() captured in a CUDA graph replays to the eager rows.
- The SF_ERR_ARG cases and sf_device_bytes."""
import ctypes as C

import numpy as np
import pytest

import agentcheck
import common
import sfo
from strikeforce_b200 import config as sfcfg
from test_gpu_launch_paths import GPU_CONFIGS, _handle, _multi_pass_batch

pytestmark = pytest.mark.gpu

BASE, MAX_STEPS, STEPS = 300, 60, 240
WINDOW = 48
TABLE = sfcfg.ACTIONS28 + b"_"
PATHS = ("step", "split", "host", "list")
ABORTS = (sfcfg.OVERFLOW, sfcfg.UB_GUARD)
DRIVEN, DIED = sfcfg.AGENT_DRIVEN, sfcfg.AGENT_DIED


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _kw(name, auto_reset=True):
    return dict(GPU_CONFIGS[name], auto_reset=auto_reset, max_steps=MAX_STEPS, env_id_base=BASE)


def _host_cfg(arena_data, name, n, base):
    """the host-check configuration of n arenas of the device handle from global id base on"""
    kw = dict(GPU_CONFIGS[name])
    mode = sfcfg.MODES[kw.pop("mode")]
    lvl = kw.pop("level", 1)
    return sfcfg.make_config(arena_data, n_envs=n, mode=mode, level_min=lvl, auto_reset=True, max_steps=MAX_STEPS,
                             env_id_base=base, **kw)


def _list(rng, n):
    """n_max = n entries: n - 7 arenas in a random order, 5 repeated ids, -1 and n; the count sometimes leaves the
    tail of the list out"""
    ids = np.concatenate([rng.permutation(n)[:n - 7], rng.integers(0, n, 5), [-1, n]]).astype(np.int32)
    count = n if rng.random() < 0.5 else int(rng.integers(n // 2, n + 1))
    return ids, count


@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_agent_out_equals_host_check(torch_cuda, monkeypatch, arena_data, name, batch):
    torch = torch_cuda
    n, lanes = (200, None) if batch == "sub-wave" else (_multi_pass_batch(torch), 1)
    dev = _handle(monkeypatch, n, lanes, agent_out=True, **_kw(name))
    windows = [(0, n)] if batch == "sub-wave" else [(0, WINDOW), (n - WINDOW, WINDOW)]
    hosts = [(s, c, agentcheck.AgentSim(_host_cfg(arena_data, name, c, BASE + s), agent_out=True)) for s, c in windows]
    rng = np.random.default_rng(sum(map(ord, name + batch)))
    out_host = np.zeros(n, dtype=sfcfg.STEP_OUT_DTYPE)
    seen = dict(driven=0, died=0)
    try:
        for t in range(STEPS):
            path = PATHS[t % len(PATHS)]
            act = common.synth_actions(range(BASE, BASE + n), dev.n_agents, t, TABLE)
            d_act = torch.as_tensor(act, device=dev.device)
            mask = dev.action_mask().cpu().numpy()
            if path == "step":
                dev.step(d_act)
            elif path == "split":
                dev.step_a()
                dev.step_b(d_act)
            elif path == "host":
                dev.step_host(act, out_host)
            else:
                ids, count = _list(rng, n)
                rows = np.full((len(ids), dev.n_agents), ord("_"), np.uint8)
                live = (ids >= 0) & (ids < n)
                rows[live] = act[ids[live]]
                dev.step_list(torch.as_tensor(rows, device=dev.device), torch.as_tensor(ids, device=dev.device),
                              torch.tensor([count], dtype=torch.int32, device=dev.device))
            rows_dev = dev.agent_out().cpu().numpy()
            hashes = dev.state_hash().cpu().numpy().astype(np.uint64)
            for s, c, hs in hosts:
                a_h = act[s:s + c]
                if path in ("step", "host"):
                    hs.step(a_h.tobytes())
                elif path == "split":
                    hs.step(None, half=1)
                    hs.step(a_h.tobytes(), half=2)
                else:
                    mine = [(i, e - s) for i, e in enumerate(ids[:count]) if s <= e < s + c]
                    hs.step_list(np.array([rows[i] for i, _ in mine], np.uint8).reshape(-1, hs.n_agents),
                                 np.array([e for _, e in mine], np.int32))
                for e in range(c):
                    assert np.uint64(hs.state_hash(e)) == hashes[s + e], "state: %s step %d arena %d" % (path, t, s + e)
                want = hs.agent_out()
                bad = np.nonzero((rows_dev[s:s + c] != want).any((1, 2)))[0]
                assert not len(bad), "rows: %s step %d arena %d: %s vs %s" % (
                    path, t, s + bad[0], rows_dev[s + bad[0]].tolist(), want[bad[0]].tolist())
            if path != "list":  # every arena took this step: DRIVEN is the mask before it
                assert ((rows_dev[:, :, 0] & DRIVEN != 0) == (mask != 0)).all(), "DRIVEN vs mask: step %d" % t
            seen["driven"] += int((rows_dev[:, :, 0] & DRIVEN != 0).sum())
            seen["died"] += int((rows_dev[:, :, 0] & DIED != 0).sum())
        assert seen["driven"] and seen["died"], seen
    finally:
        dev.close()


def _humans(rec):
    return {idx: f for (kind, idx), f in sfo.parse_record(rec).items() if kind == 3}


@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_agent_out_against_the_oracle(torch_cuda, arena_data, name):
    """12 arenas per configuration with auto-reset, stepped by sf_step; the C oracle plays the same arenas and is
    reset on the synthetic seed chain.  Rows built from the oracle's records before and after each step (Hp, damage,
    effect, kills, active) and the device mask before it equal agent_out()."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, steps = 12, 200
    kw = _kw(name)
    sim = BatchedArena(n, agent_out=True, **kw)
    lo, hi = kw.get("level", 1), kw.get("level_max", kw.get("level", 1))
    royale = kw["mode"] == "Royale"
    levels = [1 if royale else lo + (BASE + e) % (hi - lo + 1) for e in range(n)]
    okw = {k: v for k, v in GPU_CONFIGS[name].items() if k not in ("mode", "level", "level_max")}
    oracles = []
    for e in range(n):
        o = sfo.Arena(sfcfg.make_config(arena_data, mode=sfcfg.MODES[kw["mode"]], level_min=levels[e],
                                        max_steps=MAX_STEPS, **okw))
        o.reset(levels[e], common.synth_tb(BASE + e), common.synth_serial(BASE + e, 0))
        oracles.append(o)
    episode = [0] * n
    checked = died = 0
    try:
        for t in range(steps):
            act = sim.synth_actions(t, TABLE)
            act_h = act.cpu().numpy()
            mask = sim.action_mask().cpu().numpy()
            before = [_humans(o.dump()) for o in oracles]
            sim.step(act)
            rows = sim.agent_out().cpu().numpy()
            h = sim.state_hash().cpu().numpy().view(np.uint64)
            for e, o in enumerate(oracles):
                st = o.step(bytes(act_h[e]))
                after = _humans(o.dump())
                want = np.zeros((sim.n_agents, 5), np.int32)
                for a in np.nonzero(mask[e])[0]:
                    h0, h1 = before[e][a], after[a]
                    want[a] = (DRIVEN | (0 if h1[0] else DIED), h1[7] - h0[7], h1[11] - h0[11], h1[12] - h0[12],
                               h1[10] - h0[10])
                if st in ABORTS:
                    assert ((rows[e, :, 0] & DRIVEN) == (want[:, 0] & DRIVEN)).all()
                else:
                    assert (rows[e] == want).all(), "arena %d step %d: %s vs %s" % (e, t, rows[e].tolist(), want.tolist())
                    checked += 1
                died += int((want[:, 0] & DIED != 0).sum())
                if st != sfcfg.RUNNING:
                    episode[e] += 1
                    o.reset(levels[e], common.synth_tb(BASE + e), common.synth_serial(BASE + e, episode[e]))
                assert h[e] == np.uint64(o.state_hash()), "state: arena %d step %d" % (e, t)
        assert checked >= n * steps // 2 and died, (checked, died)
    finally:
        sim.close()


def test_agent_out_changes_nothing_else(torch_cuda):
    """twin handles, one with agent outputs: after every step (all four paths) the state hashes, sf_step_out, the
    launch count and the statistics are equal, and at the end the records; agent_out() adds one launch"""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 300
    rng = np.random.default_rng(3)
    for name in GPU_CONFIGS:
        on, off = BatchedArena(n, agent_out=True, **_kw(name)), BatchedArena(n, **_kw(name))
        oh, fh = np.zeros(n, dtype=sfcfg.STEP_OUT_DTYPE), np.zeros(n, dtype=sfcfg.STEP_OUT_DTYPE)
        try:
            assert on.device_bytes == off.device_bytes + n * on.n_agents * 20
            for t in range(80):
                path = PATHS[t % len(PATHS)]
                act = on.synth_actions(t, TABLE).clone()
                ids, count = _list(rng, n)
                d_ids = torch.as_tensor(ids, device=on.device)
                d_cnt = torch.tensor([count], dtype=torch.int32, device=on.device)
                rows = act[d_ids.clamp(0, n - 1).long()].contiguous()
                l0, l1 = on.launches, off.launches
                for sim, out in ((on, oh), (off, fh)):
                    if path == "step":
                        sim.step(act)
                    elif path == "split":
                        sim.step_a()
                        sim.step_b(act)
                    elif path == "host":
                        sim.step_host(act.cpu().numpy(), out)
                    else:
                        sim.step_list(rows, d_ids, d_cnt)
                assert on.launches - l0 == off.launches - l1, "%s %s" % (name, path)
                assert torch.equal(on.state_hash(), off.state_hash()), "%s %s step %d" % (name, path, t)
                assert torch.equal(on.step_out(), off.step_out())
                if path == "host":
                    assert (oh == fh).all()
                l0 = on.launches
                on.agent_out()
                assert on.launches == l0 + 1
            assert on.stats() == off.stats()
            assert torch.equal(on.save(), off.save()), name
        finally:
            on.close(), off.close()


def test_cuda_graph_replays_the_rows(torch_cuda):
    """step_list -> list_finished -> reset_finished -> agent_out() captured once and replayed equals the same calls
    run eagerly on a second handle, rows included"""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, steps = 300, 120
    kw = _kw("squad-agents", False)
    eager, graphed = BatchedArena(n, agent_out=True, **kw), BatchedArena(n, agent_out=True, **kw)
    rng = np.random.default_rng(41)
    try:
        def buffers(sim):
            return dict(ids=torch.zeros(n, dtype=torch.int32, device=sim.device),
                        count=torch.zeros(1, dtype=torch.int32, device=sim.device),
                        act=torch.zeros((n, sim.n_agents), dtype=torch.uint8, device=sim.device),
                        fin=torch.zeros(n, dtype=torch.int32, device=sim.device),
                        fin_n=torch.zeros(1, dtype=torch.int32, device=sim.device))

        def body(sim, g):
            sim.step_list(g["act"], g["ids"], g["count"])
            sim.list_finished(g["fin"], g["fin_n"])
            sim.reset_finished()
            return sim.agent_out()

        def inputs(t):
            ids = torch.as_tensor(rng.permutation(n).astype(np.int32), device=eager.device)
            k = torch.tensor([int(rng.integers(0, n + 1))], dtype=torch.int32, device=eager.device)
            return ids, k, eager.synth_actions(t, TABLE)[ids.long()]

        def feed(g, inp):
            g["ids"].copy_(inp[0]), g["count"].copy_(inp[1]), g["act"].copy_(inp[2])

        e_buf, g_buf = buffers(eager), buffers(graphed)
        inp = inputs(0)
        feed(e_buf, inp)
        e_rows = body(eager, e_buf)
        stream = torch.cuda.Stream(device=graphed.device)
        stream.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            g_rows = body(graphed, g_buf)
        torch.cuda.current_stream().wait_stream(stream)
        driven = 0
        for t in range(steps):
            if t:
                inp = inputs(t)
            feed(g_buf, inp)
            graph.replay()
            if t:
                feed(e_buf, inp)
                e_rows = body(eager, e_buf)
            assert torch.equal(g_rows, e_rows), "rows: step %d" % t
            assert torch.equal(graphed.state_hash(), eager.state_hash()), "state: step %d" % t
            driven += int(((g_rows[:, :, 0] & DRIVEN) != 0).sum())
        assert graphed.stats() == eager.stats()
        assert driven > steps
    finally:
        eager.close(), graphed.close()


def test_errors(torch_cuda):
    from strikeforce_b200.lib import lib
    torch = torch_cuda
    n = 64
    sim = _handle(pytest.MonkeyPatch(), n, None, **_kw("squad-agents"))
    try:
        L, h = lib(), sim._h
        out = torch.zeros((n, sim.n_agents, 5), dtype=torch.int32, device=sim.device)
        assert L.sf_get(h, sfcfg.FIELD_AGENT_OUT, C.c_void_p(out.data_ptr()), None) == -1  # not enabled
        bytes0 = sim.device_bytes
        sim.step_a()
        assert L.sf_enable_agent_out(h) == -1  # between the halves
        sim.step_b(sim.synth_actions(0, TABLE))
        assert L.sf_enable_agent_out(h) == 0
        assert sim.device_bytes == bytes0 + n * sim.n_agents * 20
        assert (sim.agent_out() == 0).all()  # zeroed, no step since
        sim.step(sim.synth_actions(1, TABLE))
        rows = sim.agent_out()
        assert L.sf_enable_agent_out(h) == 0  # a second call does nothing
        assert sim.device_bytes == bytes0 + n * sim.n_agents * 20
        assert torch.equal(sim.agent_out(), rows)
        assert (rows[:, 0, 0] & DRIVEN != 0).all()
        torch.cuda.synchronize()
    finally:
        sim.close()
