"""GPU tests of replay (sf_enable_replay / sf_replay_load, DESIGN.md section 7i):
- For every GPU configuration at a sub-wave and a multi-pass batch, the CUDA handle (replay, logs and agent outputs
  on together) and the host-check build run in lockstep, the step taken in turn by sf_step, sf_step_a + sf_step_b,
  sf_step_host and sf_step_list.  Every few steps tapes are loaded into random subsets of arenas through device
  lists with duplicates, -1 and n_envs; the tapes are random symbols over all 30 commands with random lengths and
  heads, so that they end exhausted, with a surplus and in every state between.  Every step the state hashes,
  SF_FIELD_REPLAY and SF_FIELD_REPLAY_DEALT equal the host-check build's.  The multi-pass batch is checked on
  windows at both ends.
- replay_load followed by steps, captured in a CUDA graph, replays to the eager result.
- The SF_ERR_ARG cases and sf_device_bytes.
- At full size: one episode of each of 131,072 squad-agents arenas is recorded with logs on, every tape is loaded
  into a fresh replay handle and played with junk rows: every arena ends with the recorded final hash and status
  and no SURPLUS, and a sample of arenas follows the recorded hashes every step."""
import ctypes as C

import numpy as np
import pytest

import replaycheck
from strikeforce_b200 import config as sfcfg
from test_gpu_launch_paths import GPU_CONFIGS, _handle, _multi_pass_batch
from test_gpu_match_log import _actions, _host_cfg, _kw

pytestmark = pytest.mark.gpu

BASE, MAX_STEPS, STEPS = 300, 60, 160
CAP = 16 * MAX_STEPS
WINDOW = 48
PATHS = ("step", "split", "host", "list")
HEAD = sfcfg.LOG_HEAD.itemsize


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _random_tapes(rng, k, royale):
    rows = np.zeros((k, sfcfg.replay_row_bytes(CAP)), np.uint8)
    for i in range(k):
        head = np.zeros(1, sfcfg.LOG_HEAD)
        n = int(rng.integers(0, CAP + 1))
        head["level"] = 1 if royale else int(rng.integers(1, 11))
        head["episode"], head["n_symbols"] = int(rng.integers(0, 5)), n
        head["tb"], head["serial"] = int(rng.integers(0, 10 ** 12)), int(rng.integers(0, 2 ** 30))
        head["flags"], head["global_id"] = int(rng.integers(0, 16)), int(rng.integers(-5, 5))  # ignored by the load
        rows[i, :HEAD] = head.view(np.uint8)
        rows[i, HEAD:HEAD + n] = np.frombuffer(sfcfg.COMMANDS, np.uint8)[rng.integers(len(sfcfg.COMMANDS), size=n)]
    return rows


def _owners(ids, count, n):
    """entry index owning each id in range (the lowest live one)"""
    own = {}
    for i, e in enumerate(ids[:count]):
        if 0 <= e < n and e not in own:
            own[int(e)] = i
    return own


@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_device_replay_equals_host_check(torch_cuda, monkeypatch, arena_data, name, batch):
    torch = torch_cuda
    n, lanes = (200, None) if batch == "sub-wave" else (_multi_pass_batch(torch), 1)
    dev = _handle(monkeypatch, n, lanes, agent_out=True, match_log=CAP, replay=CAP, **_kw(name))
    windows = [(0, n)] if batch == "sub-wave" else [(0, WINDOW), (n - WINDOW, WINDOW)]
    hosts = [(s, c, replaycheck.ReplaySim(_host_cfg(arena_data, name, c, BASE + s), agent_out=True, match_log=CAP,
                                          replay=CAP)) for s, c in windows]
    royale = GPU_CONFIGS[name]["mode"] == "Royale"
    rng = np.random.default_rng(sum(map(ord, name + batch)) + 7)
    out_host = np.zeros(n, dtype=sfcfg.STEP_OUT_DTYPE)
    dealt_seen = ended = 0
    try:
        for t in range(STEPS):
            if t % 20 == 0:  # tapes into a random subset of arenas, and always into both ends
                k = int(rng.integers(n // 4, n - 9))  # the list, repeats and ids out of range included, fits n_max <= n
                ids = np.concatenate([[0, n - 1], rng.permutation(n)[:k], rng.integers(0, n, 5), [-1, n]]).astype(np.int32)
                count = len(ids) if rng.random() < 0.5 else int(rng.integers(2, len(ids) + 1))
                rows = _random_tapes(rng, len(ids), royale)
                st = dev.replay_load(torch.as_tensor(rows, device=dev.device), torch.as_tensor(ids, device=dev.device),
                                     torch.tensor(count, dtype=torch.int32, device=dev.device))
                assert int(st.item()) == 0
                own = _owners(ids, count, n)
                for s, c, hs in hosts:
                    mine = sorted((i, e - s) for e, i in own.items() if s <= e < s + c)
                    if mine:
                        assert hs.replay_load(rows[[i for i, _ in mine]], [e for _, e in mine]) == 0
            path = PATHS[t % len(PATHS)]
            act = _actions(rng, n, dev.n_agents)
            d_act = torch.as_tensor(act, device=dev.device)
            if path == "step":
                dev.step(d_act)
            elif path == "split":
                dev.step_a()
                dev.step_b(d_act)
            elif path == "host":
                dev.step_host(act, out_host)
            else:
                ids = np.concatenate([rng.permutation(n)[:n - 7], rng.integers(0, n, 5), [-1, n]]).astype(np.int32)
                count = n if rng.random() < 0.5 else int(rng.integers(n // 2, n + 1))
                rows_a = np.full((len(ids), dev.n_agents), ord("_"), np.uint8)
                live = (ids >= 0) & (ids < n)
                rows_a[live] = act[ids[live]]
                dev.step_list(torch.as_tensor(rows_a, device=dev.device), torch.as_tensor(ids, device=dev.device),
                              torch.tensor([count], dtype=torch.int32, device=dev.device))
            state = dev.replay_state().cpu().numpy()
            dealt = dev.replay_dealt().cpu().numpy()
            hashes = dev.state_hash().cpu().numpy().astype(np.uint64)
            for s, c, hs in hosts:
                a_h = act[s:s + c]
                if path in ("step", "host"):
                    hs.step(a_h.tobytes())
                elif path == "split":
                    hs.step(None, half=1)
                    hs.step(a_h.tobytes(), half=2)
                else:
                    own = _owners(ids, count, n)
                    mine = sorted((i, e - s) for e, i in own.items() if s <= e < s + c)
                    hs.step_list(np.array([rows_a[i] for i, _ in mine], np.uint8).reshape(-1, hs.n_agents),
                                 np.array([e for _, e in mine], np.int32))
                for e in range(c):
                    assert int(hashes[s + e]) == hs.state_hash(e), "%s step %d arena %d" % (path, t, s + e)
                    assert tuple(state[s + e]) == hs.replay_state(e), "%s step %d arena %d" % (path, t, s + e)
                    assert (dealt[s + e] == hs.replay_dealt(e)).all(), "%s step %d arena %d" % (path, t, s + e)
                hs.reset_finished()
            dealt_seen += int((dealt != 0).sum())
            ended += int((state[:, 0] & sfcfg.REPLAY_ENDED != 0).sum())
            dev.reset_finished()
        assert dealt_seen and ended
    finally:
        dev.close()


def test_cuda_graph_replays_load_and_steps(torch_cuda):
    """replay_load followed by steps, captured once and replayed, equals the same calls run eagerly"""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 300
    kw = _kw("squad-agents")
    eager, graphed = BatchedArena(n, replay=CAP, **kw), BatchedArena(n, replay=CAP, **kw)
    rng = np.random.default_rng(43)
    try:
        def buffers(sim):
            return dict(rows=torch.zeros((n, sfcfg.replay_row_bytes(CAP)), dtype=torch.uint8, device=sim.device),
                        ids=torch.zeros(n, dtype=torch.int32, device=sim.device),
                        count=torch.zeros((), dtype=torch.int32, device=sim.device),
                        status=torch.zeros((), dtype=torch.int32, device=sim.device),
                        act=torch.zeros((3, n, sim.n_agents), dtype=torch.uint8, device=sim.device))

        def body(sim, g):
            sim.replay_load(g["rows"], g["ids"], g["count"], g["status"])
            for j in range(3):
                sim.step(g["act"][j])

        ge, gg = buffers(eager), buffers(graphed)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            body(graphed, gg)  # warm-up outside the capture
        torch.cuda.current_stream().wait_stream(s)
        body(eager, ge)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            body(graphed, gg)
        body(eager, ge)
        graph.replay()
        for t in range(20):
            rows = torch.as_tensor(_random_tapes(rng, n, False), device=eager.device)
            ids = torch.as_tensor(rng.permutation(n).astype(np.int32), device=eager.device)
            count = torch.tensor(int(rng.integers(0, n + 1)), dtype=torch.int32, device=eager.device)
            act = torch.as_tensor(np.stack([_actions(rng, n, eager.n_agents) for _ in range(3)]), device=eager.device)
            for g in (ge, gg):
                g["rows"].copy_(rows), g["ids"].copy_(ids), g["count"].copy_(count), g["act"].copy_(act)
            body(eager, ge)
            graph.replay()
            assert int(ge["status"].item()) == int(gg["status"].item()) == 0
            assert torch.equal(eager.state_hash(), graphed.state_hash()), "round %d" % t
            assert torch.equal(eager.replay_state(), graphed.replay_state())
            assert torch.equal(eager.replay_dealt(), graphed.replay_dealt())
        assert (eager.replay_dealt() != 0).any()
    finally:
        eager.close(), graphed.close()


def test_errors(torch_cuda):
    from strikeforce_b200.lib import lib
    torch = torch_cuda
    n = 64
    sim = _handle(pytest.MonkeyPatch(), n, None, **_kw("squad-agents"))
    try:
        L, h = lib(), sim._h
        rb = sfcfg.replay_row_bytes(64)
        rows = torch.zeros((n, rb), dtype=torch.uint8, device=sim.device)
        ids = torch.arange(n, dtype=torch.int32, device=sim.device)
        st = torch.zeros(2, dtype=torch.int32, device=sim.device)
        p, pi, ps = C.c_void_p(rows.data_ptr()), C.c_void_p(ids.data_ptr()), C.c_void_p(st.data_ptr())
        out = torch.zeros(n * 64, dtype=torch.int32, device=sim.device)
        assert L.sf_replay_load(h, p, pi, None, n, ps, None) == -1  # not enabled
        assert L.sf_replay_row_bytes(h) == 0
        assert L.sf_get(h, sfcfg.FIELD_REPLAY, C.c_void_p(out.data_ptr()), None) == -1
        assert L.sf_get(h, sfcfg.FIELD_REPLAY_DEALT, C.c_void_p(out.data_ptr()), None) == -1
        bytes0 = sim.device_bytes
        assert L.sf_enable_replay(h, 0) == -1 and L.sf_enable_replay(h, sfcfg.LOG_CAP_MAX + 1) == -1
        sim.step_a()
        assert L.sf_enable_replay(h, 64) == -1  # between the halves
        sim.step_b(sim.synth_actions(0))
        assert L.sf_enable_replay(h, 64) == 0 and L.sf_enable_replay(h, 64) == 0 and L.sf_enable_replay(h, 65) == -1
        assert L.sf_replay_row_bytes(h) == rb
        assert sim.device_bytes == bytes0 + n * rb + (n * 20 + 15) // 16 * 16 + n * sim.n_agents
        assert (sim.replay_state() == 0).all() and (sim.replay_dealt() == 0).all()
        assert L.sf_replay_load(h, None, pi, None, n, ps, None) == -1
        assert L.sf_replay_load(h, p, None, None, n, ps, None) == -1
        assert L.sf_replay_load(h, p, pi, None, n, None, None) == -1
        assert L.sf_replay_load(h, C.c_void_p(rows.data_ptr() + 8), pi, None, n, ps, None) == -1  # misaligned rows
        assert L.sf_replay_load(h, p, C.c_void_p(ids.data_ptr() + 2), None, n, ps, None) == -1
        assert L.sf_replay_load(h, p, pi, None, n, C.c_void_p(st.data_ptr() + 2), None) == -1
        assert L.sf_replay_load(h, p, pi, None, 0, ps, None) == -1
        assert L.sf_replay_load(h, p, pi, None, n + 1, ps, None) == -1
        sim.step_a()
        assert L.sf_replay_load(h, p, pi, None, n, ps, None) == -1  # between the halves
        sim.step_b(sim.synth_actions(1))
        # all-zero heads have level 0: every owning entry is refused and nothing changes
        before = sim.state_hash()
        assert int(sim.replay_load(rows, ids).item()) == n
        assert torch.equal(before, sim.state_hash()) and (sim.replay_state() == 0).all()
    finally:
        sim.close()


def test_full_size_tapes_replay(torch_cuda):
    """one episode of every one of 131,072 squad-agents arenas recorded with logs on, loaded into a fresh replay
    handle and played with junk rows: the final hash and status of every arena, no SURPLUS, and a sample of arenas
    compared every step"""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, watch = 131072, torch.tensor([0, 1, 31, 4095, 65536, 100003, 131071])
    kw = _kw("squad-agents")
    rng = np.random.default_rng(11)
    rec = BatchedArena(n, match_log=CAP, **kw)
    try:
        trail = []
        for t in range(MAX_STEPS + 1):  # max_steps ends every episode; no auto-reset
            rec.step(torch.as_tensor(_actions(rng, n, rec.n_agents), device=rec.device))
            trail.append(rec.state_hash()[watch.to(rec.device)].cpu())
        status = rec.step_out()[:, 0].clone()
        assert (status != sfcfg.RUNNING).all()
        final = rec.state_hash()
        rows = rec.match_logs()
        assert ((rows[:, :4].contiguous().view(torch.int32)[:, 0] & sfcfg.LOG_COMPLETE) != 0).all()
    finally:
        rec.close()
    play = BatchedArena(n, replay=CAP, **kw)
    try:
        st = play.replay_load(rows, torch.arange(n, dtype=torch.int32, device=play.device))
        junk = np.frombuffer(b"_3u", np.uint8)
        for t in range(MAX_STEPS + 1):
            play.step(torch.as_tensor(junk[rng.integers(3, size=(n, play.n_agents))], device=play.device))
            assert torch.equal(play.state_hash()[watch.to(play.device)].cpu(), trail[t]), "step %d" % t
        assert int(st.item()) == 0
        state = play.replay_state()
        assert torch.equal(play.state_hash(), final)
        assert (state[:, 0] == sfcfg.REPLAY_ENDED).all(), "flags %s" % state[:, 0].unique().tolist()
        assert torch.equal(state[:, 4], status) and torch.equal(state[:, 1], state[:, 2])
    finally:
        play.close()
