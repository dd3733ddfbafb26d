"""GPU tests of the match logs (sf_enable_log / sf_log_list, DESIGN.md section 7h):
- For every GPU configuration at a sub-wave and a multi-pass batch, the CUDA handle (logs and agent outputs on
  together) and the host-check build run in lockstep, the step taken in turn by sf_step, sf_step_a + sf_step_b,
  sf_step_host and sf_step_list, with reset_finished after every step.  Every step the exported rows equal
  hc_log_list, and the agent rows hc_agent_out.  The multi-pass batch is checked on windows at both ends.
- The export: all arenas, and device lists with permutations, duplicates, -1 and n_envs, a count below n_max and
  no count.
- step -> list_finished -> match_logs(count) -> reset_finished captured in a CUDA graph replays to the eager rows.
- The SF_ERR_ARG cases and sf_device_bytes.
- At full size: six arenas of a 131,072-arena squad-agents run, written as files and replayed by the C oracle to
  their recorded hashes."""
import ctypes as C

import numpy as np
import pytest

import common
import logcheck
import sfo
from strikeforce_b200 import config as sfcfg
from strikeforce_b200 import replay
from test_gpu_launch_paths import GPU_CONFIGS, _handle, _multi_pass_batch

pytestmark = pytest.mark.gpu

BASE, MAX_STEPS, STEPS = 300, 60, 240
CAP = 16 * MAX_STEPS
WINDOW = 48
PATHS = ("step", "split", "host", "list")


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _kw(name, auto_reset=False):
    return dict(GPU_CONFIGS[name], auto_reset=auto_reset, max_steps=MAX_STEPS, env_id_base=BASE)


def _host_cfg(arena_data, name, n, base):
    kw = dict(GPU_CONFIGS[name])
    mode = sfcfg.MODES[kw.pop("mode")]
    lvl = kw.pop("level", 1)
    return sfcfg.make_config(arena_data, n_envs=n, mode=mode, level_min=lvl, auto_reset=False, max_steps=MAX_STEPS,
                             env_id_base=base, **kw)


def _actions(rng, n, n_agents):
    return np.frombuffer(sfcfg.COMMANDS, np.uint8)[rng.integers(len(sfcfg.COMMANDS), size=(n, n_agents))]


@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_device_tapes_equal_host_check(torch_cuda, monkeypatch, arena_data, name, batch):
    torch = torch_cuda
    n, lanes = (200, None) if batch == "sub-wave" else (_multi_pass_batch(torch), 1)
    dev = _handle(monkeypatch, n, lanes, agent_out=True, match_log=CAP, **_kw(name))
    windows = [(0, n)] if batch == "sub-wave" else [(0, WINDOW), (n - WINDOW, WINDOW)]
    hosts = [(s, c, logcheck.LogSim(_host_cfg(arena_data, name, c, BASE + s), agent_out=True, match_log=CAP))
             for s, c in windows]
    rng = np.random.default_rng(sum(map(ord, name + batch)))
    out_host = np.zeros(n, dtype=sfcfg.STEP_OUT_DTYPE)
    complete = 0
    try:
        for t in range(STEPS):
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
                rows = np.full((len(ids), dev.n_agents), ord("_"), np.uint8)
                live = (ids >= 0) & (ids < n)
                rows[live] = act[ids[live]]
                dev.step_list(torch.as_tensor(rows, device=dev.device), torch.as_tensor(ids, device=dev.device),
                              torch.tensor([count], dtype=torch.int32, device=dev.device))
            logs = dev.match_logs().cpu().numpy()
            agent = dev.agent_out().cpu().numpy()
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
                want = hs.logs()
                bad = np.nonzero((logs[s:s + c] != want).any(1))[0]
                assert not len(bad), "tape: %s step %d arena %d: %s vs %s" % (
                    path, t, s + bad[0], logcheck.heads(logs[s + bad[0]][None]), logcheck.heads(want[bad[0]][None]))
                assert (agent[s:s + c] == hs.agent_out()).all(), "agent rows: %s step %d" % (path, t)
                hs.reset_finished()
            complete += int((logcheck.heads(logs)["flags"] & sfcfg.LOG_COMPLETE != 0).sum())
            dev.reset_finished()
        assert complete
    finally:
        dev.close()


def test_export_lists(torch_cuda, monkeypatch):
    torch = torch_cuda
    n = 300
    dev = _handle(monkeypatch, n, None, match_log=100, **_kw("royale16"))
    rng = np.random.default_rng(5)
    try:
        for t in range(30):
            dev.step(torch.as_tensor(_actions(rng, n, dev.n_agents), device=dev.device))
        rb = sfcfg.log_row_bytes(100)
        full = dev.match_logs().cpu().numpy()
        assert full.shape == (n, rb) and (logcheck.heads(full)["global_id"] == BASE + np.arange(n)).all()
        ids = np.concatenate([rng.permutation(n)[:50], [7, 7, -1, n, 3]]).astype(np.int32)
        d_ids = torch.as_tensor(ids, device=dev.device)
        for count in (None, len(ids), 20, 0):
            sentinel = torch.full((len(ids), rb), 0xAB, dtype=torch.uint8, device=dev.device)
            cnt = None if count is None else torch.tensor([count], dtype=torch.int32, device=dev.device)
            got = dev.match_logs(d_ids, cnt, out=sentinel).cpu().numpy()
            m = len(ids) if count is None else count
            for i in range(len(ids)):
                if i >= m:
                    assert (got[i] == 0xAB).all(), "row %d beyond the count was written" % i
                elif 0 <= ids[i] < n:
                    assert (got[i] == full[ids[i]]).all()
                else:
                    assert (got[i] == 0).all()
    finally:
        dev.close()


def test_cuda_graph_replays_the_export(torch_cuda):
    """step -> list_finished -> match_logs(count) -> reset_finished captured once and replayed equals the same calls
    run eagerly on a second handle"""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, steps = 300, 120
    kw = _kw("squad-agents")
    eager, graphed = BatchedArena(n, match_log=CAP, **kw), BatchedArena(n, match_log=CAP, **kw)
    rng = np.random.default_rng(41)
    rb = sfcfg.log_row_bytes(CAP)
    try:
        def buffers(sim):
            return dict(act=torch.zeros((n, sim.n_agents), dtype=torch.uint8, device=sim.device),
                        fin=torch.zeros(n, dtype=torch.int32, device=sim.device),
                        fin_n=torch.zeros(1, dtype=torch.int32, device=sim.device),
                        rows=torch.zeros((n, rb), dtype=torch.uint8, device=sim.device))

        def body(sim, g):
            sim.step(g["act"])
            sim.list_finished(g["fin"], g["fin_n"])
            sim.match_logs(g["fin"], g["fin_n"], out=g["rows"])
            sim.reset_finished()

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
        graph.replay()  # the eager handle ran the body twice above
        finished = 0
        for t in range(steps):
            a = torch.as_tensor(_actions(rng, n, eager.n_agents), device=eager.device)
            ge["act"].copy_(a)
            gg["act"].copy_(a)
            body(eager, ge)
            graph.replay()
            k = int(ge["fin_n"].item())
            assert k == int(gg["fin_n"].item())
            assert torch.equal(ge["rows"][:k], gg["rows"][:k]), "step %d" % t
            finished += k
        assert torch.equal(eager.state_hash(), graphed.state_hash())
        assert finished
    finally:
        eager.close(), graphed.close()


def test_errors(torch_cuda):
    from strikeforce_b200.lib import lib
    torch = torch_cuda
    n = 64
    sim = _handle(pytest.MonkeyPatch(), n, None, **_kw("squad-agents"))
    try:
        L, h = lib(), sim._h
        rows = torch.zeros((n, sfcfg.log_row_bytes(64)), dtype=torch.uint8, device=sim.device)
        ptr = C.c_void_p(rows.data_ptr())
        assert L.sf_log_list(h, ptr, None, None, n, None) == -1  # not enabled
        assert L.sf_log_row_bytes(h) == 0
        bytes0 = sim.device_bytes
        assert L.sf_enable_log(h, 0) == -1 and L.sf_enable_log(h, sfcfg.LOG_CAP_MAX + 1) == -1
        sim.step_a()
        assert L.sf_enable_log(h, 64) == -1  # between the halves
        sim.step_b(sim.synth_actions(0))
        assert L.sf_enable_log(h, 64) == 0 and L.sf_enable_log(h, 64) == 0 and L.sf_enable_log(h, 65) == -1
        assert L.sf_log_row_bytes(h) == sfcfg.log_row_bytes(64)
        assert sim.device_bytes == bytes0 + n * sfcfg.log_row_bytes(64)
        assert (sim.match_logs() == 0).all()  # zeroed, no step since
        ids = torch.arange(n, dtype=torch.int32, device=sim.device)
        cnt = torch.ones(1, dtype=torch.int32, device=sim.device)
        assert L.sf_log_list(h, None, None, None, n, None) == -1  # null rows
        assert L.sf_log_list(h, C.c_void_p(rows.data_ptr() + 8), None, None, n, None) == -1  # misaligned rows
        assert L.sf_log_list(h, ptr, None, C.c_void_p(cnt.data_ptr()), n, None) == -1  # count without ids
        assert L.sf_log_list(h, ptr, None, None, n - 1, None) == -1  # all arenas: n_max = n_envs
        assert L.sf_log_list(h, ptr, C.c_void_p(ids.data_ptr()), None, 0, None) == -1
        assert L.sf_log_list(h, ptr, C.c_void_p(ids.data_ptr()), None, n + 1, None) == -1
        assert L.sf_log_list(h, ptr, C.c_void_p(ids.data_ptr() + 2), None, n, None) == -1  # misaligned ids
        sim.step(sim.synth_actions(1))
        sim.step_a()
        mid = sim.match_logs()  # allowed between the halves: the tape as it stands
        assert (logcheck.heads(mid.cpu().numpy())["n_symbols"] > 0).all()
        sim.step_b(sim.synth_actions(2))
    finally:
        sim.close()


def test_full_size_tapes_replay_on_the_oracle(torch_cuda, arena_data, tmp_path):
    """131,072 squad-agents arenas (no auto-reset): six arenas' hashes are recorded every step; each episode of
    theirs that ends is written as a file and replayed by the C oracle to the recorded hashes"""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, watch = 131072, [0, 1, 4095, 65536, 100003, 131071]
    kw = _kw("squad-agents")
    dev = BatchedArena(n, match_log=CAP, **kw)
    rng = np.random.default_rng(9)
    hashes = {e: [] for e in watch}
    replayed = 0
    try:
        for t in range(150):  # reset_finished after every step: every arena runs at the start of every step
            act = _actions(rng, n, dev.n_agents)
            dev.step(torch.as_tensor(act, device=dev.device))
            status = dev.step_out()[:, 0].cpu().numpy()
            h = dev.state_hash().cpu().numpy().astype(np.uint64)
            ended = [e for e in watch if status[e] != sfcfg.RUNNING]
            for e in watch:
                hashes[e].append(int(h[e]))
            if ended:
                rows = dev.match_logs(torch.tensor(ended, dtype=torch.int32, device=dev.device)).cpu().numpy()
                for e, row in zip(ended, rows):
                    head = logcheck.heads(row[None])[0]
                    if head["flags"] & sfcfg.LOG_COMPLETE and not head["flags"] & sfcfg.LOG_UNREPLAYABLE:
                        replayed += _replay(arena_data, row, hashes[e], tmp_path, dev.cfg)
                    hashes[e] = []
            dev.reset_finished()
        assert replayed >= 6
    finally:
        dev.close()


def _replay(arena_data, row, hashes, tmp_path, cfg):
    path = str(tmp_path / "full.sf_sample")
    level = replay.write_device_log(path, row, cfg)
    log = replay.read(path)
    kw = dict(GPU_CONFIGS["squad-agents"])
    o = sfo.Arena(sfcfg.make_config(arena_data, mode=sfcfg.MODE_SQUAD, level_min=level, squad_agents=True,
                                    caps=kw["caps"], max_steps=MAX_STEPS))
    o.reset(level, log.tb, log.serial)
    pos = 0
    for t, want in enumerate(hashes):
        st = o.step_a()
        if st == sfcfg.RUNNING:
            rec = sfo.parse_record(o.dump())
            logged = [0] + [a for a in range(1, 10) if (3, a) in rec and rec[(3, a)][0] and not rec[(3, a)][1]]
            r = bytearray(b"+" * 10)
            for a in logged:
                r[a] = log.commands[pos]
                pos += 1
            st = o.step_b(bytes(r))
        if st not in (sfcfg.OVERFLOW, sfcfg.UB_GUARD):  # the state an abort leaves is undefined
            assert o.state_hash() == want, "step %d" % t
    assert pos == len(log.commands) and o.status() == int(logcheck.heads(row[None])[0]["status"])
    return 1
