"""GPU tests of sf_action_mask (DESIGN.md section 7f):
- For every GPU configuration at a sub-wave and a multi-pass batch, the CUDA handle and the host-check build run in
  lockstep (same seeds and actions, split step): the state hashes are equal, and the masks of all arenas equal the
  host-check predicate at P1 and P2 every step and the brute force of the definition (hc_action_mask_brute) on
  rotating arenas every few steps.  The multi-pass batch is checked on windows at both ends of the batch.
- The list rules: ids in order, a permutation, duplicates, the ids -1 and n_envs (zero rows), a device count below
  n_max (rows beyond it keep a sentinel), count 0 and count = NULL.
- The call changes nothing: state hashes, sf_step_out, statistics and records are identical, one launch is added.
- observe_list -> action_mask -> step_list -> list_finished -> reset_finished captured in a CUDA graph and replayed
  equals the eager run, masks included.
- action_mask(table=ACTIONS9) equals the bit unpack on the host, and the SF_ERR_ARG cases."""
import ctypes as C

import numpy as np
import pytest

import common
import maskcheck
from strikeforce_b200 import config as sfcfg
from test_gpu_launch_paths import GPU_CONFIGS, _handle, _multi_pass_batch

pytestmark = pytest.mark.gpu

BASE, MAX_STEPS, STEPS = 300, 150, 300
SENTINEL = 0x5A5A5A5A
WINDOW, BRUTE_EVERY, BRUTE_ARENAS = 48, 15, 3


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _kw(name, auto_reset=True):
    return dict(GPU_CONFIGS[name], auto_reset=auto_reset, max_steps=MAX_STEPS, env_id_base=BASE)


def _host(arena_data, name, start, count):
    """a MaskSim that plays arenas start .. start + count - 1 of the device handle (same global ids)"""
    kw = dict(GPU_CONFIGS[name])
    mode = sfcfg.MODES[kw.pop("mode")]
    lvl = kw.pop("level", 1)
    cfg = sfcfg.make_config(arena_data, n_envs=count, mode=mode, level_min=lvl, auto_reset=True, max_steps=MAX_STEPS,
                            env_id_base=BASE + start, **kw)
    return maskcheck.MaskSim(cfg, extra=maskcheck.EXTRA)


@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_mask_equals_host_check(torch_cuda, monkeypatch, arena_data, name, batch):
    torch = torch_cuda
    n, lanes = (200, None) if batch == "sub-wave" else (_multi_pass_batch(torch), 1)
    dev = _handle(monkeypatch, n, lanes, **_kw(name))
    windows = [(0, n)] if batch == "sub-wave" else [(0, WINDOW), (n - WINDOW, WINDOW)]
    hosts = [(s, c, _host(arena_data, name, s, c)) for s, c in windows]
    brute = 0
    try:
        for t in range(STEPS):
            act = dev.synth_actions(t, sfcfg.ACTIONS28)
            for half, point in ((1, "P2"), (2, "P1")):
                if half == 1:
                    dev.step_a()
                else:
                    dev.step_b(act)
                hashes = dev.state_hash().cpu().numpy().astype(np.uint64)
                masks = dev.action_mask().cpu().numpy().view(np.uint32)
                for s, c, hs in hosts:
                    hs.step(None if half == 1 else common.synth_actions(range(BASE + s, BASE + s + c), hs.n_agents, t,
                                                                          sfcfg.ACTIONS28).tobytes(), half=half)
                    for e in range(c):
                        assert np.uint64(hs.state_hash(e)) == hashes[s + e], "state: step %d %s arena %d" % (t, point, s + e)
                    want = hs.masks()
                    bad = np.nonzero((masks[s:s + c] != want).any(1))[0]
                    assert not len(bad), "mask: step %d %s arena %d" % (t, point, s + bad[0])
                    if t % BRUTE_EVERY == 0:
                        for e in ((t // BRUTE_EVERY) * BRUTE_ARENAS + np.arange(BRUTE_ARENAS)) % c:
                            assert (masks[s + e] == hs.action_mask_brute(int(e))).all(), \
                                "mask against the brute force: step %d %s arena %d" % (t, point, s + e)
                            brute += 1
        assert brute >= 2 * len(windows) * BRUTE_ARENAS * (STEPS // BRUTE_EVERY)
    finally:
        dev.close()


def test_list_rules(torch_cuda):
    torch = torch_cuda
    n = 100
    sim = _handle(pytest.MonkeyPatch(), n, None, **_kw("squad-agents"))
    rng = np.random.default_rng(5)
    try:
        for t in range(40):
            sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
        full = sim.action_mask()
        zero = torch.zeros(sim.n_agents, dtype=torch.int32, device=sim.device)
        for ids in (np.arange(n), rng.permutation(n), np.concatenate([rng.integers(0, n, 30), [-1, n, 7, 7, 7]]),
                    np.array([n - 1]), np.array([-1, n, -(1 << 31), 1 << 30])):
            d_ids = torch.as_tensor(ids.astype(np.int32), device=sim.device)
            got = sim.action_mask(env_ids=d_ids)
            for i, e in enumerate(ids):
                want = full[e] if 0 <= e < n else zero
                assert torch.equal(got[i], want), "row %d (id %d)" % (i, e)
            for k in (0, len(ids) // 2, len(ids), len(ids) + 5):
                out = torch.full((len(ids), sim.n_agents), SENTINEL, dtype=torch.int32, device=sim.device)
                cnt = torch.tensor([k], dtype=torch.int32, device=sim.device)
                sim.action_mask(env_ids=d_ids, count=cnt, out=out)
                live = min(k, len(ids))
                assert torch.equal(out[:live], got[:live])
                assert (out[live:] == SENTINEL).all(), "a row beyond the count %d was written" % k
        assert (full[:, 0] & 1).any() and not (full >> sfcfg.N_COMMANDS).any()
    finally:
        sim.close()


def test_the_call_changes_nothing(torch_cuda):
    torch = torch_cuda
    for name in GPU_CONFIGS:
        sim = _handle(pytest.MonkeyPatch(), 300, None, **_kw(name))
        try:
            for t in range(60):
                sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
                if t % 20 == 19:
                    before = (sim.state_hash(), sim.step_out(), sim.stats(), sim.save())
                    launches = sim.launches
                    sim.action_mask()
                    assert sim.launches == launches + 1
                    after = (sim.state_hash(), sim.step_out(), sim.stats(), sim.save())
                    assert torch.equal(before[0], after[0]) and torch.equal(before[1], after[1])
                    assert before[2] == after[2] and torch.equal(before[3], after[3]), name
        finally:
            sim.close()


def test_table_unpack(torch_cuda):
    torch = torch_cuda
    sim = _handle(pytest.MonkeyPatch(), 64, None, **_kw("royale16"))
    try:
        for t in range(30):
            sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
        for table in (sfcfg.ACTIONS9, sfcfg.COMMANDS, b"_3+"):
            words = sim.action_mask().cpu().numpy().view(np.uint32)
            got = sim.action_mask(table=table)
            assert got.dtype == torch.bool and tuple(got.shape) == (64, sim.n_agents, len(table))
            want = np.stack([(words >> sfcfg.COMMANDS.index(c)) & 1 for c in table], -1).astype(bool)
            assert (got.cpu().numpy() == want).all()
    finally:
        sim.close()


def test_cuda_graph_loop_with_masks(torch_cuda):
    """observe_list -> action_mask(env_ids) -> step_list -> list_finished -> reset_finished captured once and
    replayed 150 times equals the same calls run eagerly on a second handle, masks included."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, steps = 300, 150
    kw = _kw("squad-agents", False)
    eager, graphed = BatchedArena(n, **kw), BatchedArena(n, **kw)
    rng = np.random.default_rng(37)
    try:
        def buffers(sim):
            return dict(ids=torch.zeros(n, dtype=torch.int32, device=sim.device),
                        count=torch.zeros(1, dtype=torch.int32, device=sim.device),
                        act=torch.zeros((n, sim.n_agents), dtype=torch.uint8, device=sim.device),
                        obs=torch.zeros((n, 1, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN), device=sim.device),
                        mask=torch.zeros((n, sim.n_agents), dtype=torch.int32, device=sim.device),
                        fin=torch.zeros(n, dtype=torch.int32, device=sim.device),
                        fin_n=torch.zeros(1, dtype=torch.int32, device=sim.device))

        def body(sim, g):
            sim.observe(1, out=g["obs"], env_ids=g["ids"], count=g["count"])
            sim.action_mask(env_ids=g["ids"], count=g["count"], out=g["mask"])
            sim.step_list(g["act"], g["ids"], g["count"])
            sim.list_finished(g["fin"], g["fin_n"])
            sim.reset_finished()

        def inputs(t):
            ids = torch.as_tensor(rng.permutation(n).astype(np.int32), device=eager.device)
            k = torch.tensor([int(rng.integers(0, n + 1))], dtype=torch.int32, device=eager.device)
            return ids, k, eager.synth_actions(t, sfcfg.ACTIONS28)[ids.long()]

        def feed(g, inp):
            g["ids"].copy_(inp[0]), g["count"].copy_(inp[1]), g["act"].copy_(inp[2])

        e_buf, g_buf = buffers(eager), buffers(graphed)
        inp = inputs(0)
        feed(e_buf, inp)
        body(eager, e_buf)
        stream = torch.cuda.Stream(device=graphed.device)
        stream.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            body(graphed, g_buf)
        torch.cuda.current_stream().wait_stream(stream)
        masked = 0
        for t in range(steps):
            if t:
                inp = inputs(t)
            feed(g_buf, inp)
            graph.replay()
            if t:
                feed(e_buf, inp)
                body(eager, e_buf)
            k = int(inp[1])
            assert torch.equal(g_buf["mask"][:k], e_buf["mask"][:k]), "masks: step %d" % t
            assert torch.equal(graphed.state_hash(), eager.state_hash()), "state: step %d" % t
            assert torch.equal(g_buf["fin_n"], e_buf["fin_n"])
            masked += int((g_buf["mask"][:k] != 0).sum())
        assert graphed.stats() == eager.stats()
        assert masked > steps
    finally:
        eager.close(), graphed.close()


def test_errors(torch_cuda):
    from strikeforce_b200.lib import lib
    torch = torch_cuda
    n = 64
    sim = _handle(pytest.MonkeyPatch(), n, None, **_kw("solo"))
    try:
        L, h, s = lib(), sim._h, None
        out = torch.zeros((n + 1, sim.n_agents), dtype=torch.int32, device=sim.device)
        ids = torch.arange(n + 1, dtype=torch.int32, device=sim.device)
        cnt = torch.zeros(2, dtype=torch.int32, device=sim.device)
        p = lambda t, off=0: C.c_void_p(t.data_ptr() + off)  # noqa: E731
        assert L.sf_action_mask(h, None, None, None, n, s) == -1
        assert L.sf_action_mask(h, p(out), None, p(cnt), n, s) == -1      # count without env_ids
        assert L.sf_action_mask(h, p(out), None, None, n - 1, s) == -1    # n_max != n_envs without env_ids
        assert L.sf_action_mask(h, p(out), p(ids), None, 0, s) == -1
        assert L.sf_action_mask(h, p(out), p(ids), None, n + 1, s) == -1
        assert L.sf_action_mask(h, p(out, 2), None, None, n, s) == -1
        assert L.sf_action_mask(h, p(out), p(ids, 2), None, n, s) == -1
        assert L.sf_action_mask(h, p(out), p(ids), p(cnt, 2), n, s) == -1
        assert L.sf_action_mask(h, p(out), None, None, n, s) == 0
        sim.step_a()  # allowed between the halves
        assert L.sf_action_mask(h, p(out), p(ids), p(cnt), n, s) == 0
        sim.step_b(sim.synth_actions(0, sfcfg.ACTIONS28))
        torch.cuda.synchronize()
    finally:
        sim.close()
