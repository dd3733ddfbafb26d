"""GPU tests of the final-observation calls (sf_list_finished, sf_reset_finished, sf_observe_list; in Python
BatchedArena.list_finished / reset_finished / observe(env_ids=, count=)).

- auto_reset = 0 with sf_reset_finished after every step equals auto_reset = 1 at a sub-wave and a multi-pass
  batch, with the full and the split step: state hashes, sf_step_out and statistics every step, the sf_save
  records at the end; sf_list_finished equals the non-running arenas of SF_FIELD_COUNTERS every step.
- The terminal observations, taken with sf_observe_list from the listed ids and the device count before the
  reset, equal the rows of a full sf_observe and the C oracle's observations of its terminal states.
- sf_observe_list on its own against sf_observe: ids in order, permutations with duplicates, a device count
  below n_max, count = NULL, out-of-range ids, P1 and P2, both layouts, several agent masks.
- step -> list_finished -> observe_list -> reset_finished captured in a CUDA graph and replayed equals the eager
  run (no host synchronisation inside).  sf_launch_count counts the calls that enqueued work, so a captured call
  counts once, at capture, and not per replay.
- The SF_ERR_ARG cases."""
import numpy as np
import pytest

import common
import sfo
from strikeforce_b200 import config as sfcfg
from test_gpu_launch_paths import GPU_CONFIGS, _first_diff, _handle, _multi_pass_batch

pytestmark = pytest.mark.gpu

ABORTS = (sfcfg.OVERFLOW, sfcfg.UB_GUARD)
ENDS = (sfcfg.WIN, sfcfg.DEAD, sfcfg.TIMEOUT, sfcfg.TRUNCATED)
BASE, MAX_STEPS = 300, 150


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _kw(name, auto_reset, **extra):
    return dict(GPU_CONFIGS[name], auto_reset=auto_reset, max_steps=MAX_STEPS, env_id_base=BASE, **extra)


def _finished_ref(torch, sim):
    """the finished arenas as the state's status (column 6 of SF_FIELD_COUNTERS) shows them"""
    return torch.nonzero(sim.counters()[:, 6] != sfcfg.RUNNING).flatten().to(torch.int32)


def _check_list(torch, sim, what):
    ids, count = sim.list_finished()
    ref = _finished_ref(torch, sim)
    assert int(count) == ref.numel(), "%s: count %d, expected %d" % (what, int(count), ref.numel())
    assert torch.equal(ids[:ref.numel()], ref), "%s: listed ids differ" % what
    return ids, count


@pytest.mark.parametrize("split", [False, True], ids=["full-step", "split-step"])
@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_reset_finished_equals_auto_reset(torch_cuda, monkeypatch, name, batch, split):
    """Two handles on the same seeds and actions, one with auto-reset, one without it and sf_reset_finished after
    every step (after sf_step_b for the split step).  Every step: sf_list_finished before the reset equals the
    non-running arenas of SF_FIELD_COUNTERS and is empty after it (and, for the split step, between the halves);
    state hashes, sf_step_out and statistics are equal.  At the end the sf_save records are equal byte for byte."""
    torch = torch_cuda
    n, lanes = (200, None) if batch == "sub-wave" else (_multi_pass_batch(torch), 1)
    auto = _handle(monkeypatch, n, lanes, **_kw(name, True))
    manual = _handle(monkeypatch, n, lanes, **_kw(name, False))
    aborts = torch.tensor(ABORTS, dtype=torch.int32, device=auto.device)
    ends = torch.zeros((), dtype=torch.int64, device=auto.device)
    aborts_seen = torch.zeros((), dtype=torch.int64, device=auto.device)
    try:
        for t in range(300):
            act = auto.synth_actions(t, sfcfg.ACTIONS28)
            if split:
                auto.step_a()
                auto.step_b(act)
                manual.step_a()
                aborts_seen += torch.isin(manual.step_out()[:, 0], aborts).sum()
                _check_list(torch, manual, "between the halves of step %d" % t)
                manual.step_b(act)
            else:
                auto.step(act)
                manual.step(act)
                aborts_seen += torch.isin(manual.step_out()[:, 0], aborts).sum()
            ids, count = _check_list(torch, manual, "step %d" % t)
            ends += count[0]
            manual.reset_finished()
            assert int(manual.list_finished()[1]) == 0, "step %d: arenas still finished after the reset" % t
            a, b = manual.step_out(), auto.step_out()
            assert torch.equal(a, b), "step_out: step %d arena %s" % (t, _first_diff(a, b))
            a, b = manual.state_hash(), auto.state_hash()
            assert torch.equal(a, b), "state: step %d arena %s" % (t, _first_diff(a, b))
            assert manual.stats() == auto.stats(), "statistics: step %d" % t
        a, b = manual.save(), auto.save()
        assert torch.equal(a, b), "records differ: arena %s" % _first_diff(a, b)
        assert int(ends) >= n, "only %d episodes ended" % int(ends)
        assert int(aborts_seen) >= n // 8, "only %d episodes ended in an abort" % int(aborts_seen)
    finally:
        auto.close(), manual.close()


@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_final_observations(torch_cuda, arena_data, name):
    """auto_reset = 0, default capacities (the episodes end at max_steps rather than in overflows), 160 arenas,
    sf_reset_finished after every step.  Whenever arenas finish, sf_observe_list of the listed ids with the device
    count, in both layouts, equals bit for bit the rows of a full sf_observe taken at the same point; the trailing
    rows keep the sentinel.  Arenas 0..7 are followed by the C oracle across several episodes: their terminal
    observations (the player, and every agent slot for Squad with agents) equal the oracle's terminal state's."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, steps, sample = 160, 460, 8
    kw = {key: v for key, v in _kw(name, False).items() if key != "caps"}
    sim = BatchedArena(n, **kw)
    lo, hi = kw.get("level", 1), kw.get("level_max", kw.get("level", 1))
    level = lambda ge: lo + ge % (hi - lo + 1)  # noqa: E731
    ocfg = dict(mode=sfcfg.MODES[kw["mode"]], squad_agents=kw.get("squad_agents", False), max_steps=MAX_STEPS,
                player=kw.get("player", "account1"), teams=kw.get("teams"))
    oracles = []
    for e in range(sample):
        o = sfo.Arena(sfcfg.make_config(arena_data, level_min=level(BASE + e), **ocfg))
        o.reset(level(BASE + e), common.synth_tb(BASE + e), common.synth_serial(BASE + e, 0))
        oracles.append(o)
    mask = (1 << sim.n_agents) - 1 if kw.get("squad_agents") else 1
    slots = [s for s in range(32) if (mask >> s) & 1]
    episode = [0] * sample
    rounds = compared = 0
    try:
        for t in range(steps):
            act = sim.synth_actions(t, sfcfg.ACTIONS28)
            act_h = act[:sample].cpu().numpy()
            sim.step(act)
            sts = [o.step(bytes(act_h[e])) for e, o in enumerate(oracles)]
            ids, count = sim.list_finished()
            k = int(count)
            if k:
                rounds += 1
                full = sim.observe(mask).clone()
                full_cl = torch.empty((n, len(slots), 31, 31, 32), device=sim.device)  # channel-innermost memory
                sim.observe(mask, out=full_cl, channels_last=True)
                out = torch.full((n, len(slots)) + tuple(full.shape[2:]), -7.0, device=sim.device)
                got = sim.observe(mask, out=out, env_ids=ids, count=count)
                sel = ids[:k].long()
                assert torch.equal(got[:k].view(torch.int32), full[sel].view(torch.int32)), "step %d" % t
                assert bool((got[k:] == -7.0).all()), "step %d: rows beyond count were written" % t
                out_cl = torch.full((n, len(slots), 31, 31, 32), -7.0, device=sim.device)
                got_cl = sim.observe(mask, out=out_cl, channels_last=True, env_ids=ids, count=count)
                assert torch.equal(out_cl[:k].view(torch.int32), full_cl[sel].view(torch.int32)), "step %d NHWC" % t
                assert torch.equal(got_cl[:k], got[:k])
                assert bool((out_cl[k:] == -7.0).all())
                listed = ids[:k].cpu().tolist()
                rows = got[:k].cpu().numpy().reshape(k, len(slots), -1)
                for e, o in enumerate(oracles):
                    if sts[e] not in ENDS:
                        continue
                    for j, slot in enumerate(slots):
                        try:
                            ref = o.observe(slot)
                        except RuntimeError:
                            continue
                        assert (rows[listed.index(e), j].view(np.uint32) == ref.view(np.uint32)).all(), \
                            "terminal observation: arena %d slot %d step %d" % (e, slot, t)
                        compared += 1
            out = sim.step_out()[:sample, 0].cpu().numpy()
            for e, o in enumerate(oracles):
                assert out[e] == sts[e], "status: arena %d step %d" % (e, t)
            sim.reset_finished()
            h = sim.state_hash()[:sample].cpu().numpy().view(np.uint64)
            for e, o in enumerate(oracles):
                if sts[e] != sfcfg.RUNNING:
                    episode[e] += 1
                    o.reset(level(BASE + e), common.synth_tb(BASE + e), common.synth_serial(BASE + e, episode[e]))
                assert h[e] == np.uint64(o.state_hash()), "state after the reset: arena %d step %d" % (e, t)
        assert min(episode) >= 3, "episodes per sampled arena: %s" % episode
        assert rounds >= 3 and compared >= 2 * sample
    finally:
        sim.close()


def test_observe_list_against_observe(torch_cuda):
    """sf_observe_list alone, Squad with agents, 200 arenas stepped with the split step: at P1 and at P2 (between
    the halves), in both layouts, for several agent masks: all ids in order equals sf_observe byte for byte; a
    random permutation with duplicates gives the rows of sf_observe at those ids; a device count below n_max leaves
    the trailing rows of a sentinel-filled buffer untouched; count = NULL writes all n_max rows; out-of-range ids
    (negative, n_envs, large) give zero rows."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 200
    sim = BatchedArena(n, **_kw("squad-agents", True))
    rng = np.random.default_rng(17)
    dev = sim.device
    try:
        for t in range(40):
            sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
        checked = 0
        for phase in (sfcfg.OBS_P1, sfcfg.OBS_P2):
            if phase == sfcfg.OBS_P2:
                sim.step_a()
            for mask in (1, 0b1000000110, (1 << sim.n_agents) - 1):
                for cl in (False, True):
                    def obs(**kw):
                        r = sim.observe(mask, phase, channels_last=cl, **kw)
                        return r.contiguous() if cl else r
                    full = obs().clone()
                    every = torch.arange(n, dtype=torch.int32, device=dev)
                    assert torch.equal(obs(env_ids=every).view(torch.int32), full.view(torch.int32))
                    perm = rng.permutation(n).astype(np.int32)
                    perm[5] = perm[6] = perm[100]  # with duplicates
                    perm = torch.as_tensor(perm, device=dev)
                    assert torch.equal(obs(env_ids=perm).view(torch.int32), full[perm.long()].view(torch.int32))
                    ids = torch.as_tensor(rng.integers(0, n, 90).astype(np.int32), device=dev)
                    count = torch.tensor([33], dtype=torch.int32, device=dev)
                    buf = torch.full((90,) + tuple(full.shape[1:]) if not cl else (90, full.shape[1], 31, 31, 32), 3.5,
                                     device=dev)
                    got = sim.observe(mask, phase, out=buf, channels_last=cl, env_ids=ids, count=count)
                    got = got.contiguous() if cl else got
                    assert torch.equal(got[:33].view(torch.int32), full[ids[:33].long()].view(torch.int32))
                    assert bool((buf[33:] == 3.5).all()), "rows beyond the device count were written"
                    count.fill_(1000)  # above n_max: n_max rows
                    got = sim.observe(mask, phase, out=buf, channels_last=cl, env_ids=ids, count=count)
                    got = got.contiguous() if cl else got
                    assert torch.equal(got.view(torch.int32), full[ids.long()].view(torch.int32))
                    bad = torch.tensor([-1, 3, n, 1 << 30, 7, -(1 << 31)], dtype=torch.int32, device=dev)
                    got = obs(env_ids=bad)
                    zero = torch.zeros_like(got[0])
                    for i, e in enumerate(bad.tolist()):
                        if 0 <= e < n:
                            assert torch.equal(got[i].view(torch.int32), full[e].view(torch.int32))
                        else:
                            assert torch.equal(got[i].view(torch.int32), zero.view(torch.int32)), "id %d" % e
                    checked += 1
            if phase == sfcfg.OBS_P2:
                sim.step_b(sim.synth_actions(40, sfcfg.ACTIONS28))
        assert checked == 12
    finally:
        sim.close()


def test_cuda_graph_final_observation_loop(torch_cuda):
    """step -> list_finished -> observe_list -> reset_finished captured once in a torch.cuda.CUDAGraph and replayed
    300 times (the actions copied into the graph's buffer outside the graph) equals the same calls run eagerly on a
    second handle: the trajectory checksum (state hashes every step), the observation buffer every step and the
    statistics at the end.  Squad with agents, small capacities, auto_reset = 0."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, steps = 300, 300
    kw = _kw("squad-agents", False)
    eager, graphed = BatchedArena(n, **kw), BatchedArena(n, **kw)
    mask = 0b11
    try:
        def buffers(sim):
            ids = torch.empty(n, dtype=torch.int32, device=sim.device)
            count = torch.empty(1, dtype=torch.int32, device=sim.device)
            obs = torch.zeros((n, 2, sfcfg.OBS_CH, sfcfg.OBS_WIN, sfcfg.OBS_WIN), device=sim.device)
            act = torch.empty((n, sim.n_agents), dtype=torch.uint8, device=sim.device)
            return ids, count, obs, act

        def body(sim, ids, count, obs, act):
            sim.step(act)
            sim.list_finished(ids, count)
            sim.observe(mask, out=obs, env_ids=ids, count=count)
            sim.reset_finished()

        e_buf, g_buf = buffers(eager), buffers(graphed)
        e_check = torch.zeros((), dtype=torch.int64, device=eager.device)
        g_check = torch.zeros((), dtype=torch.int64, device=eager.device)
        # the eager handle runs first: every kernel is loaded before the capture starts
        e_buf[3].copy_(eager.synth_actions(0, sfcfg.ACTIONS28))
        body(eager, *e_buf)
        e_check = e_check * 1000003 + eager.state_hash().sum()
        stream = torch.cuda.Stream(device=graphed.device)
        stream.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        launches = graphed.launches
        with torch.cuda.graph(graph, stream=stream):
            body(graphed, *g_buf)
        captured = graphed.launches - launches
        torch.cuda.current_stream().wait_stream(stream)
        ended = 0
        for t in range(steps):
            g_buf[3].copy_(graphed.synth_actions(t, sfcfg.ACTIONS28))
            graph.replay()
            g_check = g_check * 1000003 + graphed.state_hash().sum()
            if t:
                e_buf[3].copy_(eager.synth_actions(t, sfcfg.ACTIONS28))
                body(eager, *e_buf)
                e_check = e_check * 1000003 + eager.state_hash().sum()
            assert torch.equal(g_buf[1], e_buf[1]), "count: step %d" % t
            assert torch.equal(g_buf[2].view(torch.int32), e_buf[2].view(torch.int32)), "observations: step %d" % t
            ended += int(e_buf[1])
        assert int(g_check) == int(e_check), "trajectory checksum"
        assert graphed.stats() == eager.stats()
        assert torch.equal(graphed.save(), eager.save())
        assert ended >= n, "only %d episodes ended" % ended
        # the capture enqueued step, list (2), observe and reset (list + reset: 3) once; outside the graph each step
        # adds sf_synth_actions and the state hash, and the save one more: the replays add nothing
        assert captured == 7
        assert graphed.launches - launches == captured + 2 * steps + 1
    finally:
        eager.close(), graphed.close()


def test_errors(torch_cuda):
    """sf_reset_finished between the halves of a split step is SF_ERR_ARG and changes no hash and no statistic;
    sf_observe_list refuses a null or misaligned buffer, n_max out of range, misaligned ids and the wrong phase;
    sf_list_finished refuses a null or misaligned buffer."""
    import ctypes as C
    from strikeforce_b200.lib import SfError, lib
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 64
    sim = BatchedArena(n, **_kw("squad-agents", False))
    try:
        for t in range(30):
            sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
        ids = torch.arange(n, dtype=torch.int32, device=sim.device)
        count = torch.tensor([n], dtype=torch.int32, device=sim.device)
        raw = torch.zeros(n * sfcfg.OBS_LEN + 8, device=sim.device)
        obs = raw[:n * sfcfg.OBS_LEN]
        stream = sim._stream()
        h = sim._h

        def refused(rc):
            assert rc == -1, "expected SF_ERR_ARG, got %d" % rc
            assert torch.equal(sim.state_hash(), before)
            assert sim.stats() == stats

        def ol(buf, phase=sfcfg.OBS_P1, id_ptr=None, n_max=n, cnt=None):
            return lib().sf_observe_list(h, C.c_void_p(buf), phase, 1,
                                         C.c_void_p(ids.data_ptr()) if id_ptr is None else id_ptr,
                                         C.c_void_p(count.data_ptr()) if cnt is None else cnt, n_max, stream)

        sim.step_a()
        before, stats = sim.state_hash(), sim.stats()
        refused(lib().sf_reset_finished(h, stream))
        with pytest.raises(SfError):
            sim.reset_finished()
        refused(ol(obs.data_ptr()))  # P1 between the halves
        sim.step_b(sim.synth_actions(30, sfcfg.ACTIONS28))
        before, stats = sim.state_hash(), sim.stats()
        refused(ol(obs.data_ptr(), phase=sfcfg.OBS_P2))
        refused(ol(obs.data_ptr(), phase=7))
        refused(ol(None))
        refused(ol(raw[1:].data_ptr()))  # misaligned observation buffer
        refused(ol(obs.data_ptr(), n_max=0))
        refused(ol(obs.data_ptr(), n_max=n + 1))
        refused(ol(obs.data_ptr(), id_ptr=C.c_void_p(None)))
        refused(ol(obs.data_ptr(), id_ptr=C.c_void_p(ids.data_ptr() + 2)))
        refused(ol(obs.data_ptr(), cnt=C.c_void_p(count.data_ptr() + 1)))
        refused(lib().sf_observe_list(h, C.c_void_p(obs.data_ptr()), sfcfg.OBS_P1, 0, C.c_void_p(ids.data_ptr()), None,
                                      n, stream))  # empty agent mask
        refused(lib().sf_list_finished(h, None, C.c_void_p(count.data_ptr()), stream))
        refused(lib().sf_list_finished(h, C.c_void_p(ids.data_ptr()), None, stream))
        refused(lib().sf_list_finished(h, C.c_void_p(ids.data_ptr() + 2), C.c_void_p(count.data_ptr()), stream))
        assert ol(obs.data_ptr()) == 0 and ol(obs.data_ptr(), cnt=C.c_void_p(None)) == 0
        sim.reset_finished()
        assert int(sim.list_finished()[1]) == 0
    finally:
        sim.close()
