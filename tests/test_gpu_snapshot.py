"""GPU tests of arena records (sf_save / sf_load, BatchedArena.save / load / clone): restore in place, checkpoint
and resume in a fresh handle, clones under other global ids against the C oracle, one root broadcast into many
slots, the record bytes against the host-check build, and the argument errors.  The configurations and small
capacities are those of test_gpu_launch_paths.py, so that many episodes end after a load."""
import numpy as np
import pytest

import common
import snapcheck
import sfo
from strikeforce_b200 import config as sfcfg
from test_gpu_launch_paths import GPU_CONFIGS, _first_diff, _handle, _multi_pass_batch

pytestmark = pytest.mark.gpu

BASE, MAX_STEPS = 300, 150


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _kw(name, **extra):
    return dict(GPU_CONFIGS[name], auto_reset=True, max_steps=MAX_STEPS, env_id_base=BASE, **extra)


def _run(sim, t0, steps):
    """steps from global step t0: per-step state hashes and sf_step_out (device tensors), then the P1
    observation of the player in both layouts"""
    hashes, outs = [], []
    for t in range(t0, t0 + steps):
        sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
        hashes.append(sim.state_hash())
        outs.append(sim.step_out())
    return hashes, outs, sim.observe(1).clone(), sim.observe(1, channels_last=True).contiguous().clone()


def _assert_same_run(torch, a, b):
    for t, (x, y) in enumerate(zip(a[0], b[0])):
        assert torch.equal(x, y), "state: step %d arena %s" % (t, _first_diff(x, y))
    for t, (x, y) in enumerate(zip(a[1], b[1])):
        assert torch.equal(x, y), "step_out: step %d arena %s" % (t, _first_diff(x, y))
    assert torch.equal(a[2].view(torch.int32), b[2].view(torch.int32)), "P1 observation"
    assert torch.equal(a[3].view(torch.int32), b[3].view(torch.int32)), "P1 observation, channels innermost"


def _ends(outs):
    return int(sum(int((o[:, 0] != sfcfg.RUNNING).sum()) for o in outs))


@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_restore_in_place(torch_cuda, monkeypatch, name, batch):
    """Step T1, save all arenas, step T2, load the records, replay T2 with the same actions: every per-step hash
    and sf_step_out and the final P1 observations (both layouts) equal the first run, across auto-resets.
    save -> load -> save gives the same bytes, and neither call touches the statistics."""
    torch = torch_cuda
    n, lanes = (200, None) if batch == "sub-wave" else (_multi_pass_batch(torch), 1)
    sim = _handle(monkeypatch, n, lanes, **_kw(name))
    try:
        _run(sim, 0, 60)
        stats = sim.stats()
        rec = sim.save()
        assert rec.shape == (n, sim.snapshot_bytes) and sim.snapshot_bytes % 128 == 0
        assert sim.stats() == stats
        first = _run(sim, 60, 150)
        assert _ends(first[1]) >= n // 4, "too few episodes ended after the save"
        stats = sim.stats()
        sim.load(rec)
        assert sim.stats() == stats
        assert torch.equal(sim.save(), rec), "save after load"
        _assert_same_run(torch, first, _run(sim, 60, 150))
    finally:
        sim.close()


@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_checkpoint_and_resume(torch_cuda, name):
    """Handle A runs T1 + T2 steps.  Handle B, created fresh with the same configuration, loads A's records of
    step T1 after a round trip through host memory and runs T2: every per-step hash and sf_step_out and the
    final observations equal A's.  B's statistics count B's own steps only."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 200
    a = BatchedArena(n, **_kw(name))
    b = None
    try:
        _run(a, 0, 70)
        ckpt = a.save().cpu().numpy()
        ref = _run(a, 70, 160)
        assert _ends(ref[1]) >= n // 4
        b = BatchedArena(n, **_kw(name))
        b.load(ckpt)
        got = _run(b, 70, 160)
        _assert_same_run(torch, ref, got)
        st = b.stats()
        assert st["steps"] + st["overflows"] + st["ub_guards"] == n * 160
    finally:
        a.close()
        if b is not None:
            b.close()


@pytest.mark.parametrize("name", ["solo", "timer", "squad-agents"])
def test_clone_follows_the_oracle(torch_cuda, arena_data, name):
    """Arenas 0..7 of a handle with env_id_base 900 are followed by the C oracle from their first step; at step
    T1 they are cloned into slots 40..47 (other global ids) and the oracles follow those: the episode goes on bit
    for bit, and every later episode of a slot starts from the slot's own level and seeds synth(ge, episode + 1).
    Squad with agents runs the split step and compares the P2 observations of every agent slot (both layouts)."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    kw = dict(GPU_CONFIGS[name], auto_reset=True, max_steps=MAX_STEPS, env_id_base=900)
    n, src, dst, T1, steps = 64, list(range(8)), list(range(40, 48)), 80, 480
    split = name == "squad-agents"
    sim = BatchedArena(n, **kw)
    lo, hi = kw.get("level", 1), kw.get("level_max", kw.get("level", 1))
    level = lambda ge: lo + ge % (hi - lo + 1)  # noqa: E731
    ocfg = dict(mode=sfcfg.MODES[kw["mode"]], squad_agents=kw.get("squad_agents", False), caps=kw["caps"],
                max_steps=MAX_STEPS, player=kw.get("player", "account1"))
    oracles, ges, episode = [], [900 + e for e in src], [0] * len(src)
    for ge in ges:
        o = sfo.Arena(sfcfg.make_config(arena_data, level_min=level(ge), **ocfg))
        o.reset(level(ge), common.synth_tb(ge), common.synth_serial(ge, 0))
        oracles.append(o)
    mask = ((1 << sim.n_agents) - 1) & ~1
    slots = [s for s in range(32) if (mask >> s) & 1]
    dst_ends = compared = 0
    try:
        for t in range(steps):
            if t == T1:
                sim.clone(src, dst)
                ges = [900 + e for e in dst]
                h = sim.state_hash().cpu().numpy()
                assert (h[dst] == h[src]).all()
            rows = src if t < T1 else dst
            act = sim.synth_actions(t, sfcfg.ACTIONS28)
            act_h = act.cpu().numpy()
            if split:
                sim.step_a()
                ended_a = [o.step_a() != sfcfg.RUNNING for o in oracles]
                if t >= T1 and t % 10 == 0:
                    p2 = sim.observe(mask, sfcfg.OBS_P2)
                    p2_cl = sim.observe(mask, sfcfg.OBS_P2, channels_last=True)
                    assert torch.equal(p2.view(torch.int32), p2_cl.contiguous().view(torch.int32))
                    p2_h = p2.cpu().numpy().reshape(n, len(slots), -1)
                    for i, o in enumerate(oracles):
                        if ended_a[i]:
                            continue
                        for j, slot in enumerate(slots):
                            try:
                                ref = o.observe(slot)
                            except RuntimeError:
                                continue
                            assert (p2_h[rows[i], j].view(np.uint32) == ref.view(np.uint32)).all(), \
                                "P2 observation: arena %d slot %d step %d" % (rows[i], slot, t)
                            compared += 1
                sim.step_b(act)
                sts = [o.status() if ended_a[i] else o.step_b(bytes(act_h[rows[i]])) for i, o in enumerate(oracles)]
            else:
                sim.step(act)
                sts = [o.step(bytes(act_h[rows[i]])) for i, o in enumerate(oracles)]
            out = sim.step_out().cpu().numpy()
            h = sim.state_hash().cpu().numpy().view(np.uint64)
            for i, o in enumerate(oracles):
                e = rows[i]
                assert out[e, 0] == sts[i], "status: arena %d step %d" % (e, t)
                if sts[i] != sfcfg.RUNNING:
                    episode[i] += 1
                    dst_ends += t >= T1
                    o.reset(level(ges[i]), common.synth_tb(ges[i]), common.synth_serial(ges[i], episode[i]))
                assert h[e] == np.uint64(o.state_hash()), "state: arena %d step %d" % (e, t)
        assert dst_ends >= 8, "only %d episodes of the clones ended" % dst_ends
        assert compared >= (200 if split else 0)
    finally:
        sim.close()


def test_broadcast_one_root(torch_cuda):
    """One root into 1,000 slots through rows: stepped with identical action rows, the slots stay hash-identical
    with the root until their first episode end, which they all reach at the same step."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 1024
    sim = BatchedArena(n, **_kw("squad-agents"))
    try:
        for t in range(30):
            sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
        sim.clone([0] * 1000, list(range(1, 1001)))
        ended = None
        for t in range(30, 30 + 400):
            act = sim.synth_actions(t, sfcfg.ACTIONS28)
            act[:] = act[0]
            sim.step(act)
            h, st = sim.state_hash()[:1001], sim.step_out()[:1001, 0]
            if ended is None:
                if bool((st != sfcfg.RUNNING).any()):
                    assert bool((st == st[0]).all()), "the copies ended at different steps"
                    ended = t
                    break
                assert bool((h == h[0]).all()), "step %d: %d copies differ" % (t, int((h != h[0]).sum()))
        assert ended is not None, "no episode ended"
    finally:
        sim.close()


@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_record_bytes(torch_cuda, name):
    """Records of all arenas (consecutive ids: coalesced reads) equal, row for row, those of a random
    permutation, of a partial list and of a list with duplicates; and they equal hc_save of the host-check build
    after the same seeds and actions, byte for byte."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, steps = 100, 150
    kw = _kw(name)
    sim = BatchedArena(n, **kw)
    hkw = dict(mode=sfcfg.MODES[kw["mode"]], level_min=kw.get("level", 1), level_max=kw.get("level_max"),
               squad_agents=kw.get("squad_agents", False), caps=kw["caps"], player=kw.get("player", "account1"),
               teams=kw.get("teams"))
    hs = snapcheck.SnapSim(sfcfg.make_config(sim.arena, n_envs=n, auto_reset=True, max_steps=MAX_STEPS, env_id_base=BASE, **hkw))
    try:
        assert hs.snapshot_bytes == sim.snapshot_bytes
        for t in range(steps):
            act = sim.synth_actions(t, sfcfg.ACTIONS28)
            sim.step(act)
            hs.step(act.cpu().numpy().tobytes())
        rec = sim.save()
        rng = np.random.default_rng(5)
        perm = rng.permutation(n)
        assert torch.equal(sim.save(perm), rec[torch.as_tensor(perm, device=rec.device)])
        for ids in ([7], [5, 7, 7, 99, 0, 5], list(range(31, 64)), list(rng.integers(0, n, 77))):
            assert torch.equal(sim.save(ids), rec[torch.as_tensor(ids, device=rec.device)]), ids
        host = rec.cpu().numpy()
        for e in range(n):
            ref = hs.save(e)
            if not (host[e] == ref).all():
                pytest.fail("arena %d: device record differs from hc_save at bytes %s" % (e, np.nonzero(host[e] != ref)[0][:16]))
    finally:
        sim.close()


def test_errors(torch_cuda, arena_data):
    """SF_ERR_ARG between the halves of a split step, for out-of-range ids, duplicate destinations, a bad rows
    entry, a misaligned buffer and a record of another configuration; a refused load changes no arena."""
    from strikeforce_b200.lib import SfError
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n = 64
    sim = BatchedArena(n, **_kw("squad-agents"))
    other = BatchedArena(n, **dict(_kw("squad-agents"), caps=dict(GPU_CONFIGS["squad-agents"]["caps"], cap_chests=77)))
    try:
        for t in range(20):
            sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
        rec = sim.save()

        def refused(fn, *args, **kw):
            with pytest.raises(SfError) as ei:
                fn(*args, **kw)
            assert ei.value.code == -1, str(ei.value)
            assert torch.equal(sim.state_hash(), before)

        sim.step_a()
        before = sim.state_hash()
        refused(sim.save)
        refused(sim.load, rec)
        sim.step_b(sim.synth_actions(20, sfcfg.ACTIONS28))
        before = sim.state_hash()
        rec = sim.save()
        refused(sim.save, [n])
        refused(sim.save, [-1])
        refused(sim.load, rec[:2], [n, 0])
        refused(sim.load, rec[:2], [3, 3])
        refused(sim.load, rec[:2], [3, 4], rows=[0, 2])
        refused(sim.load, rec[:2], [3, 4], rows=[0, -1])
        raw = torch.zeros(2 * sim.snapshot_bytes + 16, dtype=torch.uint8, device=sim.device)
        refused(sim.save, [0, 1], out=raw[1:1 + 2 * sim.snapshot_bytes].view(2, -1))
        mis = raw[8:8 + 2 * sim.snapshot_bytes].view(2, -1)
        mis.copy_(rec[:2])
        refused(sim.load, mis, [3, 4])
        assert other.snapshot_bytes == sim.snapshot_bytes
        foreign = other.save([0])
        refused(sim.load, foreign, [3])
        refused(sim.load, torch.cat([rec[:1], foreign]), [3, 4])  # all or nothing
        stats_now = sim.stats()
        sim.load(rec[:2], [3, 4])
        sim.clone([5], [6])
        assert sim.stats() == stats_now
    finally:
        sim.close(), other.close()
