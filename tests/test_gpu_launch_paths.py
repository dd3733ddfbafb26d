"""GPU tests of the launch paths the other parity tests do not reach: the split step (sf_step_a, the P2
observation point, sf_step_b) against sf_step and against the C oracle, bots.play with episodes that end
inside half A, and the launch shapes of the persistent step kernel and of sf_observe -- several passes of
the chunk loop, 1 to 32 arenas per warp, a partial last chunk, idle lanes, partial and repeated
observation runs -- all picked per handle with SF_LANES_PER_WARP / SF_OBS_RUN at sf_create."""
import math

import numpy as np
import pytest

import common
import sfo
from strikeforce_b200 import config as sfcfg
from test_split_step import ROYALE_CAPS, SMALL, SQUAD_CAPS

pytestmark = pytest.mark.gpu

ABORTS = (sfcfg.OVERFLOW, sfcfg.UB_GUARD)
WARPS_PER_SM = 28  # SF_CTA / 32: one persistent CTA of 896 threads per SM (sf_lib.cu)
GPU_CONFIGS = {
    "solo": dict(mode="Solo", level=1, level_max=10, caps=SMALL),
    "timer": dict(mode="Timer", level=1, level_max=10, caps=SMALL, player="synthetic"),
    "squad-agents": dict(mode="Squad", level=1, level_max=10, squad_agents=True, caps=SQUAD_CAPS),
    "royale16": dict(mode="Royale", teams=[1, 2, 3, 4] * 4, caps=ROYALE_CAPS),
}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _warp_slots(torch):
    return WARPS_PER_SM * torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _multi_pass_batch(torch):
    """3 passes of the chunk loop at 1 arena per warp, 2 at 2, and a partial last chunk at every width"""
    return 2 * _warp_slots(torch) + 37


def _handle(monkeypatch, n, lanes=None, run=None, **kw):
    """a BatchedArena whose sf_create saw SF_LANES_PER_WARP / SF_OBS_RUN (None: the library's own choice)"""
    from strikeforce_b200.sim import BatchedArena
    for var, v in (("SF_LANES_PER_WARP", lanes), ("SF_OBS_RUN", run)):
        if v is None:
            monkeypatch.delenv(var, raising=False)
        else:
            monkeypatch.setenv(var, str(v))
    try:
        return BatchedArena(n, **kw)
    finally:
        monkeypatch.delenv("SF_LANES_PER_WARP", raising=False)
        monkeypatch.delenv("SF_OBS_RUN", raising=False)


def _first_diff(a, b):
    rows = (a != b).reshape(a.shape[0], -1).any(1).nonzero()
    return int(rows[0]) if len(rows) else None


@pytest.mark.parametrize("batch", ["sub-wave", "multi-pass"])
@pytest.mark.parametrize("name", list(GPU_CONFIGS))
def test_split_step_equals_full_step(torch_cuda, monkeypatch, name, batch):
    """Two handles on the same seeds and actions, one stepped with sf_step and one with sf_step_a +
    sf_step_b: state hashes, sf_step_out and the statistics of all arenas after every step.  With the small
    capacities many episodes end inside half A; the multi-pass batch runs at one arena per warp."""
    torch = torch_cuda
    n, lanes = (200, None) if batch == "sub-wave" else (_multi_pass_batch(torch), 1)
    kw = dict(GPU_CONFIGS[name], auto_reset=True, max_steps=150, env_id_base=300)
    full = _handle(monkeypatch, n, lanes, **kw)
    split = _handle(monkeypatch, n, lanes, **kw)
    aborts = torch.tensor(ABORTS, dtype=torch.int32, device=full.device)
    try:
        aborts_in_a = torch.zeros((), dtype=torch.int64, device=full.device)
        for t in range(400):
            act = full.synth_actions(t, sfcfg.ACTIONS28)
            full.step(act)
            split.step_a()
            aborts_in_a += torch.isin(split.step_out()[:, 0], aborts).sum()  # with auto-reset every arena starts the step running
            split.step_b(act)
            a, b = split.step_out(), full.step_out()
            assert torch.equal(a, b), "step_out: step %d arena %s: %s vs %s" % (
                t, _first_diff(a, b), a[_first_diff(a, b)].tolist(), b[_first_diff(a, b)].tolist())
            a, b = split.state_hash(), full.state_hash()
            assert torch.equal(a, b), "state: step %d arena %s" % (t, _first_diff(a, b))
            assert split.stats() == full.stats(), "statistics: step %d" % t
        st = full.stats()
        assert st["steps"] + st["overflows"] + st["ub_guards"] == n * 400
        assert int(aborts_in_a) >= n // 4, "only %d episodes ended inside half A" % int(aborts_in_a)
    finally:
        full.close(), split.close()


def test_split_step_follows_the_oracle(torch_cuda, arena_data):
    """_run_parity for the split step: Squad with agent-driven squad humans and small capacities, auto-reset,
    45 arenas (a partly filled warp), the C oracle stepped half by half (sfo_step_a / sfo_step_b) and reset on
    the synthetic seed chain.  Status after each half, the whole sf_step_out of every step that ran to its end,
    the state hash after every step, and every 15 steps the P2 observations of all squad-agent slots in both
    layouts against the oracle bit for bit (arenas that ended in half A, and slots whose human is gone, have
    none)."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, base, max_steps, steps = 45, 300, 150, 300
    sim = BatchedArena(n, mode="Squad", level=1, level_max=10, squad_agents=True, caps=SQUAD_CAPS, auto_reset=True,
                       max_steps=max_steps, env_id_base=base)
    levels = [1 + (base + e) % 10 for e in range(n)]
    oracles = []
    for e in range(n):
        o = sfo.Arena(sfcfg.make_config(arena_data, mode=sfcfg.MODE_SQUAD, level_min=levels[e], squad_agents=True,
                                        caps=SQUAD_CAPS, max_steps=max_steps))
        o.reset(levels[e], common.synth_tb(base + e), common.synth_serial(base + e, 0))
        oracles.append(o)
    mask = ((1 << sim.n_agents) - 1) & ~1
    slots = [s for s in range(32) if (mask >> s) & 1]
    episode = [0] * n
    aborts_in_a = compared = 0
    try:
        for t in range(steps):
            act = sim.synth_actions(t, sfcfg.ACTIONS28)
            act_h = act.cpu().numpy()
            sim.step_a()
            out_a = sim.step_out()[:, 0].cpu().numpy()
            ended_in_a = [o.step_a() != sfcfg.RUNNING for o in oracles]
            aborts_in_a += sum(ended_in_a)
            for e, o in enumerate(oracles):
                assert out_a[e] == o.status(), "status after half A: arena %d step %d" % (e, t)
            if t % 15 == 0:
                p2 = sim.observe(mask, sfcfg.OBS_P2)
                p2_cl = sim.observe(mask, sfcfg.OBS_P2, channels_last=True)
                assert torch.equal(p2.view(torch.int32), p2_cl.contiguous().view(torch.int32)), "P2 layouts differ: step %d" % t
                p2_h = p2.cpu().numpy().reshape(n, len(slots), -1)
                for e, o in enumerate(oracles):
                    if ended_in_a[e]:
                        continue  # an episode that ended in half A has no P2 observation
                    for j, slot in enumerate(slots):
                        try:
                            ref = o.observe(slot)
                        except RuntimeError:
                            continue
                        assert (p2_h[e, j].view(np.uint32) == ref.view(np.uint32)).all(), \
                            "P2 observation: arena %d slot %d step %d" % (e, slot, t)
                        compared += 1
            sim.step_b(act)
            out = sim.step_out().cpu().numpy()
            h = sim.state_hash().cpu().numpy().view(np.uint64)
            for e, o in enumerate(oracles):
                st = o.status() if ended_in_a[e] else o.step_b(bytes(act_h[e]))
                assert out[e, 0] == st, "status: arena %d step %d: %d vs %d" % (e, t, out[e, 0], st)
                if st not in ABORTS:
                    so = o.step_out()
                    assert out[e].tolist() == [so[k] for k, _ in sfcfg.StepOut._fields_], "step_out: arena %d step %d" % (e, t)
                if st != sfcfg.RUNNING:
                    episode[e] += 1
                    o.reset(levels[e], common.synth_tb(base + e), common.synth_serial(base + e, episode[e]))
                if h[e] != np.uint64(o.state_hash()):
                    diff = sfo.diff_records(o.dump(), sim.export_env(e))
                    pytest.fail("state: arena %d step %d\n%s" % (e, t, "\n".join(diff)))
        st = sim.stats()
        assert st["episodes"] == sum(episode)
        assert st["steps"] + st["overflows"] + st["ub_guards"] == n * steps
        assert aborts_in_a >= 20, "only %d episodes ended inside half A" % aborts_in_a
        assert compared >= 1000
    finally:
        sim.close()


def test_bots_play_sees_every_episode_end(torch_cuda):
    """bots.play with agent-driven squad humans splits every step; with small capacities many episodes end in
    half A.  Every step of every arena is counted once (ran to its end, or aborted), and every episode that
    ended reaches Custom.new_games, which resets the recurrent rows of that arena's agents."""
    from strikeforce_b200 import bots
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, steps = 512, 200
    sim = BatchedArena(n, mode="Squad", level=1, level_max=10, squad_agents=True, caps=SQUAD_CAPS, auto_reset=True,
                       max_steps=120)
    aborts = torch.tensor(ABORTS, dtype=torch.int32, device=sim.device)

    class Counting(bots.Custom):
        def __init__(self):
            super().__init__(bots.RandomAgent(9, seed=11, device=sim.device))
            self.done = torch.zeros((), dtype=torch.int64, device=sim.device)
            self.aborts_in_a = torch.zeros((), dtype=torch.int64, device=sim.device)
            self.mid_step = False

        def bot(self, s, agent_mask=1, phase=sfcfg.OBS_P1):
            self.mid_step = phase == sfcfg.OBS_P2
            return super().bot(s, agent_mask, phase)

        def view(self, s):  # called between sf_step_a and sf_step_b, and again after the step
            if self.mid_step:
                self.aborts_in_a += torch.isin(s.step_out()[:, 0], aborts).sum()
                self.mid_step = False

        def new_games(self, s, done):
            self.done += done.sum()
            super().new_games(s, done)

    try:
        c = Counting()
        stats = bots.play(sim, c, steps)
        assert stats["steps"] + stats["overflows"] + stats["ub_guards"] == n * steps
        assert int(c.done) == stats["episodes"], "%d episode ends reached new_games, %d ended" % (int(c.done), stats["episodes"])
        assert int(c.aborts_in_a) >= 10, "only %d episodes ended inside half A" % int(c.aborts_in_a)
    finally:
        sim.close()


# (SF_LANES_PER_WARP, SF_OBS_RUN) per handle; None = the library's choice
LAUNCH_SHAPES = [(None, None), (1, 1), (2, 7), (4, 16), (8, 2), (16, 13), (32, 11)]


def test_launch_shapes_play_the_same_trajectories(torch_cuda, arena_data, monkeypatch):
    """One handle per launch shape on the same batch of 2 x (28 x SMs) + 37 arenas: at 1 arena per warp the
    step kernel makes 3 passes, at 2 it makes 2, every width has a partial last chunk, and the idle lanes of
    narrow warps read the headers of arenas 0-31 while other warps step them.  Squad with agents, levels 1-10,
    the 28-symbol alphabet, auto-reset, 256 steps; a trajectory checksum of every arena (the state hash after
    every step folded on the device) must agree in every handle, and with the C oracle for a sample that holds
    arenas 0-31, the last 40 and random ones.  Twice the observations of three slots, in both layouts, must be
    the same bits in every handle (several observation runs per CTA, partial last runs) and match the oracle
    for the sample, the very last item included."""
    torch = torch_cuda
    slots = _warp_slots(torch)
    n = _multi_pass_batch(torch)
    passes = {lpw: math.ceil(math.ceil(n / lpw) / slots) for lpw in (1, 2, 4, 8, 16, 32)}  # of the chunk loop
    assert passes[1] >= 3 and passes[2] >= 2, passes
    mask = (1 << 0) | (1 << 4) | (1 << 9)
    nsel = 3
    assert any(r and (n * nsel) % r for _, r in LAUNCH_SHAPES), "no observation handle has a partial last run"
    steps, max_steps, obs_at = 256, 100, (97, 256)
    kw = dict(mode="Squad", level=1, level_max=10, squad_agents=True, auto_reset=True, max_steps=max_steps)
    rng = np.random.default_rng(8)
    sample = sorted(set(range(32)) | set(range(n - 40, n)) | set(rng.integers(32, n - 40, size=24).tolist()))
    oracles, episode = {}, {e: 0 for e in sample}
    for e in sample:
        lvl = 1 + e % 10
        o = sfo.Arena(sfcfg.make_config(arena_data, mode=sfcfg.MODE_SQUAD, level_min=lvl, squad_agents=True,
                                        max_steps=max_steps))
        o.reset(lvl, common.synth_tb(e), common.synth_serial(e, 0))
        oracles[e] = o
    ref_chk = {e: 0 for e in sample}
    handles = []
    try:
        for lanes, run in LAUNCH_SHAPES:
            handles.append(_handle(monkeypatch, n, lanes, run, **kw))
        dev = handles[0].device
        idx = torch.tensor(sample, device=dev)
        chk = [torch.zeros(n, dtype=torch.int64, device=dev) for _ in handles]
        last_compared = 0

        def check_observations(t):
            nonlocal last_compared
            ref = handles[0].observe(mask)
            for i, h in enumerate(handles):
                for cl in (False, True):
                    if i == 0 and not cl:
                        continue
                    v = h.observe(mask, channels_last=cl).contiguous()
                    assert torch.equal(ref.view(torch.int32), v.view(torch.int32)), \
                        "observations differ: handle %s %s step %d" % (LAUNCH_SHAPES[i], "nhwc" if cl else "nchw", t)
                    del v
            picked = ref[idx].reshape(len(sample), nsel, -1).cpu().numpy()
            del ref
            for i, e in enumerate(sample):
                for j, slot in enumerate((0, 4, 9)):
                    try:
                        want = oracles[e].observe(slot)
                    except RuntimeError:
                        continue
                    assert (picked[i, j].view(np.uint32) == want.view(np.uint32)).all(), \
                        "observation: arena %d slot %d step %d" % (e, slot, t)
                    last_compared += e == n - 1 and slot == 9
            torch.cuda.empty_cache()

        for t in range(steps):
            if t in obs_at:
                check_observations(t)
            act = handles[0].synth_actions(t, sfcfg.ACTIONS28)
            for i, h in enumerate(handles):
                h.step(act)
                chk[i] = common.torch_mix64(torch, chk[i] ^ h.state_hash())
            ref_act = common.synth_actions(sample, handles[0].n_agents, t, sfcfg.ACTIONS28)
            for i, e in enumerate(sample):  # sfo_run_trace's loop: step, reset an ended episode, fold the hash
                o = oracles[e]
                if o.step(bytes(ref_act[i])) != sfcfg.RUNNING:
                    episode[e] += 1
                    o.reset(1 + e % 10, common.synth_tb(e), common.synth_serial(e, episode[e]))
                ref_chk[e] = common.mix64(ref_chk[e] ^ o.state_hash())
        if steps in obs_at:
            check_observations(steps)
        assert last_compared == len(obs_at), "the last observation item was compared %d times" % last_compared

        for i, h in enumerate(handles[1:], 1):
            assert torch.equal(chk[i], chk[0]), "trajectories differ: handle %s, first arena %s" % (
                LAUNCH_SHAPES[i], _first_diff(chk[i], chk[0]))
        got = chk[0][idx].cpu().numpy().view(np.uint64)
        bad = [e for i, e in enumerate(sample) if got[i] != np.uint64(ref_chk[e])]
        assert not bad, "%d of %d trajectories differ from the oracle, first: arena %d" % (len(bad), len(sample), bad[0])
        stats = [h.stats() for h in handles]
        for i, st in enumerate(stats):
            assert st == stats[0], "statistics differ: handle %s" % (LAUNCH_SHAPES[i],)
            assert st["steps"] + st["overflows"] + st["ub_guards"] == n * steps
        assert stats[0]["episodes"] >= 2 * n  # max_steps alone ends every episode within 100 steps
    finally:
        for h in handles:
            h.close()
