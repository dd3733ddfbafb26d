"""GPU tests of the half-precision observations (SF_OBS_F16 / SF_OBS_BF16; in Python
BatchedArena.observe(..., dtype=torch.float16 / torch.bfloat16)).

Every element the kernel writes in a half type must equal the round-to-nearest-even conversion of the element the
fp32 call writes on the same state, in the same layout and for the same rows.  Each comparison below views both as
int16 and compares bits, for both formats and both layouts:
- Squad with agents, Solo and 16-player Royale (every player), at several steps, at P1 and at P2 (split step);
- a handle whose feature table has room for 2 dynamic cells only (SF_OBS_TABLE_ROWS), so that the copy-out
  describes the others itself;
- a batch that gives every CTA several observation runs (with the library's run length and with SF_OBS_RUN), and
  a batch smaller than one wave of CTAs;
- sf_observe_list with permuted and duplicate ids, an out-of-range id and a device count below n_max, rows beyond
  the count untouched;
- six arenas against the C oracle, its fp32 observation converted by numpy (fp16) or torch (bf16);
- the device-pow fallback counter (SF_STAT_RESERVED0) moves as it does for the fp32 call;
- the errors: both flags, a misaligned buffer, an out tensor of another dtype."""
import ctypes as C

import numpy as np
import pytest

import common
from strikeforce_b200 import config as sfcfg
from test_gpu_launch_paths import _handle, _multi_pass_batch
from test_split_step import ROYALE_CAPS, SMALL, SQUAD_CAPS

pytestmark = pytest.mark.gpu

CONFIGS = {
    "squad-agents": (dict(mode="Squad", level=1, level_max=10, squad_agents=True, caps=SQUAD_CAPS), 0b1011),
    "solo": (dict(mode="Solo", level=1, level_max=10, caps=SMALL), 0b1),
    "royale16": (dict(mode="Royale", teams=[1, 2, 3, 4] * 4, caps=ROYALE_CAPS), 0xFFFF),
}


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU tests need a CUDA device; there is no CPU fallback to test")
    return torch


def _formats(torch):
    return (torch.float16, torch.bfloat16)


def _reserved0(sim):
    return int(sim.stats_tensor()[sfcfg.STAT_NAMES.index("reserved0")])


def _same_bits(torch, half, ref32, what):
    """half equals ref32.to(half.dtype) bit for bit, same shape and strides (the channels-last view included)"""
    assert half.shape == ref32.shape and half.stride() == ref32.stride(), what
    want = ref32.contiguous().to(half.dtype).view(torch.int16)
    got = half.contiguous().view(torch.int16)
    if not torch.equal(got, want):
        bad = (got != want).nonzero()[0].tolist()
        pytest.fail("%s: first difference at %s: %s vs %s" % (what, bad, half.contiguous()[tuple(bad)].item(),
                                                                 ref32.contiguous()[tuple(bad)].item()))


def _check_observe(torch, sim, mask, phase, what, **kw):
    """both layouts, both formats against the fp32 call; the fallback counter moves by the same amount"""
    for cl in (False, True):
        r0 = _reserved0(sim)
        ref = sim.observe(mask, phase, channels_last=cl, **kw)
        fb32 = _reserved0(sim) - r0
        for dt in _formats(torch):
            r0 = _reserved0(sim)
            half = sim.observe(mask, phase, channels_last=cl, dtype=dt, **kw)
            assert _reserved0(sim) - r0 == fb32, "%s: fallback count differs from fp32" % what
            _same_bits(torch, half, ref, "%s %s %s" % (what, "nhwc" if cl else "nchw", dt))


@pytest.mark.parametrize("name", list(CONFIGS))
def test_half_equals_cast_fp32_p1_and_p2(torch_cuda, monkeypatch, name):
    """Several steps of one sub-wave handle and of a handle with 2 table rows, P1 every 25 steps and P2 (between
    sf_step_a and sf_step_b) every 25 steps, offset."""
    torch = torch_cuda
    kw, mask = CONFIGS[name]
    kw = dict(kw, auto_reset=True, max_steps=150, env_id_base=300)
    sim = _handle(monkeypatch, 96, **kw)
    monkeypatch.setenv("SF_OBS_TABLE_ROWS", "2")
    small = _handle(monkeypatch, 96, **kw)
    monkeypatch.delenv("SF_OBS_TABLE_ROWS")
    try:
        for t in range(160):
            act = sim.synth_actions(t, sfcfg.ACTIONS28)
            if t % 25 == 0:
                for s, tag in ((sim, "P1"), (small, "P1 2 rows")):
                    _check_observe(torch, s, mask, sfcfg.OBS_P1, "%s %s step %d" % (name, tag, t))
            if t % 25 == 12:
                sim.step_a(), small.step_a()
                for s, tag in ((sim, "P2"), (small, "P2 2 rows")):
                    _check_observe(torch, s, mask, sfcfg.OBS_P2, "%s %s step %d" % (name, tag, t))
                sim.step_b(act), small.step_b(act)
            else:
                sim.step(act), small.step(act)
    finally:
        sim.close(), small.close()


@pytest.mark.parametrize("run", [None, 7])
def test_half_equals_cast_fp32_several_runs_per_cta(torch_cuda, monkeypatch, run):
    """A batch of 2 x (28 x SMs) + 37 arenas and three slots: every CTA writes several runs of observations (the
    library's run length; SF_OBS_RUN=7 leaves a partial last run)."""
    torch = torch_cuda
    n = _multi_pass_batch(torch)
    kw, _ = CONFIGS["squad-agents"]
    sim = _handle(monkeypatch, n, run=run, **dict(kw, auto_reset=True, max_steps=100))
    try:
        for t in range(60):
            sim.step(sim.synth_actions(t, sfcfg.ACTIONS28))
        _check_observe(torch, sim, 0b1011, sfcfg.OBS_P1, "multi-run batch, run %s" % run)
    finally:
        sim.close()


def test_half_observe_list(torch_cuda, monkeypatch):
    """sf_observe_list in half: permuted ids with duplicates and an out-of-range id (a zero row), a device count
    below n_max; rows at and beyond the count keep a sentinel; P1 and P2; the 2-row table as well."""
    torch = torch_cuda
    kw, mask = CONFIGS["squad-agents"]
    kw = dict(kw, auto_reset=True, max_steps=150)
    n = 120
    sims = [_handle(monkeypatch, n, **kw)]
    monkeypatch.setenv("SF_OBS_TABLE_ROWS", "2")
    sims.append(_handle(monkeypatch, n, **kw))
    monkeypatch.delenv("SF_OBS_TABLE_ROWS")
    rng = np.random.default_rng(11)
    ids_h = np.concatenate([rng.permutation(n)[:70], [5, 5, n + 3, 17, -1, 17]]).astype(np.int32)
    rng.shuffle(ids_h)
    n_max, cnt = len(ids_h), 61
    try:
        for s in sims:
            ids = torch.from_numpy(ids_h).to(s.device)
            count = torch.tensor([cnt], dtype=torch.int32, device=s.device)
            for t in range(90):
                act = s.synth_actions(t, sfcfg.ACTIONS28)
                if t % 30 == 29:
                    s.step_a()
                    _check_observe(torch, s, mask & ~1, sfcfg.OBS_P2, "list P2 step %d" % t, env_ids=ids)
                    s.step_b(act)
                else:
                    s.step(act)
                if t % 30 != 10:
                    continue
                _check_observe(torch, s, mask, sfcfg.OBS_P1, "list step %d" % t, env_ids=ids)
                for cl in (False, True):
                    full = s.observe(mask, channels_last=cl).contiguous()
                    for dt in _formats(torch):
                        shape = (n_max, 3) + ((31, 31, 32) if cl else (32, 31, 31))
                        out = torch.full(shape, -7.25, dtype=dt, device=s.device)
                        v = s.observe(mask, channels_last=cl, env_ids=ids, count=count, out=out, dtype=dt)
                        assert v.data_ptr() == out.data_ptr()
                        v = v.contiguous()
                        for i, e in enumerate(ids_h.tolist()):
                            if i >= cnt:
                                assert bool((out[i] == -7.25).all()), "row %d beyond the count was written" % i
                            elif 0 <= e < n:
                                _same_bits(torch, v[i], full[e], "list row %d (arena %d) %s" % (i, e, dt))
                            else:
                                assert not bool(out[i].view(torch.int16).any()), "row %d (id %d) is not zero" % (i, e)
    finally:
        for s in sims:
            s.close()


def test_half_against_the_oracle(torch_cuda, arena_data):
    """Six Squad arenas with agents and the C oracle: the oracle's fp32 observation of each slot, converted by numpy
    (float16) or torch (bfloat16), equals the device's words in both layouts."""
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    n, mask, slots = 6, 0b1011, (0, 1, 3)
    sim = BatchedArena(n, mode="Squad", level=3, squad_agents=True, auto_reset=False)
    oracles = common.make_oracles(arena_data, n, sfcfg.MODE_SQUAD, 3, squad_agents=True)
    checked = 0
    try:
        for t in range(100):
            act = sim.synth_actions(t, sfcfg.ACTIONS28)
            sim.step(act)
            act_h = act.cpu().numpy()
            for e, o in enumerate(oracles):
                o.step(bytes(act_h[e]))
            if t % 20 != 19:
                continue
            for dt in _formats(torch):
                a = sim.observe(mask, dtype=dt).cpu()
                b = sim.observe(mask, channels_last=True, dtype=dt).contiguous().cpu()
                for e, o in enumerate(oracles):
                    for j, slot in enumerate(slots):
                        try:
                            ref = o.observe(slot)
                        except RuntimeError:
                            continue
                        if dt == torch.float16:
                            want = torch.from_numpy(ref.astype(np.float16).view(np.int16))
                        else:
                            want = torch.from_numpy(ref.copy()).to(torch.bfloat16).view(torch.int16)
                        for v in (a, b):
                            assert torch.equal(v[e, j].reshape(-1).view(torch.int16), want), \
                                "env %d slot %d step %d %s" % (e, slot, t, dt)
                        checked += 1
        assert checked >= 2 * n, checked
    finally:
        sim.close()


def test_half_errors(torch_cuda):
    """Both flags at once and a misaligned buffer are SF_ERR_ARG; an out tensor of another dtype is refused in
    Python."""
    from strikeforce_b200.lib import SfError, lib
    from strikeforce_b200.sim import BatchedArena
    torch = torch_cuda
    sim = BatchedArena(4, mode="Solo", level=1)
    try:
        buf = torch.zeros(4 * sfcfg.OBS_LEN + 8, dtype=torch.float16, device=sim.device)
        with pytest.raises(SfError):
            sim._chk(lib().sf_observe(sim._h, C.c_void_p(buf.data_ptr()), sfcfg.OBS_P1 | sfcfg.OBS_F16 | sfcfg.OBS_BF16,
                                      1, sim._stream()))
        ids = torch.arange(4, dtype=torch.int32, device=sim.device)
        with pytest.raises(SfError):
            sim._chk(lib().sf_observe_list(sim._h, C.c_void_p(buf.data_ptr()),
                                           sfcfg.OBS_P1 | sfcfg.OBS_NHWC | sfcfg.OBS_F16 | sfcfg.OBS_BF16, 1,
                                           C.c_void_p(ids.data_ptr()), None, 4, sim._stream()))
        for fmt in (sfcfg.OBS_F16, sfcfg.OBS_BF16):
            with pytest.raises(SfError):
                sim._chk(lib().sf_observe(sim._h, C.c_void_p(buf.data_ptr() + 8), sfcfg.OBS_P1 | fmt, 1, sim._stream()))
            sim._chk(lib().sf_observe(sim._h, C.c_void_p(buf.data_ptr() + 16), sfcfg.OBS_P1 | fmt, 1, sim._stream()))
        for dt, other in ((torch.float16, torch.bfloat16), (torch.bfloat16, torch.float32), (torch.float32, torch.float16)):
            out = torch.empty((4, 1, 32, 31, 31), dtype=other, device=sim.device)
            with pytest.raises(AssertionError):
                sim.observe(1, out=out, dtype=dt)
        torch.cuda.synchronize()
    finally:
        sim.close()
