"""The half-precision observation flags of the C header (SF_OBS_F16 / SF_OBS_BF16) and their Python mirror."""
import os
import re

from strikeforce_b200 import config as sfcfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _const(name):
    hdr = open(os.path.join(ROOT, "include", "strikeforce_b200.h")).read()
    m = re.search(r"\b%s\s*=\s*(0x[0-9A-Fa-f]+|\d+)" % name, hdr)
    assert m, name + " is not defined in the header"
    return int(m.group(1), 0)


def test_half_flags_match_the_header():
    assert (_const("SF_OBS_F16"), _const("SF_OBS_BF16")) == (sfcfg.OBS_F16, sfcfg.OBS_BF16)


def test_half_flags_are_distinct_bits_beside_the_phase_and_layout():
    others = sfcfg.OBS_P1 | sfcfg.OBS_P2 | sfcfg.OBS_NHWC
    for flag in (sfcfg.OBS_F16, sfcfg.OBS_BF16):
        assert flag & (flag - 1) == 0, "one bit each"
        assert flag & others == 0
    assert sfcfg.OBS_F16 != sfcfg.OBS_BF16
