"""CPU checks of what tests/test_gpu_ldpc_variants.py relies on: the tiled batches never put the same frame at two
positions a kernel could confuse, and its model of the LDPC kernel choice matches the codes and the compiled
instantiations."""
import ctypes as C
import glob
import os
import re

import numpy as np
import pytest

import ldpc_variant_worker as W
from orclib import ALL_CODES, code_params, oracle

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "sdrpp-dvbs-demodulator_b200", "csrc")


@pytest.mark.parametrize("sms", [132, 148, 160])
def test_tiling_separates_confusable_positions(sms):
    n = W.batch_size(sms)
    assert n % 2 == 1 and n >= 8 * sms * 3
    content = W.tile(n)
    assert content.min() == 0 and content.max() == W.M - 1
    offsets = set(W.CONFUSABLE_OFFSETS) | {sms * 2, sms * 3, sms * 4, sms * 6}   # grids and their pairs on this part
    for d in sorted(offsets):
        assert not (content[d:] == content[:-d]).any(), d
    # a pair's partners differ, and every frame sits in lane A and in lane B, beside a different partner in each
    a, b = content[0:n - 1:2], content[1::2]
    assert not (a == b).any()
    for c in range(W.M):
        assert (a == c).any() and (b == c).any(), c
        assert set(b[a == c].tolist()) == {(c + W.STEP) % W.M} and set(a[b == c].tolist()) == {(c - W.STEP) % W.M}, c


def test_tiling_needs_the_prime():
    """a frame repeats only at multiples of M"""
    content = W.tile(10 * W.M)
    for d in range(1, 3 * W.M + 1):
        assert (content[d:] == content[:-d]).any() == (d % W.M == 0), d


@pytest.mark.parametrize("short,rate", ALL_CODES)
def test_code_links_match_the_oracle_schedule(short, rate):
    p = code_params(short, rate)
    cnc = np.zeros(p["N"] - p["K"], np.uint8)
    max_cnt = oracle().orc_ldpc_schedule(short, rate, None, cnc.ctypes.data_as(C.c_void_p))
    per_layer = cnc[: p["q"]]      # check i of layer i: every row of a layer has the same degree
    assert W.CODE_LINKS[(short, rate)] == (max_cnt, bool((per_layer == max_cnt).all()))


def _macro_list(pattern, macro_re):
    out = {}
    for path in sorted(glob.glob(os.path.join(CSRC, pattern))):
        for m in re.finditer(macro_re, open(path).read()):
            form, cnt = m.group(1), int(m.group(2))
            out[cnt] = {"U": "U", "B": "UR", "R": "R"}[form]
    return out


def test_instantiation_tables_match_the_sources():
    one = _macro_list("ldpc_inst_*.cu", r"\bV([UBR])\((\d+)\)")
    assert one == W.ONE_LANE
    assert _macro_list("ldpc2_inst_*.cu", r"\bV2([UBR])\((\d+)\)") == W.ONE_LANE
    assert _macro_list("ldpc2l_inst_*.cu", r"\bV2L([UR])\((\d+)\)") == W.TWO_LANES


def test_every_compiled_instantiation_is_reachable():
    """each code selects exactly one instantiation for a setting of the overrides; none is compiled for nothing"""
    reach = W.reachable_instantiations()
    assert reach == W.compiled_instantiations()
    assert len(reach) == 198


def test_kernel_names_parse():
    assert W.parse_kernel("void s2::v2::ldpc_v2_kernel<9, false, true, 3>(s2::LdpcParams2)") == ("ldpc_v2_kernel", 9, False, True, 3)
    assert W.parse_kernel("void s2::v2::ldpc_v2l_kernel<17, true, false>(s2::LdpcParams2)") == ("ldpc_v2l_kernel", 17, True, False)
    assert W.parse_kernel("void s2::(anonymous namespace)::ldpc_pair_kernel<5, false, true, true, 2>(s2::LdpcParams)") == \
        ("ldpc_pair_kernel", 5, False, True, True, 2)
    assert W.parse_kernel("void s2::bch_kernel(s2::BchArgs)") is None
