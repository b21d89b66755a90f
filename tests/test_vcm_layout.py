"""dvbs2fec_vcm_layout: the packed layout of a VCM / ACM batch, on the host (no handle, no device).  Every valid
(MODCOD, frame size, pilots) configuration and the DUMMY PLFRAME take the sizes dvbs2fec_modcod_info states; every
descriptor without an LDPC code fails the call with EINVAL, names the frame and leaves the output arrays alone."""
import ctypes as C

import numpy as np
import pytest

from fec import pkg

SHORT_9_10 = {11, 17, 23, 28}


def configurations():
    return [(m, s, p) for m in range(1, 29) for s in (0, 1) for p in (0, 1) if not (s and m in SHORT_9_10)]


def expected(desc):
    sizes = []
    for modcod, short, pilots, _ in desc:
        if modcod == 0:
            sizes.append((90 + 36 * 90, 0, 0))
        else:
            info = pkg.modcod_info(modcod, bool(short), bool(pilots))
            sizes.append((info["plframe_symbols"], info["nldpc"], info["kbch"] // 8))
    s = np.array(sizes, np.int64).reshape(-1, 3)
    return [np.concatenate([[0], np.cumsum(s[:, k])]) for k in range(3)]


def test_every_configuration_and_dummy():
    cfgs = configurations()
    assert len(cfgs) == 104
    rng = np.random.default_rng(3)
    desc = [(m, s, p, int(rng.integers(-5, 5))) for m, s, p in cfgs] + [(0, 0, 0, 0), (0, 1, 1, 7)]   # 4th field ignored
    desc = np.array([desc[i] for i in rng.permutation(len(desc))], np.int32)
    got = pkg.vcm_layout(desc)
    for g, w in zip(got, expected(desc)):
        assert np.array_equal(g, w)
    # nonzero shortframes / pilots values count as set, like set_modcod's
    d2 = desc.copy()
    d2[:, 1] *= 5
    d2[:, 2] *= -3
    for g, w in zip(pkg.vcm_layout(d2), got):
        assert np.array_equal(g, w)
    # BBFRAME offsets are not aligned: normal 1/4 is 2001 bytes
    assert pkg.vcm_layout([[1, 0, 0, 0]])[2].tolist() == [0, 2001]
    assert [x.tolist() for x in pkg.vcm_layout(np.zeros((0, 4), np.int32))] == [[0], [0], [0]]


def test_null_outputs_are_skipped():
    L = pkg.lib()
    d = np.array([[4, 0, 0, 0], [0, 0, 0, 0]], np.int32)
    bb = np.full(3, -1, np.int64)
    assert L.dvbs2fec_vcm_layout(2, d.ctypes.data_as(C.c_void_p), None, None, bb.ctypes.data_as(C.c_void_p)) == 0
    assert bb.tolist() == [0, 4026, 4026]


@pytest.mark.parametrize("bad", [(29, 0, 0), (31, 0, 0), (-1, 0, 0), (11, 1, 0), (17, 1, 1), (23, 1, 0), (28, 1, 1),
                                 (1000, 0, 0), (-2 ** 31, 0, 0)])
def test_invalid_descriptor(bad):
    L = pkg.lib()
    d = np.array([[4, 0, 0, 0], [0, 0, 0, 0], [bad[0], bad[1], bad[2], 0]], np.int32)
    outs = [np.full(4, 0x5A5A5A5A, np.int64) for _ in range(3)]
    rc = L.dvbs2fec_vcm_layout(3, d.ctypes.data_as(C.c_void_p), *[o.ctypes.data_as(C.c_void_p) for o in outs])
    assert rc == pkg.EINVAL
    assert "frame 2" in L.dvbs2fec_last_error().decode()
    assert all((o == 0x5A5A5A5A).all() for o in outs)
    with pytest.raises(pkg.DVBS2FecError):
        pkg.vcm_layout(d)


def test_bad_arguments():
    L = pkg.lib()
    out = np.full(2, 7, np.int64)
    assert L.dvbs2fec_vcm_layout(-1, None, out.ctypes.data_as(C.c_void_p), None, None) == pkg.EINVAL
    assert L.dvbs2fec_vcm_layout(1, None, out.ctypes.data_as(C.c_void_p), None, None) == pkg.EINVAL
    assert out.tolist() == [7, 7]
    assert L.dvbs2fec_vcm_layout(0, None, out.ctypes.data_as(C.c_void_p), None, None) == 0
    assert out.tolist() == [0, 7]
