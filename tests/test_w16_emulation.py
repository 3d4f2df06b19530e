"""The warp-per-pair register kernel's row sweep (w16::warp_sweep, bsw_warp16.cuh: the 32 lanes of a warp per pair,
the row in registers) executed on the CPU -- one host thread per lane, the warp's shuffles / REDUX / __syncwarp as
barrier-separated exchanges, the DPX .S16x2 instructions emulated (tests/emu/w16_emu.cu) -- compared bit for bit
with the oracle and the golden vectors.  Every lane must end each pair with the same state (the emulation aborts
otherwise) and no 16-bit lane may wrap."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from conftest import GOLDEN_CASES, load_golden, results_matrix

MAX_QLEN = 255            # w16::MAX_QLEN


@pytest.fixture(scope="module")
def emu():
    from emu.build import build
    lib = C.CDLL(str(build(name="w16")))
    lib.w16_emu_batch.restype = C.c_longlong
    lib.w16_emu_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int,
                                  C.c_void_p, C.c_void_p]
    return lib


def run_emu(lib, prm: dict, pairs, ref, qer, w, zmode=0, fill=0xA5):
    """fill = the byte shared memory holds before the first pair."""
    arr = np.array([prm["match"], prm["mismatch"], prm["o_del"], prm["e_del"], prm["o_ins"], prm["e_ins"],
                    prm["zdrop"], prm["end_bonus"], zmode], dtype=np.int32)
    skipped = np.zeros(len(pairs), dtype=np.uint8)
    ovf = C.c_longlong(0)
    cells = lib.w16_emu_batch(arr.ctypes.data, pairs.ctypes.data, ref.ctypes.data, qer.ctypes.data, len(pairs), w,
                              fill, skipped.ctypes.data, C.byref(ovf))
    assert cells >= 0
    return int(cells), skipped.astype(bool), int(ovf.value)


DEFAULT = dict(match=1, mismatch=4, o_del=6, e_del=1, o_ins=6, e_ins=1, zdrop=100, end_bonus=5)
MAX_GOLDEN = 150          # pairs per golden case (a pair costs milliseconds here: every collective is two barriers of 32 threads)


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_warp_sweep_matches_golden(emu, name):
    pairs, ref, qer, w, prm, expect, _ = load_golden(name)
    if prm["zdrop"] < 1:
        pytest.skip("vector z-drop needs zdrop >= 1")
    step = max(1, len(pairs) // MAX_GOLDEN)
    pairs, expect = pairs[::step].copy(), expect[::step]
    has_n = np.array([(qer[p["idq"]:p["idq"] + p["len2"]] > 3).any() or (ref[p["idr"]:p["idr"] + p["len1"]] > 3).any()
                      for p in pairs])
    _, skipped, ovf = run_emu(emu, prm, pairs, ref, qer, w)
    assert skipped[pairs["len2"] > MAX_QLEN].all()
    ok = ~skipped & ~has_n          # N pairs, long queries and out-of-domain pairs belong to the other kernels
    assert ok.sum() > 0 or has_n.all() or skipped.all()
    got = results_matrix(pairs)
    assert np.array_equal(got[ok], expect[ok]), f"{name}: {(got[ok] != expect[ok]).any(axis=1).sum()} pairs differ"
    assert ovf == 0


@pytest.mark.parametrize("config,w,zdrop", [("small", 100, 100), ("short8", 100, 100), ("long16", 100, 100),
                                            ("large", 100, 100), ("sweep", 32, 100), ("sweep", 100, 32767),
                                            ("sweep", 500, 100), ("large", 7, 20), ("long16", 40, 100),
                                            ("large", 0, 100), ("sweep", 3, 32767)])
def test_warp_sweep_matches_oracle(emu, oracle, config, w, zdrop):
    import genomicsbench_b200 as gb
    from oracle.pyoracle import make_params
    cfg = gb.gen_named_config(config)
    pairs, ref, qer = gb.gen_pairs(cfg, 4321, 260)
    pairs = pairs[pairs["len2"] <= MAX_QLEN][:160].copy()
    pairs["h0"][::11] = 0                            # h0 == 0 is in the domain
    want = pairs.copy()
    cells_o = oracle.batch(make_params(zdrop=zdrop), want, ref, qer, w)
    cells, skipped, ovf = run_emu(emu, dict(DEFAULT, zdrop=zdrop), pairs, ref, qer, w)
    assert len(pairs) > 20 and not skipped.any()
    assert np.array_equal(results_matrix(pairs), results_matrix(want))
    assert cells == cells_o
    assert ovf == 0


@pytest.mark.parametrize("prm", [dict(match=2, mismatch=3, o_del=4, e_del=2, o_ins=5, e_ins=1, zdrop=50, end_bonus=0),
                                 dict(match=1, mismatch=1, o_del=0, e_del=1, o_ins=0, e_ins=1, zdrop=10, end_bonus=5),
                                 dict(match=3, mismatch=7, o_del=10, e_del=3, o_ins=2, e_ins=4, zdrop=200, end_bonus=9)])
@pytest.mark.parametrize("zmode", [0, 1])
def test_warp_sweep_other_scorings(emu, oracle, prm, zmode):
    import genomicsbench_b200 as gb
    from oracle.pyoracle import make_params
    cfg = gb.gen_named_config("large")
    pairs, ref, qer = gb.gen_pairs(cfg, 778, 250)
    pairs = pairs[pairs["len2"] <= MAX_QLEN][:120].copy()
    want = pairs.copy()
    oracle.batch(make_params(**prm, zdrop_mode=zmode), want, ref, qer, 40)
    _, skipped, ovf = run_emu(emu, prm, pairs, ref, qer, 40, zmode=zmode)
    ok = ~skipped
    assert ok.sum() > 30
    assert np.array_equal(results_matrix(pairs)[ok], results_matrix(want)[ok])
    assert ovf == 0
