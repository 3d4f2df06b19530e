"""The packed kernel's row sweep (k16::pair_sweep, bsw_kernel16.cuh) executed on the CPU with the
DPX .S16x2 instructions emulated (tests/emu/k16_emu.cu), compared bit for bit with the oracle and
the golden vectors.  Also checks that no 16-bit lane ever wraps inside the kernel's domain."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from conftest import GOLDEN_CASES, load_golden, results_matrix


@pytest.fixture(scope="module")
def emu():
    from emu.build import build
    lib = C.CDLL(str(build()))
    lib.k16_emu_batch2.restype = C.c_longlong
    lib.k16_emu_batch2.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int,
                                   C.c_int, C.c_void_p, C.c_void_p]
    return lib


def run_emu(lib, prm: dict, pairs, ref, qer, w, zmode=0, circ=0, fill=0xA5):
    """circ = 1: rows as circular buffers of the band's width wherever the band is narrower than the query
    (what the engine launches then); circ = 0: rows that hold the whole query.  fill = the byte shared memory holds
    before a pair."""
    arr = np.array([prm["match"], prm["mismatch"], prm["o_del"], prm["e_del"], prm["o_ins"], prm["e_ins"],
                    prm["zdrop"], prm["end_bonus"], zmode], dtype=np.int32)
    skipped = np.zeros(len(pairs), dtype=np.uint8)
    ovf = C.c_longlong(0)
    cells = lib.k16_emu_batch2(arr.ctypes.data, pairs.ctypes.data, ref.ctypes.data, qer.ctypes.data, len(pairs), w,
                               circ, fill, skipped.ctypes.data, C.byref(ovf))
    return int(cells), skipped.astype(bool), int(ovf.value)


DEFAULT = dict(match=1, mismatch=4, o_del=6, e_del=1, o_ins=6, e_ins=1, zdrop=100, end_bonus=5)


@pytest.mark.parametrize("circ", [0, 1])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_emulated_sweep_matches_golden(emu, name, circ):
    pairs, ref, qer, w, prm, expect, _ = load_golden(name)
    has_n = np.array([(qer[p["idq"]:p["idq"] + p["len2"]] > 3).any() or (ref[p["idr"]:p["idr"] + p["len1"]] > 3).any()
                      for p in pairs])
    if prm["zdrop"] < 1:
        pytest.skip("vector z-drop needs zdrop >= 1")
    _, skipped, ovf = run_emu(emu, prm, pairs, ref, qer, w, circ=circ)
    ok = ~skipped & ~has_n          # N pairs and out-of-domain pairs belong to the byte kernel
    assert ok.sum() > 0 or has_n.all() or skipped.all()
    got = results_matrix(pairs)
    assert np.array_equal(got[ok], expect[ok]), f"{name}: {(got[ok] != expect[ok]).any(axis=1).sum()} pairs differ"
    assert ovf == 0


@pytest.mark.parametrize("config,w,zdrop", [("small", 100, 100), ("short8", 100, 100), ("long16", 100, 100),
                                            ("large", 100, 100), ("sweep", 32, 100), ("sweep", 100, 32767),
                                            ("sweep", 500, 100), ("large", 7, 20), ("long16", 40, 100),
                                            ("large", 0, 100), ("sweep", 3, 32767)])
@pytest.mark.parametrize("circ", [0, 1])
def test_emulated_sweep_matches_oracle(emu, oracle, config, w, zdrop, circ):
    import genomicsbench_b200 as gb
    from oracle.pyoracle import make_params
    cfg = gb.gen_named_config(config)
    pairs, ref, qer = gb.gen_pairs(cfg, 12345, 3000)
    pairs["h0"][::11] = 0                            # h0 == 0 is in the domain
    want = pairs.copy()
    cells_o = oracle.batch(make_params(zdrop=zdrop), want, ref, qer, w)
    cells, skipped, ovf = run_emu(emu, dict(DEFAULT, zdrop=zdrop), pairs, ref, qer, w, circ=circ)
    assert not skipped.any()
    assert np.array_equal(results_matrix(pairs), results_matrix(want))
    assert cells == cells_o
    assert ovf == 0


@pytest.mark.parametrize("prm", [dict(match=2, mismatch=3, o_del=4, e_del=2, o_ins=5, e_ins=1, zdrop=50, end_bonus=0),
                                 dict(match=1, mismatch=1, o_del=0, e_del=1, o_ins=0, e_ins=1, zdrop=10, end_bonus=5),
                                 dict(match=3, mismatch=7, o_del=10, e_del=3, o_ins=2, e_ins=4, zdrop=200, end_bonus=9)])
@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("circ", [0, 1])
def test_emulated_sweep_other_scorings(emu, oracle, prm, zmode, circ):
    import genomicsbench_b200 as gb
    from oracle.pyoracle import make_params
    cfg = gb.gen_named_config("large")
    pairs, ref, qer = gb.gen_pairs(cfg, 777, 2000)
    want = pairs.copy()
    oracle.batch(make_params(**prm, zdrop_mode=zmode), want, ref, qer, 40)
    _, skipped, ovf = run_emu(emu, prm, pairs, ref, qer, 40, zmode=zmode, circ=circ)
    ok = ~skipped
    assert ok.sum() > 100
    assert np.array_equal(results_matrix(pairs)[ok], results_matrix(want)[ok])
    assert ovf == 0
