"""The two-slot chunk pipeline of bsw_global and bsw_extend32 across several chunks.

bsw_global's first form cuts a call into chunks of 65 536 alignments, its second form into chunks of BSW_GLOBAL_CHUNK
alignments; bsw_extend32 cuts at 2^18 pairs or 256 MB of sequence.  Every call here spans several chunks, so both slots
are reused and drained, and the results must not depend on where the cuts fall."""
from __future__ import annotations

import numpy as np
import pytest

from conftest import GOLDEN_DIR

TILES = 300                                   # global_default tiled: 210 000 alignments
FORM1_CHUNK = 65536                           # alignments per chunk of the first form
X32_CHUNK_PAIRS = 1 << 18                     # pairs per chunk of bsw_extend32 ...
X32_CHUNK_BYTES = 256 << 20                   # ... and sequence bytes
SCORING = dict(match=1, mismatch=4, o_del=6, e_del=1, o_ins=6, e_ins=1, zdrop=100, end_bonus=5, ambig=-1)
FIELDS = ("score", "qle", "tle", "gtle", "gscore", "max_off")


@pytest.fixture(scope="module")
def tiled(lib):
    """global_default tiled TILES times: (params, pairs, ref, qer, w, score, n_cigar, cigar) with the golden results."""
    z = np.load(GOLDEN_DIR / "global" / "global_default.npz")
    P = dict(zip(("o_del", "e_del", "o_ins", "e_ins", "match", "mismatch", "ambig"), (int(v) for v in z["params"])))
    pairs = np.zeros(len(z["w"]), dtype=lib.SEQPAIR_DTYPE)
    pairs["len1"], pairs["len2"] = z["len1"], z["len2"]
    pairs["idr"] = np.concatenate([[0], np.cumsum(z["len1"])[:-1]])
    pairs["idq"] = np.concatenate([[0], np.cumsum(z["len2"])[:-1]])
    pairs["h0"] = 1
    return (P, np.tile(pairs, TILES), np.ascontiguousarray(z["target"]), np.ascontiguousarray(z["query"]),
            np.tile(z["w"], TILES), np.tile(z["score"], TILES), np.tile(z["n_cigar"], TILES), np.tile(z["cigar"], TILES))


def _form(monkeypatch, kernel, chunk):
    for var, value in (("BSW_GLOBAL_KERNEL", kernel), ("BSW_GLOBAL_CHUNK", chunk)):
        if value:
            monkeypatch.setenv(var, value)
        else:
            monkeypatch.delenv(var, raising=False)


def _offsets(n_cigar):
    return np.concatenate([[0], np.cumsum(n_cigar)]).astype(np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,chunk", [("1", None), ("", "1000"), ("2w", "1000")])
def test_global_several_chunks(lib, tiled, kernel, chunk, monkeypatch):
    """kernel "1": the first form, chunks of 65 536; "" / "2w": the second form with 16- / 64-bit slots, chunks of
    1000."""
    _form(monkeypatch, kernel, chunk)
    P, pairs, ref, qer, w, score_g, ncig_g, cigar_g = tiled
    with lib.Engine(**P) as eng:
        score, cigar, off = eng.global_align(pairs, ref, qer, w)
        st = eng.stats()
    assert np.array_equal(score, score_g)
    assert np.array_equal(off, _offsets(ncig_g))
    assert np.array_equal(cigar, cigar_g)
    # the form that ran (the first packs the gathered bytes tight) and the number of chunks (>= 3 launches each)
    l1, l2 = pairs["len1"].astype(np.int64), pairs["len2"].astype(np.int64)
    assert (st["h2d_bytes"] == 40 * len(pairs) + int(l1.sum() + l2.sum())) == (kernel == "1")
    per_chunk = FORM1_CHUNK if kernel == "1" else int(chunk)
    assert st["kernel_launches"] >= 3 * -(-len(pairs) // per_chunk)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,chunk,first", [("1", None, FORM1_CHUNK), ("", "1000", 1000)])
def test_global_cigar_cap_error_then_reuse(lib, tiled, kernel, chunk, first, monkeypatch):
    """A cigar buffer that holds the first chunk's operations but not the call's is refused in a later chunk, after the
    first chunk's results are out; the same engine's next call is complete."""
    _form(monkeypatch, kernel, chunk)
    P, pairs, ref, qer, w, score_g, ncig_g, cigar_g = tiled
    n = len(pairs)
    cap = int(ncig_g[:first].sum())
    out = (np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(cap, np.uint32), np.zeros(n + 1, np.int64))
    with lib.Engine(**P) as eng:
        with pytest.raises(lib.BswError) as ei:
            eng.global_align(pairs, ref, qer, w, out=out)
        assert ei.value.code == -1 and "cigar buffer too small" in str(ei.value)
        assert np.array_equal(out[0][:first], score_g[:first]) and np.array_equal(out[2], cigar_g[:cap])
        score, cigar, off = eng.global_align(pairs, ref, qer, w)
    assert np.array_equal(score, score_g)
    assert np.array_equal(off, _offsets(ncig_g))
    assert np.array_equal(cigar, cigar_g)


def _results(pairs):
    return np.stack([pairs[f] for f in FIELDS], axis=1)


@pytest.mark.gpu
def test_extend32_cut_by_pair_count(lib):
    """More pairs than one chunk holds, all inside the 16-bit domain: bsw_extend's results, and the effective cells of
    one call per chunk."""
    pairs, ref, qer = lib.gen_pairs(lib.gen_named_config("short8"), 4243, 300000)
    head = pairs[:X32_CHUNK_PAIRS]
    assert int(head["len1"].astype(np.int64).sum() + head["len2"].sum()) <= X32_CHUNK_BYTES     # cut by count alone
    with lib.Engine(**SCORING) as eng:
        want = pairs.copy()
        eng.extend(want, ref, qer, 100)
        got = pairs.copy()
        eng.extend32(got, ref, qer, 100)
        cells = eng.stats()["cells_effective"]
        parts = 0
        for part in (pairs[:X32_CHUNK_PAIRS].copy(), pairs[X32_CHUNK_PAIRS:].copy()):
            eng.extend32(part, ref, qer, 100)
            parts += eng.stats()["cells_effective"]
    assert np.array_equal(_results(got), _results(want))
    assert cells == parts


@pytest.mark.gpu
def test_extend32_cut_by_bytes(lib, oracle):
    """Pairs of ~500 kb on each side, more sequence than one chunk holds: the same results and effective cells as the
    pairs split into calls of one chunk each, and the oracle's results on every 30th pair."""
    from oracle.pyoracle import make_params
    rng = np.random.default_rng(0xB5B2050C)
    n = 300
    lens = rng.integers(480000, 520000, n)
    qer = rng.integers(0, 4, int(lens.sum()) + 64).astype(np.uint8)
    ref = qer.copy()
    sub = rng.random(len(ref)) < 0.02
    ref[sub] = (ref[sub] + rng.integers(1, 4, int(sub.sum()))) % 4
    pairs = np.zeros(n, dtype=lib.SEQPAIR_DTYPE)
    pairs["len1"] = pairs["len2"] = lens
    pairs["idr"] = pairs["idq"] = np.concatenate([[0], np.cumsum(lens)[:-1]])
    pairs["h0"] = rng.integers(20, 100, n)                  # a seed's score (h0 = 0 leaves nothing to extend from)
    assert 2 * int(lens.sum()) > X32_CHUNK_BYTES and 2 * int(lens[:n // 2].sum()) < X32_CHUNK_BYTES
    with lib.Engine(zdrop_mode=0, **SCORING) as eng:
        got = pairs.copy()
        eng.extend32(got, ref, qer, 8)
        cells = eng.stats()["cells_effective"]
        want, parts = pairs.copy(), 0
        for a, b in ((0, n // 2), (n // 2, n)):
            part = want[a:b].copy()
            eng.extend32(part, ref, qer, 8)
            want[a:b] = part
            parts += eng.stats()["cells_effective"]
    assert np.array_equal(_results(got), _results(want))
    assert cells == parts
    assert (got["score"] > 32767).all()                     # outside bsw_extend's 16-bit domain
    some = pairs[::30].copy()
    oracle.batch(make_params(**SCORING, zdrop_mode=0), some, ref, qer, 8)
    assert np.array_equal(_results(got[::30]), _results(some))
