"""genomicsbench_b200 -- B200-native banded Smith-Waterman extension (GenomicsBench `bsw`).

Host-side mirror of the reference operator interface (benchmarks/bsw/bandedSWA.h:114-342):
`BandedPairWiseSW` with the reference's constructor arguments and `getScores16` /
`getScores8` / `scalarBandedSWAWrapper` methods, over numpy views of the reference's
`SeqPair` records.  Everything is a thin ctypes call into libbsw_b200.so (CUDA, sm_100a).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

# One hardware queue per stream of the engine's pipeline (bsw_create sets the same default, but the
# variable only counts before the process's first CUDA call -- e.g. torch's, in bench.py).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import numpy as np

from ._lib import (ABI, ALN_DTYPE, ALNREG_DTYPE, ALNREG_FIELDS, BSW_PACKED_MAX_QLEN, REG_IN_DTYPE, BSW_PAIR_RAW, BSW_ZDROP_SCALAR, BSW_ZDROP_VECTOR,
                   CHAIN_DTYPE, OUTSCORE_DTYPE, PAIR_DESC_DTYPE, RESULT_FIELDS, SCORE16_DTYPE, SEED_DTYPE, SEQPAIR_DTYPE,
                   BswChainOpt, BswGenConfig, BswPackedBatch, BswParams, BswStats, LIB_PATH, load_host_library,
                   load_library, ptr)

__all__ = [
    "BandedPairWiseSW", "Engine", "BswError", "SEQPAIR_DTYPE", "RESULT_FIELDS", "default_params",
    "gen_named_config", "gen_pairs", "bucket_order", "split_by_cost", "read_pairs_file",
    "write_pairs_file", "load_library", "NAMED_CONFIGS", "pinned_empty", "pinned_copy",
    "SEED_DTYPE", "CHAIN_DTYPE", "ALNREG_DTYPE", "ALNREG_FIELDS", "PackedBatch", "PAIR_DESC_DTYPE", "OUTSCORE_DTYPE",
    "SCORE16_DTYPE", "BSW_PAIR_RAW", "BSW_PACKED_MAX_QLEN", "load_host_library", "REG_IN_DTYPE", "ALN_DTYPE",
    "reg_inputs", "cigar_string", "reg2aln_capacity",
]

NAMED_CONFIGS = {"small": 0, "short8": 1, "long16": 2, "large": 3, "sweep": 4}


class BswError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"bsw error {code}: {msg}")
        self.code = code


def default_params(**over) -> BswParams:
    p = BswParams()
    load_library().bsw_default_params(C.byref(p))
    for k, v in over.items():
        if k == "devices":
            p.n_devices = len(v)
            for i, d in enumerate(v):
                p.devices[i] = int(d)
        else:
            setattr(p, k, v)
    return p


def _check_arrays(pairs: np.ndarray, seq_ref: np.ndarray, seq_qer: np.ndarray):
    if pairs.dtype != SEQPAIR_DTYPE or not pairs.flags.c_contiguous:
        raise TypeError("pairs must be a C-contiguous array of SEQPAIR_DTYPE")
    for a in (seq_ref, seq_qer):
        if a.dtype != np.uint8 or not a.flags.c_contiguous:
            raise TypeError("sequence buffers must be C-contiguous uint8 arrays")


class Engine:
    """Owns one bsw_engine (C ABI).  One instance may drive several GPUs of the box."""

    def __init__(self, params: Optional[BswParams] = None, **over):
        self._lib = load_library()
        self._h = None
        p = params if params is not None else default_params(**over)
        err = C.c_int(0)
        h = self._lib.bsw_create(C.byref(p), C.byref(err))
        if not h:
            raise BswError(err.value, self._lib.bsw_last_error(None).decode())
        self._h = h
        self.params = p

    def close(self):
        if self._h:
            self._lib.bsw_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _rc(self, rc: int):
        if rc != 0:
            raise BswError(rc, self._lib.bsw_last_error(self._h).decode())

    def extend(self, pairs: np.ndarray, seq_ref: np.ndarray, seq_qer: np.ndarray, w: int) -> None:
        _check_arrays(pairs, seq_ref, seq_qer)
        self._rc(self._lib.bsw_extend(self._h, ptr(pairs), ptr(seq_ref), ptr(seq_qer), len(pairs), w))

    def extend32(self, pairs: np.ndarray, seq_ref: np.ndarray, seq_qer: np.ndarray, w: int) -> None:
        """bsw_extend32: ksw_extend2 in int32 for pairs outside extend()'s 16-bit domain (long-read flanks: lengths up
        to 2^24 - 1, h0 + len2 * max score + end_bonus up to 2^30).  Results in place, like extend()."""
        _check_arrays(pairs, seq_ref, seq_qer)
        self._rc(self._lib.bsw_extend32(self._h, ptr(pairs), ptr(seq_ref), ptr(seq_qer), len(pairs), w))

    def extend_async(self, pairs: np.ndarray, seq_ref: np.ndarray, seq_qer: np.ndarray, w: int) -> int:
        """bsw_extend_async: queues the call, returns its ticket (the arrays must stay alive until wait())."""
        _check_arrays(pairs, seq_ref, seq_qer)
        t = C.c_int64(0)
        self._rc(self._lib.bsw_extend_async(self._h, ptr(pairs), ptr(seq_ref), ptr(seq_qer), len(pairs), w, C.byref(t)))
        return int(t.value)

    def wait(self, ticket: int) -> int:
        """bsw_wait: blocks until the ticket's results are in its records; returns the call's share of effective cells."""
        cells = C.c_int64(0)
        self._rc(self._lib.bsw_wait(self._h, ticket, C.byref(cells)))
        return int(cells.value)

    def async_stats(self) -> tuple:
        a, b = C.c_int64(0), C.c_int64(0)
        self._rc(self._lib.bsw_async_stats(self._h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def extend_retry(self, pairs: np.ndarray, seq_ref: np.ndarray, seq_qer: np.ndarray, w: int,
                     max_try: int = 2, prev_score: Optional[np.ndarray] = None) -> np.ndarray:
        """Band-doubling retry of the aligner (tools/bwa/bwamem.c:630,723-753,770-800; MAX_BAND_TRY = 2).
        Returns the band each pair's last try ran with."""
        _check_arrays(pairs, seq_ref, seq_qer)
        band = np.zeros(len(pairs), dtype=np.int32)
        prev = None
        if prev_score is not None:
            prev = np.ascontiguousarray(prev_score, dtype=np.int32)
            if len(prev) != len(pairs):
                raise ValueError("prev_score must have one entry per pair")
        self._rc(self._lib.bsw_extend_retry(self._h, ptr(pairs), ptr(seq_ref), ptr(seq_qer), len(pairs), w,
                                            max_try, ptr(prev) if prev is not None else None, ptr(band)))
        return band

    def global_align(self, pairs: np.ndarray, seq_ref: np.ndarray, seq_qer: np.ndarray, w, out=None) -> tuple:
        """ksw_global2 for a batch (tools/bwa/ksw.c:502-606): banded global alignment + CIGAR.  w = one band
        or one per pair.  Returns (score int32[n], cigar uint32[total], cigar_off int64[n + 1]); the operations
        of pair i are cigar[cigar_off[i]:cigar_off[i + 1]] (len << 4 | op, op 0 M / 1 I / 2 D).
        out = (score int32[>= n], n_cigar int32[>= n], cigar uint32[cap], cigar_off int64[>= n + 1]): caller-owned
        result arrays, reused across calls like a C caller's; the returned arrays are then views of them."""
        return self._global(self._lib.bsw_global, pairs, seq_ref, seq_qer, w, out)

    def global_align32(self, pairs: np.ndarray, seq_ref: np.ndarray, seq_qer: np.ndarray, w, out=None) -> tuple:
        """bsw_global32: global_align() for alignment regions of up to 2^24 - 1 bases (long-read regions), one warp
        per alignment.  Same arguments, results and errors; inside global_align()'s domain the same results."""
        return self._global(self._lib.bsw_global32, pairs, seq_ref, seq_qer, w, out)

    def _global(self, fn, pairs, seq_ref, seq_qer, w, out) -> tuple:
        _check_arrays(pairs, seq_ref, seq_qer)
        n = len(pairs)
        wv = np.ascontiguousarray(np.broadcast_to(np.asarray(w, dtype=np.int32), (n,)))
        if out is not None:
            score, ncig, cigar, off = out
            for a, dt, need in ((score, np.int32, n), (ncig, np.int32, n), (cigar, np.uint32, 1), (off, np.int64, n + 1)):
                if a.dtype != dt or not a.flags.c_contiguous or len(a) < need:
                    raise ValueError("out = (score int32[n], n_cigar int32[n], cigar uint32[cap], cigar_off int64[n + 1]), contiguous")
            self._rc(fn(self._h, ptr(pairs), ptr(seq_ref), ptr(seq_qer), n, ptr(wv), ptr(score), ptr(ncig), ptr(cigar),
                        len(cigar), ptr(off)))
            return score[:n], cigar[:int(off[n])], off[:n + 1]
        score = np.zeros(max(n, 1), dtype=np.int32); ncig = np.zeros(max(n, 1), dtype=np.int32)
        cap = int((pairs["len1"].astype(np.int64) + pairs["len2"]).sum()) if n else 0
        cigar = np.zeros(max(cap, 1), dtype=np.uint32); off = np.zeros(n + 1, dtype=np.int64)
        self._rc(fn(self._h, ptr(pairs), ptr(seq_ref), ptr(seq_qer), n, ptr(wv), ptr(score), ptr(ncig), ptr(cigar), cap,
                    ptr(off)))
        return score[:n], cigar[:int(off[n])].copy(), off

    def chain_window(self, w: int, l_pac: int, seeds: np.ndarray, l_query: int) -> tuple:
        """Reference window [rmax0, rmax1) of a chain of seeds (tools/bwa/bwamem.c:643-659)."""
        seeds = np.ascontiguousarray(seeds, dtype=SEED_DTYPE)
        r0, r1 = C.c_int64(0), C.c_int64(0)
        self._rc(self._lib.bsw_chain_window(C.byref(self.params), w, l_pac, ptr(seeds), len(seeds), l_query,
                                            C.byref(r0), C.byref(r1)))
        return int(r0.value), int(r1.value)

    def extend_chains(self, chains: np.ndarray, seeds: np.ndarray, query: np.ndarray, ref: np.ndarray, w: int,
                      pen_clip5: int = 5, pen_clip3: int = 5, max_band_try: int = 2, out=None):
        """mem_chain2aln for a batch of chains (tools/bwa/bwamem.c:632-822): seed -> left / right pair
        construction, band-doubling retry, local-vs-to-end decision.  chains = CHAIN_DTYPE, seeds = SEED_DTYPE;
        returns (regs ALNREG_DTYPE[len(seeds)], count int32[len(chains)]): the regions of chain c are
        regs[chains[c].seed_first : + count[c]] in the order the reference pushes them."""
        chains = np.ascontiguousarray(chains, dtype=CHAIN_DTYPE)
        seeds = np.ascontiguousarray(seeds, dtype=SEED_DTYPE)
        if query.dtype != np.uint8 or ref.dtype != np.uint8 or not query.flags.c_contiguous or not ref.flags.c_contiguous:
            raise ValueError("query / ref must be contiguous uint8 arrays (one base code per byte)")
        if out is not None:                                  # caller-owned result arrays (reused across calls, like a C caller's)
            regs, count = out
            if regs.dtype != ALNREG_DTYPE or count.dtype != np.int32 or len(regs) < len(seeds) or len(count) < len(chains):
                raise ValueError("out = (regs ALNREG_DTYPE[>= len(seeds)], count int32[>= len(chains)])")
        else:
            regs = np.zeros(max(len(seeds), 1), dtype=ALNREG_DTYPE)
            count = np.zeros(max(len(chains), 1), dtype=np.int32)
        opt = BswChainOpt(w, pen_clip5, pen_clip3, max_band_try)
        self._rc(self._lib.bsw_extend_chains(self._h, ptr(chains), len(chains), ptr(seeds), ptr(query), ptr(ref),
                                             C.byref(opt), ptr(regs), ptr(count)))
        return regs[:len(seeds)], count[:len(chains)]

    def reg2aln(self, regs_in: np.ndarray, query: np.ndarray, ref: np.ndarray, l_pac: int, w: int, out=None) -> tuple:
        """mem_reg2aln's alignment part for a batch of regions (bsw_reg2aln; bwamem.c mem_reg2aln, bwa.c bwa_gen_cigar2):
        band inference, the band-doubling loop, CIGAR with soft clips (ops "MIDSH": 3 = soft clip), NM and MD.
        regs_in = REG_IN_DTYPE (reg_inputs builds it from extend_chains' output).  Returns (aln ALN_DTYPE[n],
        cigar uint32[total], cigar_off int64[n + 1], md uint8[total], md_off int64[n + 1]); region i's operations are
        cigar[cigar_off[i]:cigar_off[i + 1]], its MD md[md_off[i]:md_off[i + 1]] (ASCII, no NUL).
        out = (aln ALN_DTYPE[>= n], cigar uint32[cap], cigar_off int64[>= n + 1], md uint8[cap], md_off int64[>= n + 1]):
        caller-owned result arrays, reused across calls; the returned arrays are then views of them."""
        regs_in = np.ascontiguousarray(regs_in, dtype=REG_IN_DTYPE)
        if query.dtype != np.uint8 or ref.dtype != np.uint8 or not query.flags.c_contiguous or not ref.flags.c_contiguous:
            raise ValueError("query / ref must be contiguous uint8 arrays (one base code per byte)")
        n = len(regs_in)
        if out is not None:
            aln, cigar, coff, md, moff = out
            for a, dt, need in ((aln, ALN_DTYPE, n), (cigar, np.uint32, 1), (coff, np.int64, n + 1), (md, np.uint8, 1),
                                (moff, np.int64, n + 1)):
                if a.dtype != dt or not a.flags.c_contiguous or len(a) < need:
                    raise ValueError("out = (aln ALN_DTYPE[n], cigar uint32[cap], cigar_off int64[n + 1], md uint8[cap], "
                                     "md_off int64[n + 1]), contiguous")
        else:
            ccap, mcap = reg2aln_capacity(regs_in)
            aln = np.zeros(max(n, 1), dtype=ALN_DTYPE)
            cigar, md = np.zeros(max(ccap, 1), dtype=np.uint32), np.zeros(max(mcap, 1), dtype=np.uint8)
            coff, moff = np.zeros(n + 1, dtype=np.int64), np.zeros(n + 1, dtype=np.int64)
        self._rc(self._lib.bsw_reg2aln(self._h, ptr(regs_in), n, ptr(query), ptr(ref), l_pac, w, ptr(aln), ptr(cigar),
                                       len(cigar), ptr(coff), ptr(md), len(md), ptr(moff)))
        return aln[:n], cigar[:int(coff[n])], coff[:n + 1], md[:int(moff[n])], moff[:n + 1]

    def extend_packed(self, batch: "PackedBatch", w: int, out: Optional[np.ndarray] = None, compact: bool = False) -> np.ndarray:
        """bsw_extend_packed / bsw_extend_packed16: a packed batch in, OUTSCORE_DTYPE (24 B) or SCORE16_DTYPE (16 B)
        records out, input order.  `out` = a caller-owned result array (page-locked for the DMA route)."""
        dt = SCORE16_DTYPE if compact else OUTSCORE_DTYPE
        if out is None:
            out = np.zeros(max(batch.n_pairs, 1), dtype=dt)
        if out.dtype != dt or not out.flags.c_contiguous or len(out) < batch.n_pairs:
            raise TypeError(f"out must be a C-contiguous {dt} array with one entry per pair")
        fn = self._lib.bsw_extend_packed16 if compact else self._lib.bsw_extend_packed
        self._rc(fn(self._h, C.byref(batch.c), w, ptr(out)))
        return out[:batch.n_pairs]

    def stage(self, pairs, seq_ref, seq_qer, w: int) -> None:
        _check_arrays(pairs, seq_ref, seq_qer)
        self._rc(self._lib.bsw_stage(self._h, ptr(pairs), ptr(seq_ref), ptr(seq_qer), len(pairs), w))

    def run_staged(self) -> None:
        self._rc(self._lib.bsw_run_staged(self._h))

    def fetch(self, pairs: np.ndarray) -> None:
        self._rc(self._lib.bsw_fetch(self._h, ptr(pairs), len(pairs)))

    def stats(self) -> dict:
        s = BswStats()
        self._rc(self._lib.bsw_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    def measure_int_peak(self) -> float:
        return float(self._lib.bsw_measure_int_peak(self._h))


class BandedPairWiseSW:
    """Mirror of the reference class (bandedSWA.h:114-342, ctor bandedSWA.cpp:51-100).

    Same argument order and meaning as the C++ constructor; `mat` is accepted for
    signature parity (the vector path ignores it, exactly like the reference,
    bandedSWA.cpp:69)."""

    def __init__(self, o_del: int, e_del: int, o_ins: int, e_ins: int, zdrop: int, end_bonus: int,
                 mat: Optional[Sequence[int]], w_match: int, w_mismatch: int, numThreads: int = 1,
                 devices: Optional[Sequence[int]] = None):
        # tiny_batch: like the C++ class (csrc/bsw_shim.cpp) -- the reference driver's habit is -b 512 pairs per call
        self._kw = dict(o_del=o_del, e_del=e_del, o_ins=o_ins, e_ins=e_ins, zdrop=zdrop,
                        end_bonus=end_bonus, match=w_match, mismatch=w_mismatch, tiny_batch=1536)
        if devices is not None:
            self._kw["devices"] = list(devices)
        self._mat = None if mat is None else [int(x) for x in mat]
        self._vec: Optional[Engine] = None
        self._scalar: Optional[Engine] = None
        self.SW_cells = 0
        self.last_stats: dict = {}

    def _engine(self, scalar: bool) -> Engine:
        if scalar:
            if self._scalar is None:
                kw = dict(self._kw, zdrop_mode=BSW_ZDROP_SCALAR)
                if self._mat is not None:
                    kw["ambig"] = self._mat[4]
                self._scalar = Engine(**kw)
            return self._scalar
        if self._vec is None:
            self._vec = Engine(**dict(self._kw, zdrop_mode=BSW_ZDROP_VECTOR))
        return self._vec

    def _run(self, scalar, pairs, seq_ref, seq_qer, numPairs, w):
        eng = self._engine(scalar)
        eng.extend(pairs[:numPairs], seq_ref, seq_qer, w)
        self.last_stats = eng.stats()
        self.SW_cells += self.last_stats["cells_effective"]

    def getScores16(self, pairArray, seqBufRef, seqBufQer, numPairs, numThreads, w):
        self._run(False, pairArray, seqBufRef, seqBufQer, numPairs, w)

    def getScores8(self, pairArray, seqBufRef, seqBufQer, numPairs, numThreads, w):
        self._run(False, pairArray, seqBufRef, seqBufQer, numPairs, w)

    def scalarBandedSWAWrapper(self, seqPairArray, seqBufRef, seqBufQer, numPairs, nthreads, w):
        self._run(True, seqPairArray, seqBufRef, seqBufQer, numPairs, w)

    def close(self):
        for e in (self._vec, self._scalar):
            if e is not None:
                e.close()
        self._vec = self._scalar = None


# ---------------------------------------------------------------------------------------
# alignment records (bsw_reg2aln)
# ---------------------------------------------------------------------------------------
def reg_inputs(chains: np.ndarray, regs: np.ndarray, count: np.ndarray) -> np.ndarray:
    """bsw_reg_in records for every region extend_chains() returned: the chain's read, and its reference bases
    ref[chain.ref_off + rb - rmax0 ..] inside the chain's window (the same ref buffer extend_chains() read)."""
    chains = np.asarray(chains, dtype=CHAIN_DTYPE)
    idx = np.concatenate([np.arange(int(c["seed_first"]), int(c["seed_first"]) + int(k)) for c, k in zip(chains, count)]
                         + [np.zeros(0, np.int64)]).astype(np.int64)
    ch = np.repeat(np.arange(len(chains)), np.asarray(count, dtype=np.int64))
    out = np.zeros(len(idx), dtype=REG_IN_DTYPE)
    out["reg"] = regs[idx]
    out["query_off"] = chains["query_off"][ch]
    out["l_query"] = chains["l_query"][ch]
    out["ref_off"] = chains["ref_off"][ch] + out["reg"]["rb"] - chains["rmax0"][ch]
    return out


def reg2aln_capacity(regs_in: np.ndarray) -> tuple:
    """(cigar entries, MD bytes) that always suffice for these regions (include/bsw.h: (qe - qb) + (re - rb) + 2
    operations and 4 (qe - qb) + (re - rb) + 1 MD bytes per mapped region)."""
    r = regs_in["reg"]
    mapped = (r["rb"] >= 0) & (r["re"] >= 0)
    ql = np.where(mapped, r["qe"].astype(np.int64) - r["qb"], 0)
    rl = np.where(mapped, r["re"] - r["rb"], 0)
    return int((ql + rl + 2 * mapped).sum()), int((4 * ql + rl + mapped).sum())


def cigar_string(ops) -> str:
    """len << 4 | op operations -> CIGAR text with bwa's op letters "MIDSH" (3 = S)."""
    return "".join(f"{int(c) >> 4}{'MIDSH'[int(c) & 0xf]}" for c in ops)


# ---------------------------------------------------------------------------------------
# pinned host buffers (bsw_host_alloc): numpy views the engine can DMA directly
# ---------------------------------------------------------------------------------------
class _PinnedBlock:
    """Owns one bsw_host_alloc allocation; freed when the last numpy view of it dies."""

    def __init__(self, nbytes: int):
        self._lib = load_library()
        self.ptr = self._lib.bsw_host_alloc(max(int(nbytes), 1))
        if not self.ptr:
            raise BswError(-4, f"bsw_host_alloc({nbytes}) failed (no CUDA device or out of pinned memory)")
        self.nbytes = int(nbytes)

    def __del__(self):
        if getattr(self, "ptr", None):
            self._lib.bsw_host_free(self.ptr)
            self.ptr = None


def pinned_empty(shape, dtype) -> np.ndarray:
    """numpy array over page-locked memory: buffers like this take the engine's direct route.
    The block is freed when the array (and every view of it) is garbage-collected."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape))
    blk = _PinnedBlock(n * dtype.itemsize + 64)
    raw = (C.c_ubyte * max(n * dtype.itemsize, 1)).from_address(blk.ptr)
    raw._owner = blk                                  # arr.base -> raw -> blk
    return np.frombuffer(raw, dtype=dtype, count=n).reshape(shape)


def pinned_copy(a: np.ndarray) -> np.ndarray:
    out = pinned_empty(a.shape, a.dtype)
    out[...] = a
    return out


# ---------------------------------------------------------------------------------------
# the packed host format (include/bsw.h: bsw_packed_batch)
# ---------------------------------------------------------------------------------------
class PackedBatch:
    """Owns one bsw_packed_batch built by the library (2 bits per base + 16-byte descriptors; RAW pairs keep one byte
    per base).  pinned=True allocates the buffers with bsw_host_alloc (needs a CUDA device), else with malloc;
    host_only=True builds through libbsw_host.so (no CUDA library mapped)."""

    def __init__(self, pinned: bool = False, host_only: bool = False):
        if pinned and host_only:
            raise ValueError("page-locked buffers come from the CUDA library")
        self._lib = load_host_library() if host_only else load_library()
        self.c = BswPackedBatch()
        if pinned:
            cuda = load_library()
            self._alloc = C.cast(cuda.bsw_host_alloc, C.c_void_p)
            self._release = C.cast(cuda.bsw_host_free, C.c_void_p)
        else:
            self._alloc = self._release = None
        self._built = False

    def _done(self, rc: int, what: str):
        if rc:
            raise BswError(rc, what)
        self._built = True
        return self

    @classmethod
    def from_pairs(cls, pairs, seq_ref, seq_qer, raw_min_qlen: int = 0, pinned: bool = False, host_only: bool = False):
        _check_arrays(pairs, seq_ref, seq_qer)
        b = cls(pinned, host_only)
        return b._done(b._lib.bsw_batch_from_pairs(ptr(pairs), ptr(seq_ref), ptr(seq_qer), len(pairs), raw_min_qlen,
                                                   b._alloc, b._release, C.byref(b.c)), "bsw_batch_from_pairs")

    @classmethod
    def from_file(cls, path: str, max_pairs: int = -1, raw_min_qlen: int = 0, pinned: bool = False, host_only: bool = False):
        b = cls(pinned, host_only)
        return b._done(b._lib.bsw_batch_from_file(path.encode(), max_pairs, raw_min_qlen, b._alloc, b._release,
                                                  C.byref(b.c)), f"bsw_batch_from_file({path})")

    @classmethod
    def gen(cls, cfg: BswGenConfig, first: int = 0, n: Optional[int] = None, raw_min_qlen: int = 0, pinned: bool = False,
            host_only: bool = False):
        b = cls(pinned, host_only)
        n = int(cfg.n_pairs if n is None else n)
        return b._done(b._lib.bsw_batch_gen(C.byref(cfg), first, n, raw_min_qlen, b._alloc, b._release, C.byref(b.c)),
                       "bsw_batch_gen")

    @property
    def n_pairs(self) -> int:
        return int(self.c.n_pairs)

    def _view(self, p, count, dtype):
        if not p or count <= 0:
            return np.zeros(0, dtype=dtype)
        dtype = np.dtype(dtype)
        raw = (C.c_ubyte * (count * dtype.itemsize)).from_address(p)
        raw._owner = self
        return np.frombuffer(raw, dtype=dtype, count=count)

    @property
    def desc(self) -> np.ndarray:
        return self._view(self.c.desc, self.n_pairs, PAIR_DESC_DTYPE)

    @property
    def q2(self) -> np.ndarray:
        return self._view(self.c.q2, int(self.c.q2_words), np.uint32)

    @property
    def r2(self) -> np.ndarray:
        return self._view(self.c.r2, int(self.c.r2_words), np.uint32)

    @property
    def raw_q(self) -> np.ndarray:
        return self._view(self.c.raw_q, int(self.c.raw_q_bytes), np.uint8)

    @property
    def raw_r(self) -> np.ndarray:
        return self._view(self.c.raw_r, int(self.c.raw_r_bytes), np.uint8)

    def nbytes(self) -> int:
        """bytes a call moves host -> device for this batch"""
        return 16 * self.n_pairs + 4 * int(self.c.q2_words + self.c.r2_words) + int(self.c.raw_q_bytes + self.c.raw_r_bytes)

    def to_pairs(self):
        """-> (pairs, seq_ref, seq_qer) in the reference's layout (bsw_batch_to_pairs)."""
        d = self.desc
        pairs = np.zeros(max(self.n_pairs, 1), dtype=SEQPAIR_DTYPE)
        rcap, qcap = int(d["len1"].astype(np.int64).sum()) + 64, int(d["len2"].astype(np.int64).sum()) + 64
        ref, qer = np.zeros(rcap, dtype=np.uint8), np.zeros(qcap, dtype=np.uint8)
        rc = self._lib.bsw_batch_to_pairs(C.byref(self.c), ptr(pairs), ptr(ref), rcap, ptr(qer), qcap)
        if rc:
            raise BswError(rc, "bsw_batch_to_pairs")
        return pairs[:self.n_pairs], ref, qer

    def close(self):
        if getattr(self, "_built", False):
            self._lib.bsw_batch_release(C.byref(self.c), self._release)
            self._built = False

    __del__ = close


# ---------------------------------------------------------------------------------------
# host utilities (no GPU needed)
# ---------------------------------------------------------------------------------------
def gen_named_config(which, host_only: bool = False) -> BswGenConfig:
    idx = NAMED_CONFIGS[which] if isinstance(which, str) else int(which)
    cfg = BswGenConfig()
    rc = (load_host_library() if host_only else load_library()).bsw_gen_named_config(idx, C.byref(cfg))
    if rc:
        raise BswError(rc, "unknown named config")
    return cfg


def gen_pairs(cfg: BswGenConfig, first: int = 0, n: Optional[int] = None, host_only: bool = False):
    """Returns (pairs, seq_ref, seq_qer) for pairs [first, first+n) of the config's stream."""
    lib = load_host_library() if host_only else load_library()
    n = int(cfg.n_pairs if n is None else n)
    sub = BswGenConfig.from_buffer_copy(cfg)
    sub.n_pairs = n
    rb, qb = C.c_int64(0), C.c_int64(0)
    rc = lib.bsw_gen_bounds(C.byref(sub), C.byref(rb), C.byref(qb))
    if rc:
        raise BswError(rc, "bad generator config")
    pairs = np.zeros(n, dtype=SEQPAIR_DTYPE)
    ref = np.empty(rb.value, dtype=np.uint8)
    qer = np.empty(qb.value, dtype=np.uint8)
    ru, qu = C.c_int64(0), C.c_int64(0)
    rc = lib.bsw_gen_pairs(C.byref(cfg), first, n, ptr(pairs), ptr(ref), ptr(qer), C.byref(ru), C.byref(qu))
    if rc:
        raise BswError(rc, "generator failed")
    ref[ru.value: ru.value + 64] = 0          # slack after the last sequence, never addressed by a pair
    qer[qu.value: qu.value + 64] = 0
    return pairs, ref[: ru.value + 64], qer[: qu.value + 64]


def bucket_order(pairs: np.ndarray) -> np.ndarray:
    order = np.empty(len(pairs), dtype=np.int64)
    rc = load_library().bsw_bucket_order(ptr(pairs), len(pairs), ptr(order))
    if rc:
        raise BswError(rc, "bucket_order")
    return order


def split_by_cost(pairs: np.ndarray, w: int, n_shards: int) -> np.ndarray:
    """Contiguous cut of the input order into n_shards ranges of equal estimated DP cost (bsw_split_by_cost)."""
    if pairs.dtype != SEQPAIR_DTYPE or not pairs.flags.c_contiguous:
        raise TypeError("pairs must be a C-contiguous array of SEQPAIR_DTYPE")
    begin = np.zeros(n_shards + 1, dtype=np.int64)
    rc = load_library().bsw_split_by_cost(ptr(pairs), len(pairs), w, n_shards, ptr(begin))
    if rc:
        raise BswError(rc, "split_by_cost")
    return begin


def read_pairs_file(path: str, max_pairs: Optional[int] = None):
    lib = load_library()
    n = lib.bsw_count_pairs_file(path.encode())
    if n < 0:
        raise BswError(int(n), f"cannot read {path}")
    if max_pairs is not None:
        n = min(n, max_pairs)
    import os
    cap = os.path.getsize(path) + 64
    pairs = np.zeros(n, dtype=SEQPAIR_DTYPE)
    ref = np.zeros(cap, dtype=np.uint8)
    qer = np.zeros(cap, dtype=np.uint8)
    got = C.c_int64(0)
    rc = lib.bsw_read_pairs_file(path.encode(), n, ptr(pairs), ptr(ref), cap, ptr(qer), cap, C.byref(got))
    if rc:
        raise BswError(rc, f"parse error in {path}")
    return pairs[: got.value], ref, qer


def write_pairs_file(path: str, pairs: np.ndarray, seq_ref: np.ndarray, seq_qer: np.ndarray) -> None:
    rc = load_library().bsw_write_pairs_file(path.encode(), ptr(pairs), len(pairs), ptr(seq_ref), ptr(seq_qer))
    if rc:
        raise BswError(rc, f"cannot write {path}")
