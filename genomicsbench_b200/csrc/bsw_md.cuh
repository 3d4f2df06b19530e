// bsw_md.cuh -- the finishing pass of bsw_reg2aln: NM and the MD string of every alignment region from its final
// operation list (bwa_gen_cigar2's NM / MD walk, tools/bwa/bwa.c:196-227), sm_100a.
//
// One warp per region.  The operations are walked in order by the whole warp; an M run is taken 32 bases at a time
// (lane l compares query[x + c + l] with the reference base under it), __ballot_sync gives the chunk's mismatch mask,
// and the run of matches u in front of each mismatch falls out of the mask: the previous mismatch is the highest set
// bit below the lane (__clz), or, for the first one of the chunk, the run carried in from earlier chunks and across I
// operations (which do not reset it, bwa.c:222).  A D operation that is neither the first nor the last emits
// "u^bases" (the reference bases through int2base); the first and the last D are skipped, y moves on (bwa.c:214-220).
// After the last operation the final u is emitted.
//
// Two sweeps over the same walk: md_count gives n_mm, n_gap, the MD length and the sum of the M columns' scores (the
// fast path's score, bwa.c:184-185: a region whose CIGAR is one M run); md_write places every number, letter and ^ run
// at its exclusive-scan position inside the warp.  Between them the host pipeline scans the lengths on the device
// (bsw_cigar_offsets).  Both sweeps are __host__ __device__: tests/emu/md_emu.cu runs them on the CPU with the 32 lanes
// as coroutines (l32::Warp's host exchange).
//
// Sequences arrive as bwa_gen_cigar2 aligns them: for a reverse-strand region (rb >= l_pac) both the query segment
// and the reference bases are reversed, and int2base is "TGCAN" instead of "ACGTN" (bwa.c:199).
#pragma once
#include "bsw_long32.cuh"
#include "bsw_global.cuh"

namespace bsw {
namespace md {

using l32::Warp;

constexpr int WARPS = 4;                // warps (regions in flight) per block

struct MdDesc {                         // one region of a chunk
    long long qoff, roff;               // byte offsets into the chunk's (possibly reversed) query / reference bytes
    long long coff;                     // word offset of its final operation list (before the end-D squeeze and clips)
    int32_t n_cig;
    int32_t rev;                        // 1: reverse strand (int2base "TGCAN")
};

struct MdCount { int n_mm, n_gap, md_len, msc; };

struct MdScore { int match, mismatch_neg, ambig; };

BSW_HD int md_digits(int u)
{
    int d = 1;
    while (u >= 10) { u /= 10; ++d; }
    return d;
}

BSW_HD int md_hibit(unsigned m)                   // index of the highest set bit (m != 0)
{
#if defined(__CUDA_ARCH__)
    return 31 - __clz(m);
#else
    return 31 - __builtin_clz(m);
#endif
}

BSW_HD int md_popc(unsigned m)
{
#if defined(__CUDA_ARCH__)
    return __popc(m);
#else
    return __builtin_popcount(m);
#endif
}

BSW_HD void md_put_dec(char* p, int u, int nd)
{
    for (int k = nd - 1; k >= 0; --k) { p[k] = (char)('0' + u % 10); u /= 10; }
}

BSW_HD char md_base(int rev, uint8_t b)
{
    const char* s = rev ? "TGCAN" : "ACGTN";
    return s[b < 4 ? b : 4];
}

// inclusive prefix sum over the warp
BSW_HD int md_scan(const Warp& wp, int v)
{
    for (int d = 1; d < 32; d <<= 1) {
        const int o = wp.up(v, d);
        if (wp.lane >= d) v += o;
    }
    return v;
}

// Walks the operations of one region.  WRITE = false: returns the counts (every lane the same values);
// WRITE = true: writes the MD bytes to out[0 .. md_len).
template <bool WRITE>
BSW_HD MdCount md_sweep(const uint8_t* __restrict__ q, const uint8_t* __restrict__ r, const uint32_t* __restrict__ cig,
                        int n_cig, int rev, const MdScore& S, char* __restrict__ out, const Warp& wp)
{
    const int lane = wp.lane;
    MdCount c{0, 0, 0, 0};
    int u = 0;                           // matches since the last emitted mismatch / deletion (warp-uniform)
    long long x = 0, y = 0;
    for (int k = 0; k < n_cig; ++k) {
        const int op = (int)(cig[k] & 0xf), len = (int)(cig[k] >> 4);
        if (op == 0) {
            for (int b = 0; b < len; b += 32) {
                const int p = b + lane;
                const bool in = p < len;
                const uint8_t qv = in ? q[x + p] : 0, rv = in ? r[y + p] : 0;
                const bool mm = in && qv != rv;
                const unsigned mask = wp.ballot(mm);
                const int nin = len - b < 32 ? len - b : 32;
                int run = 0, emit = 0;
                if (mm) {
                    const unsigned lower = mask & ((1u << lane) - 1u);
                    run = lower ? lane - md_hibit(lower) - 1 : u + lane;
                    emit = md_digits(run) + 1;
                }
                const int incl = md_scan(wp, emit);
                if (WRITE && mm) {
                    char* o = out + c.md_len + (incl - emit);
                    md_put_dec(o, run, emit - 1);
                    o[emit - 1] = md_base(rev, rv);
                }
                if (!WRITE) {
                    const int sc = !in ? 0 : (qv >= 4 || rv >= 4) ? S.ambig : qv == rv ? S.match : S.mismatch_neg;
                    c.msc += wp.bcast(md_scan(wp, sc), 31);
                }
                c.md_len += wp.bcast(incl, 31);
                if (mask) { u = nin - 1 - md_hibit(mask); c.n_mm += md_popc(mask); }
                else u += nin;
            }
            x += len; y += len;
        } else if (op == 2) {
            if (k > 0 && k < n_cig - 1) {
                const int nd = md_digits(u);
                if (WRITE) {
                    char* o = out + c.md_len;
                    if (lane == 0) { md_put_dec(o, u, nd); o[nd] = '^'; }
                    for (int b = lane; b < len; b += 32) o[nd + 1 + b] = md_base(rev, r[y + b]);
                }
                c.md_len += nd + 1 + len;
                c.n_gap += len;
                u = 0;
            }
            y += len;
        } else if (op == 1) {
            x += len;
            c.n_gap += len;
        }
    }
    const int nd = md_digits(u);
    if (WRITE && lane == 0) md_put_dec(out + c.md_len, u, nd);
    c.md_len += nd;
    return c;
}

// count pass: md_len[i], nm[i], msc[i] of every region of the chunk (one warp per region, grid-stride)
__global__ void __launch_bounds__(WARPS * 32)
bsw_md_count_kernel(const MdDesc* __restrict__ desc, int n, const uint8_t* __restrict__ q, const uint8_t* __restrict__ r,
                    const uint32_t* __restrict__ cig, const MdScore S, int32_t* __restrict__ md_len,
                    int32_t* __restrict__ nm, int32_t* __restrict__ msc)
{
    Warp wp;
    wp.lane = threadIdx.x & 31; wp.hx = nullptr;
    for (int i = blockIdx.x * WARPS + (threadIdx.x >> 5); i < n; i += gridDim.x * WARPS) {
        const MdDesc d = desc[i];
        const MdCount c = md_sweep<false>(q + d.qoff, r + d.roff, cig + d.coff, d.n_cig, d.rev, S, nullptr, wp);
        if (wp.lane == 0) { md_len[i] = c.md_len; nm[i] = c.n_mm + c.n_gap; msc[i] = c.msc; }
    }
}

// write pass: the MD bytes of region i at md[md_off[i] ..)
__global__ void __launch_bounds__(WARPS * 32)
bsw_md_write_kernel(const MdDesc* __restrict__ desc, int n, const uint8_t* __restrict__ q, const uint8_t* __restrict__ r,
                    const uint32_t* __restrict__ cig, const MdScore S, const long long* __restrict__ md_off,
                    char* __restrict__ md)
{
    Warp wp;
    wp.lane = threadIdx.x & 31; wp.hx = nullptr;
    for (int i = blockIdx.x * WARPS + (threadIdx.x >> 5); i < n; i += gridDim.x * WARPS) {
        const MdDesc d = desc[i];
        md_sweep<true>(q + d.qoff, r + d.roff, cig + d.coff, d.n_cig, d.rev, S, md + md_off[i], wp);
    }
}

} // namespace md
} // namespace bsw
