// bsw_global32.cuh -- ksw_global2 (tools/bwa/ksw.c:502-606; push_cigar :489-500) for alignment regions of any length
// up to 2^24 - 1 (bsw_global32): one warp per alignment, the row in a ring, 4-bit directions in HBM, and a backtrack
// that walks tiles of the direction matrix staged in shared memory.
//
// Row sweep (sweep).  The band is fixed, [beg, end) = [max(0, i - w), min(qlen, i + w + 1)), and is cut into chunks of
// 128 cells starting at beg & ~3; lane l owns the 4 cells 4 l .. 4 l + 3 of a chunk (bsw_long32.cuh's layout).  Every
// cell follows ksw_global2's int32 arithmetic and its order of comparisons:
//   M = H(i-1, j-1) + s (no clamp at 0);  H = max(M, E, F) with ties to M, then E, then F;
//   E(i+1, j) = max(E - e_del, M - oe_del);  F(j+1) = max(F(j) - e_ins, M(j) - oe_ins).
// F is fed by M, not by H, so it is a pure max-plus scan over M: the 5-step __shfl_up_sync scan of l32::sweep with a
// carry across chunks.  F(beg) is the sentinel; a lane's cells left of beg feed nothing into the scan, so the F of any
// cell right of beg is a maximum over real terms, which is ksw_global2's value (a real value is far above the sentinel,
// see the value bound in include/bsw.h), and F(beg) stays at or below the sentinel, where it loses every comparison it
// takes part in as the sentinel does.
//
// Ring.  Cell j lives in slot j mod K, K = l32::ring_slots(qlen, w) (2 w + 8, or the whole row, columns 0 .. qlen + 3,
// rounded up to 128).  A row touches columns beg & ~3 .. end + 3, at most 2 w + 8 of them, so no two share a slot; row i
// reads columns [i - w, i + w] and every column written before it is <= i + w.  Unlike ksw_extend2 the band never
// shrinks: row i reads columns up to i + w, and row i - 1 wrote exactly those, column i + w as its end
// (eh[end] = {h1, -inf}, ksw.c:588).  So only the first row's columns 0 .. w are initialised; every other cell is
// written before it is read (tests/emu/g32_emu.cu fills the ring with garbage before every alignment).
//
// Directions.  4 bits per cell: bits 0-1 H's source (0 M, 1 E, 2 F), bit 2 E extended, bit 3 F extended.  ksw_global2's
// byte f << 4 | e << 2 | h is (bit3 << 5) | (bit2 << 2) | (bits 0-1).  Row i of an alignment's matrix holds the cells
// j - (beg & ~3), one 64-byte block per chunk (a 16-bit store per lane), pitch = dir_pitch bytes.
//
// Backtrack (backtrack).  ksw.c:591-603 from (tlen - 1, min(tlen + w, qlen) - 1).  Each step moves up at most one row,
// and its band column moves by at most a few cells, so the warp loads a tile of TILE_ROWS rows x TILE_BYTES bytes
// (one coalesced 128-byte row per load round) into shared memory and lane 0 walks it; the walk stops where it leaves
// the tile and the warp loads the next one around the current cell.  The run being built stays in registers; the list
// is written in walk order and reversed by the warp at the end.
//
// sweep and backtrack are __host__ __device__: tests/emu/g32_emu.cu runs them on the CPU with the 32 lanes as
// coroutines (l32::Warp's host exchange).
#pragma once
#include "bsw_long32.cuh"
#include "bsw_global.cuh"

namespace bsw {
namespace g32 {

using l32::CHUNK;
using l32::Warp;
using l32::imax;
using l32::imin;

constexpr int WARPS = 4;                // warps (alignments in flight) per block, both kernels
constexpr int TILE_ROWS = 32;           // backtrack tile: rows ...
constexpr int TILE_BYTES = 128;         // ... x bytes (256 band cells) of each row

// bytes of one row of the direction matrix: 64 per chunk of the widest window (n_col = min(qlen, 2 w + 1) cells from
// beg & ~3 on: up to n_col + 3 columns)
BSW_HD long long dir_pitch(int qlen, int w)
{
    const long long ncol = 2ll * w + 1 < qlen ? 2ll * w + 1 : (long long)qlen;
    return (ncol + 3 + CHUNK - 1) / CHUNK * 64;
}

// ------------------------------------------------------------------------------------------------
// Row sweep of one alignment by the 32 lanes of a warp.  w: the band, at most max(qlen, tlen) (a wider band is the
// same band).  hr / er: the ring (K slots each, K >= l32::ring_slots(qlen, w), a multiple of CHUNK; 16-byte aligned).
// dz: the alignment's direction matrix (64-byte aligned), pitch = dir_pitch(qlen, w).  Returns the score
// (H(tlen - 1, qlen - 1), ksw.c:590) on every lane.
// ------------------------------------------------------------------------------------------------
BSW_HD int sweep(const GlobalParams& P, const uint8_t* __restrict__ qb, int qlen, const uint8_t* __restrict__ tb, int tlen,
                 int w, int* __restrict__ hr, int* __restrict__ er, int K, uint8_t* __restrict__ dz, long long pitch,
                 const Warp& wp)
{
    const int lane = wp.lane;
    const int oe_del = P.o_del + P.e_del, oe_ins = P.o_ins + P.e_ins;
    const int e_ins4 = 4 * P.e_ins;
    for (int j = lane; j <= imin(w, qlen); j += 32) {                         // first row, ksw.c:521-525
        hr[j % K] = j == 0 ? 0 : -(P.o_ins + P.e_ins * j);
        er[j % K] = G_MINUS_INF;
    }
    wp.sync();
    for (int i = 0; i < tlen; ++i) {                                          // ksw.c:527-589
        const int ti = tb[i];
        const int beg = imax(i - w, 0), end = imin(i + w + 1, qlen);
        const int h1_init = beg == 0 ? -(P.o_del + P.e_del * (i + 1)) : G_MINUS_INF;
        int f_carry = G_MINUS_INF, h_carry = h1_init;
        uint8_t* const zrow = dz + (size_t)i * (size_t)pitch;
        int s0 = (beg & ~3) % K;                                              // slot of the chunk's first column
        for (int cbase = beg & ~3, zb = 0; cbase <= end; cbase += CHUNK, zb += 64) {
            const int j0 = cbase + 4 * lane;
            int s = s0 + 4 * lane;
            s = s >= K ? s - K : s;
            int hd[4] = {0, 0, 0, 0}, ed[4] = {0, 0, 0, 0};
            uint32_t qw = 0;
            if (j0 <= end) {
                const int4 h4 = *reinterpret_cast<const int4*>(hr + s);
                const int4 e4 = *reinterpret_cast<const int4*>(er + s);
                hd[0] = h4.x; hd[1] = h4.y; hd[2] = h4.z; hd[3] = h4.w;
                ed[0] = e4.x; ed[1] = e4.y; ed[2] = e4.z; ed[3] = e4.w;
                qw = l32::load4(qb, j0, qlen);
            }
            int M[4], E[4], g[5];
            g[0] = G_MINUS_INF;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int j = j0 + c;
                const bool in = j >= beg && j < end;
                const int qk = (int)((qw >> (8 * c)) & 0xffu);
                const int sc = (qk | ti) > 3 ? P.ambig : (qk == ti ? P.match : P.mismatch_neg);
                M[c] = in ? hd[c] + sc : 0;
                E[c] = in ? ed[c] : G_MINUS_INF;
                g[c + 1] = imax(in ? M[c] - oe_ins : G_MINUS_INF, g[c] - P.e_ins);
            }
            // inclusive max-plus scan of the lanes' outgoing F (decay 4 e_ins per lane)
            int x = g[4];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = wp.up(x, d);
                if (lane >= d) x = imax(x, y - e_ins4 * d);
            }
            int fin = wp.up(x, 1);
            fin = lane == 0 ? f_carry : imax(fin, f_carry - e_ins4 * lane);
            int H[4], NE[4];
            uint32_t dirs = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {                                     // ksw.c:544-566
                const int F = imax(g[c], fin - c * P.e_ins);
                int d = M[c] >= E[c] ? 0 : 1;
                int h = M[c] >= E[c] ? M[c] : E[c];
                d = h >= F ? d : 2;
                h = h >= F ? h : F;
                H[c] = h;
                int t = M[c] - oe_del;
                const int e = E[c] - P.e_del;
                d |= e > t ? 4 : 0;
                NE[c] = e > t ? e : t;
                t = M[c] - oe_ins;
                d |= F - P.e_ins > t ? 8 : 0;
                const int j = j0 + c;
                if (j >= beg && j < end) dirs |= (uint32_t)d << (4 * c);
            }
            int hprev = wp.up(H[3], 1);
            if (lane == 0) hprev = h_carry;
            // new cells: h = H(i, j - 1) (h1_init at beg), e = E(i + 1, j); column end gets {H(i, end - 1), -inf}
            int nh[4], ne[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int j = j0 + c;
                const int hp = j == beg ? h1_init : (c == 0 ? hprev : H[c - 1]);
                nh[c] = hd[c]; ne[c] = ed[c];
                if (j >= beg && j < end) { nh[c] = hp; ne[c] = NE[c]; }
                else if (j == end) { nh[c] = hp; ne[c] = G_MINUS_INF; }
            }
            if (j0 <= end) {
                *reinterpret_cast<int4*>(hr + s) = make_int4(nh[0], nh[1], nh[2], nh[3]);
                *reinterpret_cast<int4*>(er + s) = make_int4(ne[0], ne[1], ne[2], ne[3]);
            }
            if (cbase < end) *reinterpret_cast<uint16_t*>(zrow + zb + 2 * lane) = (uint16_t)dirs;
            f_carry = imax(wp.bcast(x, 31), f_carry - e_ins4 * 32);
            h_carry = wp.bcast(H[3], 31);
            s0 += CHUNK;
            s0 = s0 >= K ? s0 - K : s0;
        }
        wp.sync();
    }
    return hr[qlen % K];                                                      // eh[qlen].h, ksw.c:590 (the last row's end is qlen)
}

// ------------------------------------------------------------------------------------------------
// Backtrack of one alignment by the 32 lanes of a warp (ksw.c:591-603): dz / pitch as in sweep, tile = the warp's
// TILE_ROWS x TILE_BYTES bytes (4-byte aligned).  Writes the merged operations (len << 4 | op) in read order to cg and
// returns their number on every lane.
// ------------------------------------------------------------------------------------------------
BSW_HD int backtrack(const uint8_t* __restrict__ dz, long long pitch, int qlen, int tlen, int w, uint32_t* __restrict__ cg,
                     uint8_t* __restrict__ tile, const Warp& wp)
{
    const int lane = wp.lane;
    int i = tlen - 1, k = imin(i + w + 1, qlen) - 1, which = 0;
    int n_op = 0, op = -1, len = 0;                                           // lane 0: the list so far and the open run
    auto push = [&](int o, int l) {                                           // push_cigar, ksw.c:489-500
        if (o == op) { len += l; return; }
        if (len) cg[n_op++] = (uint32_t)len << 4 | (uint32_t)op;
        op = o; len = l;
    };
    while (i >= 0 && k >= 0) {
        // the tile: rows top - TILE_ROWS + 1 .. top, bytes s .. s + TILE_BYTES of each (clipped to the row's pitch)
        const int top = i;
        const int s = imax(((k - (imax(i - w, 0) & ~3)) >> 1) - TILE_BYTES / 2, 0) & ~3;
        for (int r = 0; r < TILE_ROWS && top - r >= 0; ++r)
            if (s + 4 * lane < pitch)
                reinterpret_cast<uint32_t*>(tile)[r * (TILE_BYTES / 4) + lane] =
                    *reinterpret_cast<const uint32_t*>(dz + (size_t)(top - r) * (size_t)pitch + s + 4 * lane);
        wp.sync();
        if (lane == 0) {
            while (i >= 0 && k >= 0) {
                const int r = top - i;
                const int x = k - (imax(i - w, 0) & ~3);
                const int b = (x >> 1) - s;
                if (r >= TILE_ROWS || b < 0 || b >= TILE_BYTES) break;
                const int nib = tile[r * TILE_BYTES + b] >> (4 * (x & 1)) & 15;
                which = which == 0 ? nib & 3 : which == 1 ? nib >> 2 & 1 : nib >> 2 & 2;
                if (which == 0) { push(0, 1); --i; --k; }
                else if (which == 1) { push(2, 1); --i; }
                else { push(1, 1); --k; }
            }
        }
        i = wp.bcast(i, 0); k = wp.bcast(k, 0); which = wp.bcast(which, 0);
        wp.sync();
    }
    if (lane == 0) {
        if (i >= 0) push(2, i + 1);
        if (k >= 0) push(1, k + 1);
        push(-1, 0);                                                          // closes the last run
    }
    n_op = wp.bcast(n_op, 0);
    wp.sync();
    for (int a = lane; a < n_op >> 1; a += 32) {                              // into read order
        const uint32_t t = cg[a];
        cg[a] = cg[n_op - 1 - a];
        cg[n_op - 1 - a] = t;
    }
    wp.sync();
    return n_op;
}

// ------------------------------------------------------------------------------------------------
// Kernels: WARPS alignments in flight per block, alignments pulled from an atomic queue in the order perm[] gives
// (longest estimated work first).  desc[] in the chunk's input order (desc[s].idx == s).
// DP: the rings live in dynamic shared memory (2 K ints per warp) when SMEM, else in the global scratch (2 K ints per
// resident warp; the launch is sized to it); score[s] = the alignment's score.
// Backtrack: the tiles live in static shared memory; n_cigar[s] = its operations, at cigar + desc[s].coff.
// ------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
template <bool SMEM>
__global__ void __launch_bounds__(WARPS * 32)
bsw_global32_dp_kernel(const GlobalDesc* __restrict__ desc, const uint32_t* __restrict__ perm, const uint8_t* __restrict__ qbytes,
                       const uint8_t* __restrict__ tbytes, uint8_t* __restrict__ z, int32_t* __restrict__ score, int count,
                       int K, const __grid_constant__ GlobalParams P, int* __restrict__ scratch, unsigned int* __restrict__ queue)
{
    extern __shared__ __align__(16) int g32_smem[];
    const int wib = threadIdx.x >> 5;
    int* const ring = SMEM ? g32_smem + (size_t)wib * 2 * K : scratch + ((size_t)blockIdx.x * WARPS + wib) * 2 * (size_t)K;
    Warp wp;
    wp.lane = threadIdx.x & 31;
    wp.hx = nullptr;
    for (;;) {
        unsigned k = 0;
        if (wp.lane == 0) k = atomicAdd(queue, 1u);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= (unsigned)count) break;
        const int s = (int)perm[k];
        const GlobalDesc d = desc[s];
        const int sc = sweep(P, qbytes + d.qoff, d.qlen, tbytes + d.roff, d.tlen, d.w, ring, ring + K, K, z + d.zoff,
                             dir_pitch(d.qlen, d.w), wp);
        if (wp.lane == 0) score[s] = sc;
        __syncwarp();
    }
}

__global__ void __launch_bounds__(WARPS * 32)
bsw_global32_bt_kernel(const GlobalDesc* __restrict__ desc, const uint32_t* __restrict__ perm, const uint8_t* __restrict__ z,
                       uint32_t* __restrict__ cigar, int32_t* __restrict__ n_cigar, int count, unsigned int* __restrict__ queue)
{
    __shared__ __align__(16) uint8_t tiles[WARPS][TILE_ROWS * TILE_BYTES];
    const int wib = threadIdx.x >> 5;
    Warp wp;
    wp.lane = threadIdx.x & 31;
    wp.hx = nullptr;
    for (;;) {
        unsigned k = 0;
        if (wp.lane == 0) k = atomicAdd(queue, 1u);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= (unsigned)count) break;
        const int s = (int)perm[k];
        const GlobalDesc d = desc[s];
        const int n = backtrack(z + d.zoff, dir_pitch(d.qlen, d.w), d.qlen, d.tlen, d.w, cigar + d.coff, tiles[wib], wp);
        if (wp.lane == 0) n_cigar[s] = n;
        __syncwarp();
    }
}
#endif

} // namespace g32
} // namespace bsw
