// bsw_long32.cuh -- ksw_extend2 (tools/bwa/ksw.c:380-479) in int32 for pairs outside the 16-bit domain: one warp per
// pair, the row held in a ring of K slots instead of a full row (bsw_extend32).
//
// Same per-pair semantics as bsw_long_kernel (SURVEY.md Appendix A, the z-drop rule of KParams::zmode) and the same row
// sweep: the window [beg, end) of a row is cut into chunks of 128 cells, lane l owns the 4 cells 4 l .. 4 l + 3 of a
// chunk, M and E are elementwise in the previous row, a 5-step max-plus __shfl_up_sync scan resolves F, one
// __shfl_up_sync hands H(i, j - 1) to the next lane, ballot probes find the next row's beg / end.  Unlike the 16-bit
// kernels nothing is packed: a cell is {h, e} as two int32 (the ring's h and e planes), M = Hd ? Hd + sc : 0, and the
// row argmax is two 32-bit reductions (the largest H, then the largest j holding it: the oracle's
// `mj = m > h ? mj : j`).
//
// Ring.  Cell j lives in slot j mod K, K >= 2 w' + 8 (w' = the clamped band; or the whole row, columns 0 .. qlen + 3,
// when that is smaller) rounded up to the chunk width: a row touches columns beg & ~3 .. end + 3, at most 2 w' + 8 of
// them, so no two columns of one row share a slot.  A cell read
// in row i has j >= beg_i >= i - w'; every cell written before row i has j <= i + w', and K >= 2 w' + 2, so two live
// cells never share a slot either.  The one hazard is a VIRGIN cell, one that no row has written yet: the reference
// still holds its first-row value there (max(h0 - oe_ins - (j - 1) e_ins, 0), h0 at j = 0, e = 0), and since end grows
// by up to 2 per row such cells are read.  `hw` is the highest column written so far; before row i's sweep the slots of
// columns hw + 1 .. end_i receive the first-row values (they held columns j - K < beg_i: dead).  Columns a row touches
// outside [beg, end] are written back unchanged.
//
// The sweep is __host__ __device__: tests/emu/l32_emu.cu runs it on the CPU with the 32 lanes as coroutines that meet at
// every collective, against the oracle and the golden vectors.
#pragma once
#include "bsw_kernels.cuh"

namespace bsw {
namespace l32 {

constexpr int CHUNK = 128;              // cells of a chunk: 32 lanes x 4
constexpr int WARPS = 4;                // warps (pairs in flight) per block

// 32 bytes; sequences one base code per byte (0-4), qoff / toff relative to the launch's query / target bases
struct Desc {
    long long qoff, toff;
    int qlen, tlen, h0, pad;
};

// 32 bytes: the six result fields of ksw_extend2 and the pair's effective cells
struct Result {
    int score, qle, tle, gtle, gscore, max_off;
    long long cells;
};

// slots of the ring for a query of qlen bases and the clamped band wc: 2 wc + 8, or the whole row (columns 0 .. qlen + 3)
// when that is smaller, rounded up to the chunk width
BSW_HD int ring_slots(int qlen, int wc)
{
    const long long need = 2ll * wc + 8 < (long long)qlen + 4 ? 2ll * wc + 8 : (long long)qlen + 4;
    return (int)((need + CHUNK - 1) / CHUNK * CHUNK);
}

// host emulation of a warp's collectives (tests/emu only; defined in tests/emu/l32_emu.cu): every lane hands in its
// value and receives all 32
struct HostExchange;
const int* hx_all(HostExchange* hx, int lane, int v);

struct Warp {
    int lane;
    HostExchange* hx;           // host emulation only

    // value of lane - d (own value where there is no such lane)
    BSW_HD int up(int v, int d) const
    {
#if defined(__CUDA_ARCH__)
        return __shfl_up_sync(0xffffffffu, v, (unsigned)d);
#else
        const int* s = hx_all(hx, lane, v);
        return lane >= d ? s[lane - d] : v;
#endif
    }
    BSW_HD int bcast(int v, int src) const
    {
#if defined(__CUDA_ARCH__)
        return __shfl_sync(0xffffffffu, v, src);
#else
        return hx_all(hx, lane, v)[src];
#endif
    }
    BSW_HD unsigned ballot(bool p) const
    {
#if defined(__CUDA_ARCH__)
        return __ballot_sync(0xffffffffu, p);
#else
        const int* s = hx_all(hx, lane, p ? 1 : 0);
        unsigned b = 0;
        for (int k = 0; k < 32; ++k) b |= (unsigned)(s[k] != 0) << k;
        return b;
#endif
    }
    BSW_HD int rmax(int v) const
    {
#if defined(__CUDA_ARCH__)
        return __reduce_max_sync(0xffffffffu, v);
#else
        const int* s = hx_all(hx, lane, v);
        int r = s[0];
        for (int k = 1; k < 32; ++k) r = r > s[k] ? r : s[k];
        return r;
#endif
    }
    // the ring's writes of every lane are visible to every lane
    BSW_HD void sync() const
    {
#if defined(__CUDA_ARCH__)
        __syncwarp();
#else
        hx_all(hx, lane, 0);
#endif
    }
};

BSW_HD int imax(int a, int b) { return a > b ? a : b; }
BSW_HD int imin(int a, int b) { return a < b ? a : b; }
BSW_HD int ffs32(unsigned b)                       // 1 + index of the lowest set bit, 0 for none
{
#if defined(__CUDA_ARCH__)
    return __ffs((int)b);
#else
    return __builtin_ffs((int)b);
#endif
}

// 4 query codes from byte j0 on (any alignment), zero bytes from qlen on
BSW_HD uint32_t load4(const uint8_t* __restrict__ q, int j0, int qlen)
{
    uint32_t qw = 0;
    if (j0 >= qlen) return 0;
#if defined(__CUDA_ARCH__)
    if (j0 + 8 <= qlen) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(q + j0);
        const uint32_t* aw = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        return __funnelshift_r(__ldg(aw), __ldg(aw + 1), (unsigned)(a & 3) * 8u);
    }
#endif
    for (int c = 0; c < 4; ++c)
        if (j0 + c < qlen) qw |= (uint32_t)q[j0 + c] << (8 * c);
    return qw;
}

// (64-bit: (j - 1) e_ins passes 2^31 on long queries)
BSW_HD int first_row(int h0, int oe_ins, int e_ins, int j)
{
    const long long v = (long long)h0 - oe_ins - (long long)(j - 1) * e_ins;
    return j == 0 ? h0 : (v > 0 ? (int)v : 0);
}

// ------------------------------------------------------------------------------------------------
// Row sweep of one pair by the 32 lanes of a warp.  hr / er: the pair's ring (K slots each, K = ring_slots(qlen, w') or
// larger, a multiple of CHUNK; 16-byte aligned).  Every lane returns the same st; cells is counted by lane 0.
// ------------------------------------------------------------------------------------------------
BSW_HD void sweep(const KParams& P, const uint8_t* __restrict__ qb, int qlen, const uint8_t* __restrict__ tb, int tlen,
                  int h0, int* __restrict__ hr, int* __restrict__ er, int K, const Warp& wp, PairState& st,
                  long long& cells)
{
    const int lane = wp.lane;
    const int e_ins4 = 4 * P.e_ins;
    const int w = bsw_clamp_band(P, qlen);
    st.max = h0; st.max_i = -1; st.max_j = -1; st.max_ie = -1; st.gscore = -1; st.max_off = 0;
    int beg = 0, end = qlen;
    int hw = -1;                                          // highest column written so far

    for (int i = 0; i < tlen; ++i) {
        const int ti = tb[i];
        beg = imax(beg, i - w);
        end = imin(imin(end, i + w + 1), qlen);
        // virgin columns hw + 1 .. end get the first row's values
        if (end > hw) {
            for (int j = hw + 1 + lane; j <= end; j += 32) {
                const int s = j % K;
                hr[s] = first_row(h0, P.oe_ins, P.e_ins, j);
                er[s] = 0;
            }
            hw = end;
            wp.sync();
        }
        const int h1_init = beg == 0 ? imax(h0 - (P.o_del + P.e_del * (i + 1)), 0) : 0;
        int f_carry = 0, h_carry = h1_init;
        int mh = 0, mj = -1;                              // this lane's row maximum and the last column holding it
        int h_end = -1;                                   // H(i, end - 1), found by its owner lane
        if (end > beg) {
            int s0 = (beg & ~3) % K;                      // slot of the chunk's first column
            for (int cbase = beg & ~3; cbase <= end; cbase += CHUNK) {
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
                    qw = load4(qb, j0, qlen);
                }
                int M[4], E[4], g[5];
                g[0] = 0;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int j = j0 + c;
                    const bool in = j >= beg && j < end;
                    const int Hd = in ? hd[c] : 0;
                    E[c] = in ? ed[c] : 0;
                    const int qk = (int)((qw >> (8 * c)) & 0xffu);
                    int sc = qk == ti ? P.match : P.mismatch_neg;
                    if ((qk | ti) > 3) sc = P.ambig;
                    M[c] = Hd ? imax(Hd + sc, 0) : 0;          // a negative M acts as 0 in every use
                    g[c + 1] = imax(imax(M[c] - P.oe_ins, 0), g[c] - P.e_ins);
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
                int H[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int F = imax(g[c], fin - c * P.e_ins);
                    H[c] = imax(imax(M[c], E[c]), F);
                }
                int hprev = wp.up(H[3], 1);
                if (lane == 0) hprev = h_carry;
                // new cells: h = H(i, j - 1), e = E(i + 1, j); column end gets {H(i, end - 1), 0}
                int nh[4], ne[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int j = j0 + c;
                    const int hp = c == 0 ? hprev : H[c - 1];
                    nh[c] = hd[c]; ne[c] = ed[c];
                    if (j >= beg && j < end) {
                        nh[c] = hp;
                        ne[c] = imax(imax(M[c] - P.oe_del, 0), E[c] - P.e_del);
                        if (H[c] >= mh) { mh = H[c]; mj = j; }
                        if (j == end - 1) h_end = H[c];
                    } else if (j == end) {
                        nh[c] = hp; ne[c] = 0;
                    }
                }
                if (j0 <= end) {
                    *reinterpret_cast<int4*>(hr + s) = make_int4(nh[0], nh[1], nh[2], nh[3]);
                    *reinterpret_cast<int4*>(er + s) = make_int4(ne[0], ne[1], ne[2], ne[3]);
                }
                f_carry = imax(wp.bcast(x, 31), f_carry - e_ins4 * 32);
                h_carry = wp.bcast(H[3], 31);
                s0 += CHUNK;
                s0 = s0 >= K ? s0 - K : s0;
            }
            if (lane == 0) cells += end - beg;
        } else if (lane == 0) {
            hr[end % K] = h1_init; er[end % K] = 0;       // bandedSWA.cpp:213 with an empty window
        }
        wp.sync();
        const int m = wp.rmax(mh);
        const int mjr = wp.rmax(mh == m ? mj : -1);
        const int h1 = end > beg ? wp.rmax(h_end) : h1_init;
        const int jfin = end > beg ? end : beg;
        if (jfin == qlen) {
            if (!(st.gscore > h1)) st.max_ie = i;
            st.gscore = imax(st.gscore, h1);
        }
        if (bsw_row_update(P, st, i, m, mjr)) break;
        // next row's window (bandedSWA.cpp:230-233), 32 cells per probe
        {
            int j = beg;
            while (j < end) {
                const int idx = j + lane;
                const bool nz = idx < end ? (hr[idx % K] | er[idx % K]) != 0 : true;
                const unsigned b = wp.ballot(nz);
                if (b) { j += ffs32(b) - 1; break; }
                j += 32;
            }
            beg = j;
            j = end;
            while (j >= beg) {
                const int idx = j - lane;
                const bool nz = idx >= beg ? (hr[idx % K] | er[idx % K]) != 0 : true;
                const unsigned b = wp.ballot(nz);
                if (b) { j -= ffs32(b) - 1; break; }
                j -= 32;
            }
            end = imin(j + 2, qlen);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Kernel: WARPS pairs in flight per block, pairs pulled from an atomic queue in the order perm[] gives (longest
// estimated work first).  SMEM: the rings live in dynamic shared memory (2 K ints per warp), else in the global scratch
// (2 K ints per resident warp; the launch is sized to the scratch).  res[s] in input order; one cell atomic per warp.
// ------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
template <bool SMEM>
__global__ void __launch_bounds__(WARPS * 32)
bsw_long32_kernel(const Desc* __restrict__ desc, const uint32_t* __restrict__ perm, const uint8_t* __restrict__ qbytes,
                  const uint8_t* __restrict__ tbytes, Result* __restrict__ res, int count, int K,
                  const __grid_constant__ KParams P, int* __restrict__ scratch, unsigned int* __restrict__ queue,
                  unsigned long long* __restrict__ cell_counter)
{
    extern __shared__ __align__(16) int l32_smem[];
    const int wib = threadIdx.x >> 5;
    int* const ring = SMEM ? l32_smem + (size_t)wib * 2 * K : scratch + ((size_t)blockIdx.x * WARPS + wib) * 2 * (size_t)K;
    Warp wp;
    wp.lane = threadIdx.x & 31;
    wp.hx = nullptr;
    long long my_cells = 0;
    for (;;) {
        unsigned k = 0;
        if (wp.lane == 0) k = atomicAdd(queue, 1u);
        k = __shfl_sync(0xffffffffu, k, 0);
        if (k >= (unsigned)count) break;
        const int s = (int)perm[k];
        const Desc d = desc[s];
        PairState st;
        long long c = 0;
        sweep(P, qbytes + d.qoff, d.qlen, tbytes + d.toff, d.tlen, d.h0, ring, ring + K, K, wp, st, c);
        if (wp.lane == 0) {
            Result r;
            r.score = st.max; r.qle = st.max_j + 1; r.tle = st.max_i + 1; r.gtle = st.max_ie + 1;
            r.gscore = st.gscore; r.max_off = st.max_off; r.cells = c;
            res[s] = r;
            my_cells += c;
        }
        __syncwarp();
    }
    if (wp.lane == 0 && my_cells) atomicAdd(cell_counter, (unsigned long long)my_cells);
}
#endif

} // namespace l32
} // namespace bsw
