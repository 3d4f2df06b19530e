// bsw_warp16.cuh -- the warp-per-pair kernel with the row in REGISTERS: for calls too small to fill the GPU.
//
// Same per-pair semantics and the same packed arithmetic as the thread-per-pair kernel (bsw_kernel16.cuh;
// SURVEY.md Appendix A == benchmarks/bsw/bandedSWA.cpp:128-249 with the z-drop rule of :323-336).  One thread
// sweeps a 151-bp pair in ~0.4 ms whatever the batch, so a call that leaves most schedulers without a warp (the
// reference driver's 512-pair calls, scripts/run-cpu.sh:30) is bound by that latency.  Here the 32 lanes of a
// warp sweep ONE pair's rows together; lane l owns columns 8 l .. 8 l + 7 for the whole pair (queries up to
// 255 bases) and keeps them in eight registers -- four h words, four e words in the thread-per-pair kernel's layout
// (hs[j] = eh[j].h = H(i-1, j-1), es[j] = eh[j].e) -- so a row costs no shared-memory round trip and no barrier:
//   masks   a row's window [beg, end] becomes two 128-bit masks per lane, read from a 9 x 9 table in shared memory:
//           in    columns < beg and columns >= end enter as h = e = 0 (left of beg they are dead for good:
//                 bandedSWA.cpp:175,230; right of end their results are discarded)
//           store columns <= end are written, columns > end keep their old content (the reference leaves them
//                 untouched and later rows may read them: SURVEY.md Appendix B, stale eh[])
//           Lanes left of the window compute and store zeros, lanes right of it store nothing.
//   scores  a lane's query bases never change, so its four score words for each of the four target bases are
//           written to shared memory once; a row reads them back with one LDS.128 at [target base][lane]
//   local   the block's recurrence with F entering as 0 (K16-style word macro): M, E', A are elementwise in the
//           previous row, the block's own F chain runs in the high halves
//   scan    F(j+1) = max(F(j) - e_ins, A(j)) is a max-plus prefix: the blocks' outgoing F values are scanned over
//           the warp (5 shuffle steps, decay 8 e_ins per lane), shifted one lane to the right
//   fix     H = max(H_local, F_in - k e_ins) for column k of the block: one VIADDMNMX.S16x2 per column pair
//   shift   H(i, last column of the block) goes to the right neighbour (eh[j].h receives H(i, j-1)); lane 0
//           receives H(i, -1) = h1 (bandedSWA.cpp:176-179)
//   key     every lane: (max of its columns < end) << 16 | the LAST of its columns holding it; one REDUX.MAX gives
//           the row maximum and the last column holding it (bandedSWA.cpp:202-203)
//   window  the next row's [beg, end] (bandedSWA.cpp:230-233) from the non-zero maps of what the lanes stored:
//           REDUX.MIN / REDUX.MAX
// Rows stay sequential (SURVEY.md finding 0.6).
//
// The sweep is __host__ __device__: tests/emu runs it on the CPU with the 32 lanes as coroutines that meet at every
// collective (tests/emu/w16_emu.cu), against the oracle and the golden vectors.
#pragma once
#include "bsw_kernel16.cuh"

namespace bsw {
namespace w16 {

using namespace k16;

constexpr int MAX_QLEN = 255;                  // column qlen must exist: 32 lanes x 8 columns
constexpr int MASK_BYTES = 81 * 16;            // mask table: [lo][hi], lo, hi in 0 .. 8
constexpr int SCORE_BYTES = 4 * 32 * 16;       // per warp: [target base][lane] four score words

// host emulation of a warp's collectives (tests/emu only; defined in tests/emu/w16_emu.cu): every lane hands in its
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
    BSW_HD int rmin(int v) const
    {
#if defined(__CUDA_ARCH__)
        return __reduce_min_sync(0xffffffffu, v);
#else
        const int* s = hx_all(hx, lane, v);
        int r = s[0];
        for (int k = 1; k < 32; ++k) r = r < s[k] ? r : s[k];
        return r;
#endif
    }
};

// word k (columns 2k, 2k+1 of a block) of the mask [lo][hi]: halfwords of the columns < lo or >= hi are set
BSW_HD uint32_t mask_word(int lo, int hi, int k)
{
    const int c0 = 2 * k, c1 = 2 * k + 1;
    return ((c0 < lo || c0 >= hi) ? 0x0000ffffu : 0u) | ((c1 < lo || c1 >= hi) ? 0xffff0000u : 0u);
}

BSW_HD int clamp08(int v) { v = v > 0 ? v : 0; return v < 8 ? v : 8; }

// true when a scoring scheme may run on this kernel: the decay of an F entering a block at its last column, -7 e_ins
// (dec3 in warp_sweep), must fit one signed halfword.  The engine's routes and the CPU emulation both ask this.
BSW_HD bool scoring_ok(const KParams& P) { return 7 * P.e_ins <= 32767; }

// a loop constant that stays in its register: ptxas otherwise re-derives it from the constant bank inside every row
// (an LDC + two or three dependent instructions each; SASS of the first build)
BSW_HD uint32_t pin(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    asm volatile("mov.b32 %0, %0;" : "+r"(x));
#endif
    return x;
}

// ------------------------------------------------------------------------------------------------
// Row sweep of one pair by the 32 lanes of a warp.
//   md       {-, -, qlen | tlen << 16, h0}, qlen <= MAX_QLEN
//   qw, tw   2-bit packed query / target, 16 bases per word
//   mk_sa    the mask table (MASK_BYTES, mask_word())
//   sc_sa    the warp's score words (SCORE_BYTES), written here
// Every lane returns the same st; my_cells is counted by lane 0.
// ------------------------------------------------------------------------------------------------
template <bool SAMEGAP>
BSW_HD void warp_sweep(const KParams& P, const int4 md, const uint32_t* __restrict__ qw,
                       const uint32_t* __restrict__ tw, const uint32_t mk_sa_in, const uint32_t sc_sa_in,
                       const Warp& wp, PairState& st, long long& my_cells)
{
    const int qlen = md.z & 0xffff, tlen = (md.z >> 16) & 0xffff, h0 = md.w & 0xffff;
    const int l = (int)pin((uint32_t)wp.lane);
    const int jb = (int)pin((uint32_t)(8 * l));
    const uint32_t mk_sa = pin(mk_sa_in);
    const uint32_t sc_sa = pin(sc_sa_in + 16u * (uint32_t)l);
    const int zdrop_r = (int)pin((uint32_t)P.zdrop), zmode_r = (int)pin((uint32_t)P.zmode);
    const int e_del_r = (int)pin((uint32_t)P.e_del), h1_base = (int)pin((uint32_t)(h0 - P.o_del));
    const int e_ins8 = (int)pin((uint32_t)(8 * P.e_ins));

    // ---- first row (closed form of bandedSWA.cpp:155-157), the lane's score words
    uint32_t H0, H1, H2, H3, E0 = 0, E1 = 0, E2 = 0, E3 = 0;
    {
        uint32_t v[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int j = jb + c;
            const int hv = j == 0 ? h0 : h0 - P.oe_ins - (j - 1) * P.e_ins;
            v[c] = j <= qlen && hv > 0 ? (uint32_t)hv : 0u;
        }
        H0 = v[0] | (v[1] << 16); H1 = v[2] | (v[3] << 16); H2 = v[4] | (v[5] << 16); H3 = v[6] | (v[7] << 16);
        const uint32_t q8 = jb < qlen ? (ldg32(qw + (l >> 1)) >> (16 * (l & 1))) & 0xffffu : 0u;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const uint32_t x = q8 ^ ((uint32_t)t * 0x5555u);
            sts128(sc_sa + 512u * (uint32_t)t, table_word(P, (int)(x & 15u)), table_word(P, (int)((x >> 4) & 15u)),
                   table_word(P, (int)((x >> 8) & 15u)), table_word(P, (int)((x >> 12) & 15u)));
        }
    }
    const int w = bsw_clamp_band(P, qlen);     // (a lane reads back only the score words it wrote itself)

    st.max = h0; st.max_i = -1; st.max_j = -1; st.max_ie = -1; st.gscore = -1; st.max_off = 0;
    int beg = 0, end = qlen;
    uint32_t tword = 0;
    const uint32_t noe_del2 = pin(pack2(-P.oe_del, -P.oe_del));
    const uint32_t noe_ins2 = SAMEGAP ? 0u : pin(pack2(-P.oe_ins, -P.oe_ins));
    const uint32_t ne_del2 = pin(pack2(-P.e_del, -P.e_del));
    const uint32_t negg_hi = pin(pack2(-P.e_ins, 0));
    const uint32_t capmul = pin((uint32_t)(1 + P.match));
    const uint32_t k65536 = pin(65536u * (uint32_t)P.kone);
    const uint32_t k10001 = pin(0x10001u * (uint32_t)P.kone);
    // decay of the F entering a block at its column pairs: {-(2k+1) e_ins, -2k e_ins}
    const uint32_t dec0 = pin(pack2(-1 * P.e_ins, 0)), dec1 = pin(pack2(-3 * P.e_ins, -2 * P.e_ins));
    const uint32_t dec2 = pin(pack2(-5 * P.e_ins, -4 * P.e_ins)), dec3 = pin(pack2(-7 * P.e_ins, -6 * P.e_ins));
    (void)noe_ins2;

    // one pair word with the block's own F chain (fc: F entering the next column, high half)
#define W16_WORD(HW, EW, SW, HN, EN)                                                              \
    {                                                                                             \
        const uint32_t cap_ = mad_u((HW), capmul, 0u);                                            \
        const uint32_t M_ = addmin_relu((HW), (SW), cap_);                                        \
        const uint32_t U_ = addmax_relu(M_, noe_del2, 0u);                                      \
        EN = addmax((EW), ne_del2, U_);                                                           \
        const uint32_t A_ = SAMEGAP ? U_ : addmax_relu(M_, noe_ins2, 0u);                       \
        const uint32_t ME_ = max2(M_, (EW));                                                      \
        const uint32_t f1_ = addmax(fc, negg_hi, mad_u(A_, k65536, 0u));                          \
        const uint32_t Fc_ = prmt(fc, f1_, 0x7632);                                               \
        fc = addmax(f1_, negg_hi, A_);                                                            \
        HN = max2(ME_, Fc_);                                                                      \
    }
    // 8-bit map of the halfwords of (Z0 .. Z3) that are non-zero
#define W16_ZMAP(Z0, Z1, Z2, Z3, ZMAP)                                                            \
    {                                                                                             \
        const uint32_t f0_ = minu2((Z0), 0x00010001u), f1_ = minu2((Z1), 0x00010001u);            \
        const uint32_t f2_ = minu2((Z2), 0x00010001u), f3_ = minu2((Z3), 0x00010001u);            \
        const uint32_t zb_ = mad_u(f3_, 64u, mad_u(f2_, 16u, mad_u(f1_, 4u, f0_)));               \
        ZMAP = (zb_ | (zb_ >> 15)) & 0xffu;                                                       \
    }

    for (int i = 0; i < tlen; ++i) {
        if ((i & 15) == 0) tword = ldg32(tw + (i >> 4));
        const uint32_t ti = (tword >> ((i & 15) * 2)) & 3u;
        beg = beg > i - w ? beg : i - w;                      // (the column the band cuts is masked from here on)
        end = end < i + w + 1 ? end : i + w + 1;
        end = end < qlen ? end : qlen;
        int h1 = 0;
        if (beg == 0) { h1 = h1_base - e_del_r * (i + 1); h1 = h1 > 0 ? h1 : 0; }
        int key = 0;                      // (max of this lane's columns < end) << 16 | the last of them holding it
        int fnz = 0x7fffffff, lnz = -1;   // first non-zero stored column of [beg, end), last one of [beg, end]
        int hend = -1;                    // H(i, end - 1), known to the lane that owns column end
        if (end > beg) {
            const int hi = clamp08(end - jb);
            const uint4 rk = lds128(mk_sa + 16u * (uint32_t)(clamp08(beg - jb) * 9 + hi));
            const uint4 sk = lds128(mk_sa + 16u * (uint32_t)clamp08(end + 1 - jb));
            const uint4 sc = lds128(sc_sa + 512u * ti);
            uint32_t fc = 0;
            uint32_t hn0, hn1, hn2, hn3, en0, en1, en2, en3;
            W16_WORD(H0 & ~rk.x, E0 & ~rk.x, sc.x, hn0, en0)
            W16_WORD(H1 & ~rk.y, E1 & ~rk.y, sc.y, hn1, en1)
            W16_WORD(H2 & ~rk.z, E2 & ~rk.z, sc.z, hn2, en2)
            W16_WORD(H3 & ~rk.w, E3 & ~rk.w, sc.w, hn3, en3)
            // the F entering this lane's block: inclusive max-plus scan of the blocks' outgoing F, one lane to the right
            int x = (int)(fc >> 16);
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = wp.up(x, d) - e_ins8 * d;
                x = x > y ? x : y;
            }
            int fin = wp.up(x, 1);
            fin = l == 0 ? 0 : fin;
            const uint32_t finrep = mad_u((uint32_t)fin, k10001, 0u);
            hn0 = addmax(finrep, dec0, hn0); hn1 = addmax(finrep, dec1, hn1);
            hn2 = addmax(finrep, dec2, hn2); hn3 = addmax(finrep, dec3, hn3);
            const uint32_t hrot = (uint32_t)wp.up((int)hn3, 1);
            const uint32_t carry = l == 0 ? (uint32_t)h1 << 16 : hrot;
            const uint32_t hw0 = prmt(carry, hn0, 0x5432), hw1 = prmt(hn0, hn1, 0x5432);
            const uint32_t hw2 = prmt(hn1, hn2, 0x5432), hw3 = prmt(hn2, hn3, 0x5432);
            H0 = bitsel(H0, hw0, sk.x); H1 = bitsel(H1, hw1, sk.y); H2 = bitsel(H2, hw2, sk.z); H3 = bitsel(H3, hw3, sk.w);
            E0 = bitsel(E0, en0, sk.x); E1 = bitsel(E1, en1, sk.y); E2 = bitsel(E2, en2, sk.z); E3 = bitsel(E3, en3, sk.w);
            // key: the lane's maximum over its columns < end and the last column holding it
            {
                const uint32_t m0 = hn0 & ~rk.x, m1 = hn1 & ~rk.y, m2 = hn2 & ~rk.z, m3 = hn3 & ~rk.w;
                const uint32_t g = max2(max3(m0, m1, m2), m3);
                const uint32_t glo = g & 0xffffu, ghi = g >> 16;
                const uint32_t mx = glo > ghi ? glo : ghi;
                const uint32_t dm = mad_u((1u - mx) & 0xffffu, k10001, 0u);          // {1 - mx, 1 - mx}
                const uint32_t one2 = 0x00010001u;
                const uint32_t f0 = addmin_relu(m0, dm, one2), f1 = addmin_relu(m1, dm, one2);
                const uint32_t f2 = addmin_relu(m2, dm, one2), f3 = addmin_relu(m3, dm, one2);
                const uint32_t cb = mad_u(f3, 64u, mad_u(f2, 16u, mad_u(f1, 4u, f0)));
                const uint32_t cm = (cb | (cb >> 15)) & 0xffu;                        // != 0: some column holds the maximum
                key = (int)((mx << 16) | (uint32_t)(jb + hibit(cm)));
            }
            // what was stored: non-zero map for the next row's window, H(i, end - 1)
            {
                uint32_t zm;
                W16_ZMAP((hw0 | en0) & ~sk.x, (hw1 | en1) & ~sk.y, (hw2 | en2) & ~sk.z, (hw3 | en3) & ~sk.w, zm)
                const int p = end - jb;                         // column end inside this lane's block: 0 .. 7
                if (zm) lnz = jb + hibit(zm);
                if (end == qlen && (unsigned)p < 8u) {          // H(i, end - 1) is only asked for in rows that reach the query's end
                    const uint32_t ws = (p & 4) ? ((p & 2) ? hw3 : hw2) : ((p & 2) ? hw1 : hw0);
                    hend = (int)((p & 1) ? ws >> 16 : ws & 0xffffu);
                }
                zm &= ~shl_sat(1u, p);                            // column end counts for the last, not for the first
                if (zm) fnz = jb + lobit(zm);
            }
            if (l == 0) my_cells += end - beg;
        } else {
            // empty window: eh[end] = {h1, 0}  (bandedSWA.cpp:213)
            const int p = end - jb;
            const uint4 nk = lds128(mk_sa + 16u * (uint32_t)(clamp08(p) * 9 + clamp08(p + 1)));    // clear = column end only
            const uint32_t h1rep = mad_u((uint32_t)h1, k10001, 0u);
            H0 = bitsel(H0, h1rep, nk.x); H1 = bitsel(H1, h1rep, nk.y); H2 = bitsel(H2, h1rep, nk.z); H3 = bitsel(H3, h1rep, nk.w);
            E0 &= nk.x; E1 &= nk.y; E2 &= nk.z; E3 &= nk.w;
        }
        key = wp.rmax(key);
        const int jfin = end > beg ? end : beg;
        if (jfin == qlen) {                                   // bandedSWA.cpp:214-217
            if (end > beg) h1 = wp.rmax(hend);
            if (!(st.gscore > h1)) st.max_ie = i;
            st.gscore = st.gscore > h1 ? st.gscore : h1;
        }
        const int m = key >> 16, mj = key & 0xffff;
        // row epilogue: global max / max_off / z-drop (bsw_row_update on the register copies of the parameters)
        if (m == 0) break;
        if (m > st.max) {
            st.max = m; st.max_i = i; st.max_j = mj;
            int d = mj - i; d = d < 0 ? -d : d;
            st.max_off = st.max_off > d ? st.max_off : d;
        } else {
            const int di = i - st.max_i, dj = mj - st.max_j;
            bool stop;
            if (zmode_r == 0) stop = st.max - m - (di > dj ? di - dj : dj - di) > zdrop_r;
            else if (zdrop_r > 0) stop = di > dj ? st.max - m - (di - dj) * P.e_del > zdrop_r : st.max - m - (dj - di) * P.e_ins > zdrop_r;
            else stop = false;
            if (stop) break;
        }
        // next row's window (bandedSWA.cpp:230-233) from the non-zero maps of what this row stored
        // (m != 0 here, so the window was not empty)
        {
            const int f_ = wp.rmin(fnz);
            beg = f_ < end ? f_ : end;
            int jj = wp.rmax(lnz);
            jj = jj >= 0 ? jj : beg - 1;
            end = jj + 2 < qlen ? jj + 2 : qlen;
        }
    }
#undef W16_WORD
#undef W16_ZMAP
}

} // namespace w16

// ------------------------------------------------------------------------------------------------
// Kernel: one pair per warp, BLOCK / 32 pairs per block; arguments as bsw_short16_kernel.  Every pair of
// [first, first + count) must have a query of at most w16::MAX_QLEN bases.  perm == nullptr: results in input
// order (the latency route); cell_counter == nullptr: a result's .w carries the pair's effective cells.
// Dynamic shared memory: w16::MASK_BYTES + (BLOCK / 32) * w16::SCORE_BYTES.
// ------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
template <int BLOCK, bool SAMEGAP>
__global__ void __launch_bounds__(BLOCK)
bsw_warp16_kernel(const int4* __restrict__ meta, const uint32_t* __restrict__ perm,
                  const uint32_t* __restrict__ qseq, const uint32_t* __restrict__ tseq,
                  int4* __restrict__ res, int first, int count,
                  const __grid_constant__ KParams P, unsigned long long* __restrict__ cell_counter)
{
    extern __shared__ __align__(16) uint32_t w16_smem[];
    const int tid = threadIdx.x;
    for (int k = tid; k < w16::MASK_BYTES / 4; k += BLOCK) w16_smem[k] = w16::mask_word((k >> 2) / 9, (k >> 2) % 9, k & 3);
    __syncthreads();
    const int local = blockIdx.x * (BLOCK / 32) + (tid >> 5);
    if (local >= count) return;
    const int4 md = meta[first + local];
    if (md.w & BSW_META_NFLAG) return;
    const uint32_t smem_sa = (uint32_t)__cvta_generic_to_shared(w16_smem);
    w16::Warp wp;
    wp.lane = tid & 31;
    wp.hx = nullptr;
    PairState st;
    long long my_cells = 0;
    w16::warp_sweep<SAMEGAP>(P, md, qseq + (uint32_t)md.x, tseq + (uint32_t)md.y, smem_sa,
                             smem_sa + w16::MASK_BYTES + (uint32_t)(tid >> 5) * w16::SCORE_BYTES, wp, st, my_cells);
    if (wp.lane == 0) {
        int4 r = bsw_pack_result(st);
        if (cell_counter) atomicAdd(cell_counter, (unsigned long long)my_cells);
        else r.w = (int)my_cells;
        res[perm ? perm[first + local] : (uint32_t)(first + local)] = r;
    }
}
#endif

} // namespace bsw
