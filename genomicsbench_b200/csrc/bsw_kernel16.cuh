// bsw_kernel16.cuh -- the packed short-pair kernel: two DP columns per DPX instruction.
//
// Same per-pair semantics as bsw_short_kernel (bsw_kernels.cuh; SURVEY.md Appendix A ==
// benchmarks/bsw/bandedSWA.cpp:128-249 with the z-drop rule of :323-336), same thread-per-pair
// row sweep over the adaptive window, but the row lives in shared memory as two 16-bit planes
// and the recurrence runs on the .S16x2 forms of the DPX instructions (VIADDMNMX.S16x2,
// VIMNMX.S16x2, VIMNMX3.S16x2 -- same issue rate as the 32-bit forms, two cells each):
//
//   group g of a thread's row (16 bytes, one LDS.128 / STS.128) = columns 4g .. 4g+3:
//     word 0 = hs[4g+1] << 16 | hs[4g]      word 1 = hs[4g+3] << 16 | hs[4g+2]
//     word 2 = es[4g+1] << 16 | es[4g]      word 3 = es[4g+3] << 16 | es[4g+2]
//   hs[j] = eh[j].h = H(i-1, j-1), es[j] = eh[j].e = E(i, j)  (bandedSWA.cpp:196-213)
//
//   per pair word (columns c, c+1), everything elementwise in the two halves:
//     M  = max(min(Hd + S, Hd * (1 + match)), 0)   M = Hd ? Hd + s : 0, clamped (the cap is 0 iff Hd is)
//     U  = max(M - oe_del, 0)          E' = max(E - e_del, U)
//     A  = max(M - oe_ins, 0)          (= U when oe_ins == oe_del: template SAMEGAP)
//     ME = max(M, E)
//   the only sequential part is F; it runs in the HIGH halves, one VIADDMNMX per column:
//     F(c+1) = max(F(c) - e_ins, A(c))   F(c+2) = max(F(c+1) - e_ins, A(c+1))
//   and one PRMT gathers (F(c+1) | F(c)) for  H = max(ME, F).  One more PRMT per word shifts the
//   new H values by one column (eh[j].h receives H(i, j-1)).
//   The match scores S of a column pair come from a 16-entry table (one copy per lane, bank =
//   lane) indexed by the pair's 4 bits of  query ^ target;  the index arithmetic runs on the
//   FMA pipe (IMAD.SHL + IMAD.HI), so a score costs no ALU-pipe instruction.
//   Row maximum: per 8-column block one key  max(H) << 16 | last column of the block; the exact
//   column (the LAST one holding the maximum, bandedSWA.cpp:202-203) is resolved after the row
//   from the h plane, and only when the row epilogue needs it.
//
// Domain of this kernel: (h0 + len2 * match) * (1 + match) <= 32767: every H, E, F and every
// intermediate computed from them fits 16 signed bits and the cap trick holds.  The pack kernel
// routes everything else, and the pairs that contain N, to the 32-bit byte kernel.
// One computation may wrap, harmlessly: the row-maximum epilogue flags, with hs + (1 - m), the
// halfwords of the block that holds the row maximum m plus one halfword on either side, and the
// halfwords of columns from end on are not values of this row: they hold stale values, first-row
// values or, never written, whatever shared memory held (a fill byte in the host emulation).  A
// negative one v wraps whenever v + 1 - m < -32768 (for -32768 already at m = 2), and one above m
// would be flagged; neither matters, because the flags of those columns, and of the two halfwords
// outside the block, are masked off before the highest flag is taken.
// tests/test_scoring_domain.py runs the emulation with several fill bytes and requires equal results.
//
// The row sweep is __host__ __device__: tests/k16_emu.cu runs it on the CPU with emulated DPX
// instructions and an emulated shared-memory window, so the arithmetic is checked against the
// oracle without a GPU as well.
#pragma once
#include <cstring>
#include "bsw_kernels.cuh"

namespace bsw {
namespace k16 {

constexpr int TAB_WORDS = 16 * 32;            // 16 pair patterns x 32 lane copies
constexpr int TAB_BYTES = TAB_WORDS * 4;

// host emulation state (tests/emu; unused by the product)
inline thread_local uint8_t* emu_smem = nullptr;
inline thread_local long long emu_overflows = 0;
#if !defined(__CUDA_ARCH__)
inline int16_t emu_wrap(int v)
{
    if (v < -32768 || v > 32767) ++emu_overflows;
    return (int16_t)v;
}
#endif

// ---- shared-memory accessors (addresses are 32-bit shared-window addresses) ------------------
BSW_HD uint4 lds128(uint32_t a)
{
    uint4 v;
#if defined(__CUDA_ARCH__)
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
#else
    memcpy(&v, emu_smem + a, 16);
#endif
    return v;
}
BSW_HD void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w)
{
#if defined(__CUDA_ARCH__)
    asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
#else
    const uint32_t v[4] = {x, y, z, w};
    memcpy(emu_smem + a, v, 16);
#endif
}
BSW_HD uint32_t lds32(uint32_t a)
{
    uint32_t v;
#if defined(__CUDA_ARCH__)
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
#else
    memcpy(&v, emu_smem + a, 4);
#endif
    return v;
}
BSW_HD uint32_t lds16(uint32_t a)
{
    uint32_t v;
#if defined(__CUDA_ARCH__)
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
#else
    uint16_t h;
    memcpy(&h, emu_smem + a, 2);
    v = h;
#endif
    return v;
}
BSW_HD void sts16(uint32_t a, uint32_t x)
{
#if defined(__CUDA_ARCH__)
    asm volatile("st.shared.u16 [%0], %1;" :: "r"(a), "r"(x) : "memory");
#else
    const uint16_t h = (uint16_t)x;
    memcpy(emu_smem + a, &h, 2);
#endif
}
BSW_HD uint32_t ldg32(const uint32_t* p)
{
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

// ---- DPX .S16x2 instructions and the FMA-pipe helpers -----------------------------------------
#if !defined(__CUDA_ARCH__)
#define K16_EMU2(EXPR)                                                                            \
    uint32_t r_ = 0;                                                                              \
    for (int s_ = 0; s_ < 32; s_ += 16) {                                                         \
        const int x = (int16_t)(a >> s_), y = (int16_t)(b >> s_), z = (int16_t)(c >> s_);        \
        (void)x; (void)y; (void)z;                                                                \
        r_ |= (uint32_t)(uint16_t)(EXPR) << s_;                                                   \
    }                                                                                             \
    return r_;
#endif
BSW_HD uint32_t addmin_relu(uint32_t a, uint32_t b, uint32_t c)     // max(min(a + b, c), 0)
{
#if defined(__CUDA_ARCH__)
    return __viaddmin_s16x2_relu(a, b, c);
#else
    K16_EMU2(std::max<int>(std::min<int>(emu_wrap(x + y), z), 0))
#endif
}
BSW_HD uint32_t addmax_relu(uint32_t a, uint32_t b, uint32_t c)     // max(a + b, c, 0)
{
#if defined(__CUDA_ARCH__)
    return __viaddmax_s16x2_relu(a, b, c);
#else
    K16_EMU2(std::max<int>(std::max<int>(emu_wrap(x + y), z), 0))
#endif
}
BSW_HD uint32_t addmax(uint32_t a, uint32_t b, uint32_t c)          // max(a + b, c)
{
#if defined(__CUDA_ARCH__)
    return __viaddmax_s16x2(a, b, c);
#else
    K16_EMU2(std::max<int>(emu_wrap(x + y), z))
#endif
}
BSW_HD uint32_t max2(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __vmaxs2(a, b);
#else
    const uint32_t c = 0;
    K16_EMU2(std::max<int>(x, y))
#endif
}
BSW_HD uint32_t max3(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    return __vimax3_s16x2(a, b, c);
#else
    K16_EMU2(std::max<int>(std::max<int>(x, y), z))
#endif
}
BSW_HD uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(a, b, sel);
#else
    const uint64_t ab = ((uint64_t)b << 32) | a;
    uint32_t r = 0;
    for (int k = 0; k < 4; ++k) r |= (uint32_t)((ab >> (8 * ((sel >> (4 * k)) & 7))) & 0xff) << (8 * k);
    return r;
#endif
}
BSW_HD int imax3(int a, int b, int c)
{
#if defined(__CUDA_ARCH__)
    return __vimax3_s32(a, b, c);
#else
    return std::max(std::max(a, b), c);
#endif
}
// a * b + c on the FMA pipe (IMAD)
BSW_HD uint32_t mad_u(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
#else
    return a * b + c;
#endif
}
// hi32(a * b) + c on the FMA pipe (IMAD.HI.U32)
BSW_HD uint32_t madhi_u(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("mad.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
#else
    return (uint32_t)(((uint64_t)a * b) >> 32) + c;
#endif
}

// index of the highest set bit (x != 0)
BSW_HD int hibit(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return 31 - __clz((int)x);
#else
    int r = 0;
    while (x >>= 1) ++r;
    return r;
#endif
}

// a << s: 0 for s >= 32 and for negative s (PTX shl takes the amount as unsigned and clamps it; C++ << does not)
BSW_HD uint32_t shl_sat(uint32_t a, int s)
{
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(s));
    return r;
#else
    return (unsigned)s >= 32u ? 0u : a << s;
#endif
}
BSW_HD int imax0(int a) { return a > 0 ? a : 0; }
// per-halfword unsigned minimum
BSW_HD uint32_t minu2(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __vminu2(a, b);
#else
    const uint32_t lo = std::min(a & 0xffffu, b & 0xffffu), hi = std::min(a >> 16, b >> 16);
    return lo | (hi << 16);
#endif
}
// bits of b where the mask is set, bits of a elsewhere (one LOP3)
BSW_HD uint32_t bitsel(uint32_t a, uint32_t b, uint32_t keep_b_mask_inv)
{
    // keep_b_mask_inv = 1 bits: keep a (the old content); 0 bits: take b (the new content)
    return (a & keep_b_mask_inv) | (b & ~keep_b_mask_inv);
}
// index of the lowest set bit (x != 0)
BSW_HD int lobit(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __ffs((int)x) - 1;
#else
    int r = 0;
    while (!(x & 1u)) { x >>= 1; ++r; }
    return r;
#endif
}

BSW_HD uint32_t pack2(int hi, int lo) { return ((uint32_t)hi << 16) | ((uint32_t)lo & 0xffffu); }

// score-table word of pattern idx = x1 << 2 | x0 (x = query ^ target of the two columns, 0 = match)
BSW_HD uint32_t table_word(const KParams& P, int idx)
{
    return pack2((idx >> 2) ? P.mismatch_neg : P.match, (idx & 3) ? P.mismatch_neg : P.match);
}

// true when the packed kernel may run the pair (see the header comment)
BSW_HD bool eligible(int match, int qlen, int h0)
{
    return (long long)(h0 + (long long)qlen * match) * (1 + match) <= 32767;
}

// ------------------------------------------------------------------------------------------------
// Row sweep of one pair.
//   md        {query word offset (unused here), target word offset (unused), qlen | tlen << 16, h0}
//   qw, tw    2-bit packed query / target, 16 bases per word
//   eh_sa     this thread's row (S words, groups of 16 bytes as described above)
//   qp_sa     this thread's slot of the query plane: halfword k (columns 8k .. 8k+7, 2 bits per
//             base) at qp_sa + k * qp_stride
//   tab_sa    score table + 4 * lane
//
// A row's window [beg, end) is swept in aligned blocks of 8 columns, from the block holding column
// beg to the block holding column end (which receives eh[end] = {H(i, end-1), 0},
// bandedSWA.cpp:213).
//   Left of beg: the columns between the block boundary and beg are dead for good (beg never
//   decreases) and hold zeros -- a column leaves the window either because its (h | e) is zero
//   (bandedSWA.cpp:230) or because the band cuts it (:175), and then the row prologue zeroes it.
//   Swept as zeros they produce zeros, the state the reference enters beg with when beg > 0, so
//   the first block needs no mask.
//   Right of end: the last block runs the same recurrence under three halfword masks:
//     in    columns >= end enter as h = e = 0 (their results are discarded)
//     key   the row maximum only looks at columns < end (F leaks into the discarded ones)
//     store columns <= end are written, columns > end keep their old content (the reference leaves
//           them untouched, and later rows may read them: SURVEY.md Appendix B, stale eh[])
// The first and the last block also produce, from the values they store, an 8-bit map of the
// columns whose (h | e) is non-zero; the next row's window (bandedSWA.cpp:230-233) is read off
// these two maps and only falls back to scanning shared memory when a map is empty.
// ------------------------------------------------------------------------------------------------
// CIRC = true: the row is a circular buffer of wcols columns (a multiple of 8, >= 2 w + 16): a row sweep only
// ever touches the columns [beg, end] with beg >= i - w and end <= i + w + 1, column j lives in slot j mod wcols,
// and a column's slot is reused wcols columns later, when that column has been dead (left of the first block)
// for good.  Columns that enter the band for the first time receive their first-row value
// max(h0 - oe_ins - (j-1) e_ins, 0) (the closed form of bandedSWA.cpp:155-157) just before the first row whose
// last block can cover them, so the stale-eh[] behaviour (SURVEY.md Appendix B) is unchanged.  Queries longer
// than the band then cost the band's shared memory, not the query's.
template <bool SAMEGAP, bool CIRC = false>
BSW_HD void pair_sweep(const KParams& P, const int4 md, const uint32_t* __restrict__ qw,
                       const uint32_t* __restrict__ tw, const uint32_t eh_sa_in, const uint32_t qp_sa,
                       const uint32_t qp_stride, const uint32_t tab_sa, PairState& st, long long& my_cells,
                       const uint32_t wcols = 0)
{
    const int qlen = md.z & 0xffff, tlen = (md.z >> 16) & 0xffff, h0 = md.w & 0xffff;
    // loop constants are pinned in registers through an opaque zero (see bsw_short_kernel): the row's address -- else
    // the shared window's base is re-derived from special registers inside every row epilogue -- and the z-drop
    // parameters, which the compiler otherwise re-loads from the constant bank in every row, a dependent stall each
    // time (profiles/r02k_sass_sweep_w100_launch0.txt)
    const uint32_t zero = (uint32_t)md.z >> 31;
    const uint32_t eh_sa = eh_sa_in + zero;
    const int zdrop_r = P.zdrop + (int)zero, zmode_r = P.zmode + (int)zero;
    const int e_del_r = P.e_del + (int)zero, h1_base = h0 - P.o_del + (int)zero;

    // ---- first row (bandedSWA.cpp:155-157) and the query plane; the row is initialised up to the
    // end of the block that holds column qlen
    // x mod wcols for x < 2^16 (one IMAD.HI + one IMAD on the FMA pipe); identity when the row is not circular
    const uint32_t rcpw = CIRC ? (uint32_t)((0x100000000ull + wcols - 1) / wcols) : 0u;
#define K16_MODW(X) (CIRC ? (uint32_t)(X) - wcols * madhi_u((uint32_t)(X), rcpw, 0u) : (uint32_t)(X))
#define K16_NEXT(SA) (CIRC ? ((SA) + 32u == row_end ? eh_sa : (SA) + 32u) : (SA) + 32u)
    const uint32_t row_end = eh_sa + 4u * wcols;
    const int init_cols = CIRC && (int)wcols < (qlen | 7) + 1 ? (int)wcols : (qlen | 7) + 1;
    int init_next = init_cols;                        // CIRC: first column whose slot still holds an older column
    {
        int hv = h0;
        for (int j0 = 0; j0 < init_cols; j0 += 4) {
            uint32_t v[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int j = j0 + c;
                if (j == 1) hv = h0 > P.oe_ins ? h0 - P.oe_ins : 0;
                else if (j >= 2) hv = hv > P.e_ins ? hv - P.e_ins : 0;
                v[c] = j <= qlen ? (uint32_t)hv : 0u;
            }
            sts128(eh_sa + 4u * (uint32_t)j0, v[0] | (v[1] << 16), v[2] | (v[3] << 16), 0u, 0u);
        }
        const int nw = (qlen + 15) >> 4;
        uint32_t qa = qp_sa;
        for (int k = 0; k < nw; ++k) {
            const uint32_t v = ldg32(qw + k);
            sts16(qa, v & 0xffffu);
            sts16(qa + qp_stride, v >> 16);
            qa += 2 * qp_stride;
        }
    }
    const int w = bsw_clamp_band(P, qlen);

    st.max = h0; st.max_i = -1; st.max_j = -1; st.max_ie = -1; st.gscore = -1; st.max_off = 0;
    int beg = 0, end = qlen;
    uint32_t tword = 0;
    const uint32_t noe_del2 = zero + pack2(-P.oe_del, -P.oe_del);
    const uint32_t noe_ins2 = zero + pack2(-P.oe_ins, -P.oe_ins);
    const uint32_t ne_del2 = zero + pack2(-P.e_del, -P.e_del);
    const uint32_t negg_hi = zero + pack2(-P.e_ins, 0);
    const uint32_t capmul = zero + (uint32_t)(1 + P.match);
    const uint32_t k65536 = zero + 65536u * (uint32_t)P.kone;
    const uint32_t k16c = zero + 16u * (uint32_t)P.kone;
    const uint32_t k128 = zero + 128u * (uint32_t)P.kone;
    (void)noe_ins2;

    // address of column j's h half (its e half is 8 bytes further)
#define K16_HADDR(J) (eh_sa + ((K16_MODW(J) >> 2) << 4) + (((uint32_t)(J) & 3u) << 1))
    // score word of pair K (columns 2K, 2K+1 of the block) from the block's x halfword: the pair's
    // nibble is isolated by a left shift + IMAD.HI (x 16 = >> 28), scaled to the table stride by an IMAD
#define K16_SCORE(X, K) lds32(mad_u(madhi_u((X) << (28 - 4 * (K)), k16c, 0u), k128, tab_sa))
    // one pair word: HW / EW loaded halves, SW scores; HN = new H of the two columns, EN = new E
#define K16_WORD(HW, EW, SW, HN, EN)                                                              \
    {                                                                                             \
        const uint32_t cap_ = mad_u((HW), capmul, 0u);                                            \
        const uint32_t M_ = addmin_relu((HW), (SW), cap_);                                        \
        const uint32_t U_ = addmax_relu(M_, noe_del2, zero);                                      \
        EN = addmax((EW), ne_del2, U_);                                                           \
        const uint32_t A_ = SAMEGAP ? U_ : addmax_relu(M_, noe_ins2, zero);                       \
        const uint32_t ME_ = max2(M_, (EW));                                                      \
        const uint32_t f1_ = addmax(fc, negg_hi, mad_u(A_, k65536, 0u));                          \
        const uint32_t Fc_ = prmt(fc, f1_, 0x7632);                                               \
        fc = addmax(f1_, negg_hi, A_);                                                            \
        HN = max2(ME_, Fc_);                                                                      \
    }
    // one interior 4-column group: CUR = its four words, SA / SB = scores of its two pairs
#define K16_GROUP(CUR, SA, SB, ADDR, HN0, HN1)                                                    \
    {                                                                                             \
        uint32_t en0_, en1_;                                                                      \
        K16_WORD((CUR).x, (CUR).z, (SA), HN0, en0_)                                               \
        K16_WORD((CUR).y, (CUR).w, (SB), HN1, en1_)                                               \
        sts128((ADDR), prmt(carry, HN0, 0x5432), prmt(HN0, HN1, 0x5432), en0_, en1_);             \
        carry = HN1;                                                                              \
    }
    // row-maximum key of a block whose packed maximum is G and whose last column is CODE
#define K16_KEY(G, CODE)                                                                          \
    mkey = imax3(mkey, (int)(((G) & 0xffff0000u) | (uint32_t)(CODE)), (int)mad_u((G), k65536, (uint32_t)(CODE)));
    // the block at sa computes from (c0, c1, s0..s3) while the next block's row words, score words
    // and the query halfword after that are loaded into (n0, n1, t0..t3, xb); xa = the next block's
    // query halfword ^ target.  (The shared-memory accesses are volatile, so ptxas keeps the loads
    // ahead of the block's stores instead of sinking them to their use.)
#define K16_PREFETCH(XA, N0, N1, T0, T1, T2, T3, XB)                                              \
    const uint32_t san_ = K16_NEXT(sa);                                                           \
    N0 = lds128(san_); N1 = lds128(san_ + 16);                                                    \
    T0 = K16_SCORE(XA, 0); T1 = K16_SCORE(XA, 1); T2 = K16_SCORE(XA, 2); T3 = K16_SCORE(XA, 3);   \
    XB = lds16(qa + 2 * qp_stride) ^ trep;
#define K16_BLOCK(C0, C1, S0, S1, S2, S3, XA, N0, N1, T0, T1, T2, T3, XB)                         \
    {                                                                                             \
        uint32_t hn0, hn1, hn2, hn3;                                                              \
        K16_PREFETCH(XA, N0, N1, T0, T1, T2, T3, XB)                                              \
        K16_GROUP(C0, S0, S1, sa, hn0, hn1)                                                       \
        K16_GROUP(C1, S2, S3, sa + 16, hn2, hn3)                                                  \
        const uint32_t g_ = max2(max3(hn0, hn1, hn2), hn3);                                       \
        K16_KEY(g_, code)                                                                         \
        sa = san_; qa += qp_stride; code += 8;                                                    \
    }
    // 8-bit map of the non-zero halfwords of four words (bit c = column c of the block)
#define K16_ZMAP(Z0, Z1, Z2, Z3, ZMAP)                                                            \
    {                                                                                             \
        const uint32_t f0_ = minu2((Z0), 0x00010001u), f1_ = minu2((Z1), 0x00010001u);            \
        const uint32_t f2_ = minu2((Z2), 0x00010001u), f3_ = minu2((Z3), 0x00010001u);            \
        const uint32_t zb_ = mad_u(f3_, 64u, mad_u(f2_, 16u, mad_u(f1_, 4u, f0_)));               \
        ZMAP = (zb_ | (zb_ >> 15)) & 0xffu;                                                       \
    }
    // first block of a window that spans several blocks: the bare recurrence + the non-zero map
#define K16_FIRST(ZMAP)                                                                           \
    {                                                                                             \
        uint4 n0, n1;                                                                             \
        uint32_t t0, t1, t2, t3, xb;                                                              \
        K16_PREFETCH(xa, n0, n1, t0, t1, t2, t3, xb)                                              \
        uint32_t hn0, hn1, hn2, hn3, en0, en1, en2, en3;                                          \
        K16_WORD(c0.x, c0.z, s0, hn0, en0)                                                        \
        K16_WORD(c0.y, c0.w, s1, hn1, en1)                                                        \
        const uint32_t hw0 = prmt(carry, hn0, 0x5432), hw1 = prmt(hn0, hn1, 0x5432);              \
        sts128(sa, hw0, hw1, en0, en1);                                                           \
        K16_WORD(c1.x, c1.z, s2, hn2, en2)                                                        \
        K16_WORD(c1.y, c1.w, s3, hn3, en3)                                                        \
        const uint32_t hw2 = prmt(hn1, hn2, 0x5432), hw3 = prmt(hn2, hn3, 0x5432);                \
        sts128(sa + 16, hw2, hw3, en2, en3);                                                      \
        carry = hn3;                                                                              \
        const uint32_t g_ = max2(max3(hn0, hn1, hn2), hn3);                                       \
        K16_KEY(g_, code)                                                                         \
        K16_ZMAP(hw0 | en0, hw1 | en1, hw2 | en2, hw3 | en3, ZMAP)                                \
        sa = san_; qa += qp_stride; code += 8;                                                    \
        c0 = n0; c1 = n1; s0 = t0; s1 = t1; s2 = t2; s3 = t3; xa = xb;                            \
    }
    // halfword mask of word K of a block: the columns >= D16 / 16 (D16 = 16 x a column count in 0..8)
#define K16_GE(D16, K) shl_sat(0xffffffffu, imax0((D16) - 32 * (K)))
    // last block: LIVE16 = 16 x (columns of the block left of end, 0..7).  ZMAP receives the non-zero
    // map of the stored columns (<= end), HEND the h half stored at column end (H(i, end - 1)).
#define K16_EDGE(LIVE16, ZMAP, HEND)                                                              \
    {                                                                                             \
        const int l16_ = (LIVE16);                                                                \
        const uint32_t rk0 = K16_GE(l16_, 0), rk1 = K16_GE(l16_, 1), rk2 = K16_GE(l16_, 2), rk3 = K16_GE(l16_, 3);   \
        const uint32_t sk0 = K16_GE(l16_ + 16, 0), sk1 = K16_GE(l16_ + 16, 1), sk2 = K16_GE(l16_ + 16, 2), sk3 = K16_GE(l16_ + 16, 3); \
        uint32_t hn0, hn1, hn2, hn3, en0, en1, en2, en3;                                          \
        K16_WORD(c0.x & ~rk0, c0.z & ~rk0, s0, hn0, en0)                                          \
        K16_WORD(c0.y & ~rk1, c0.w & ~rk1, s1, hn1, en1)                                          \
        K16_WORD(c1.x & ~rk2, c1.z & ~rk2, s2, hn2, en2)                                          \
        K16_WORD(c1.y & ~rk3, c1.w & ~rk3, s3, hn3, en3)                                          \
        const uint32_t hw0 = prmt(carry, hn0, 0x5432), hw1 = prmt(hn0, hn1, 0x5432);              \
        const uint32_t hw2 = prmt(hn1, hn2, 0x5432), hw3 = prmt(hn2, hn3, 0x5432);                \
        sts128(sa, bitsel(c0.x, hw0, sk0), bitsel(c0.y, hw1, sk1), bitsel(c0.z, en0, sk0), bitsel(c0.w, en1, sk1));       \
        sts128(sa + 16, bitsel(c1.x, hw2, sk2), bitsel(c1.y, hw3, sk3), bitsel(c1.z, en2, sk2), bitsel(c1.w, en3, sk3));  \
        const uint32_t g_ = max2(max3(hn0 & ~rk0, hn1 & ~rk1, hn2 & ~rk2), hn3 & ~rk3);          \
        K16_KEY(g_, code)                                                                         \
        K16_ZMAP((hw0 | en0) & ~sk0, (hw1 | en1) & ~sk1, (hw2 | en2) & ~sk2, (hw3 | en3) & ~sk3, ZMAP)  \
        {                                                                                         \
            const uint32_t ws_ = (l16_ & 64) ? ((l16_ & 32) ? hw3 : hw2) : ((l16_ & 32) ? hw1 : hw0);   \
            HEND = (int)((l16_ & 16) ? ws_ >> 16 : ws_ & 0xffffu);                                \
        }                                                                                         \
    }

    for (int i = 0; i < tlen; ++i) {
        if ((i & 15) == 0) tword = ldg32(tw + (i >> 4));
        const int ti = (int)((tword >> ((i & 15) * 2)) & 3u);
        if (beg < i - w) {
            // the band cuts column beg (at most one column per row: beg >= i - 1 - w): dead for good,
            // zeroed so that the first block can sweep it unmasked
            const uint32_t ha = K16_HADDR(beg);
            sts16(ha, 0u);
            sts16(ha + 8, 0u);
            beg = i - w;
        }
        end = end < i + w + 1 ? end : i + w + 1;
        end = end < qlen ? end : qlen;
        int h1 = 0;
        if (beg == 0) { h1 = h1_base - e_del_r * (i + 1); h1 = h1 > 0 ? h1 : 0; }
        if (CIRC) {
            // first-row values for the columns this row's last block may reach for the first time
            int need_hi = i + w + 1 < qlen ? i + w + 1 : qlen;
            need_hi |= 7;
            while (init_next <= need_hi) {
                uint32_t v[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int j = init_next + c;
                    const int hv = h0 - P.oe_ins - (j - 1) * P.e_ins;
                    v[c] = j <= qlen && hv > 0 ? (uint32_t)hv : 0u;
                }
                sts128(eh_sa + 4u * K16_MODW(init_next), v[0] | (v[1] << 16), v[2] | (v[3] << 16), 0u, 0u);
                init_next += 4;
            }
        }
        int mkey = 0;                     // (row max << 16) | last column of the block that holds it
        uint32_t zf = 0, zl = 0;          // non-zero maps of the first / last block
        const int fb = beg & ~7, lb = end & ~7;
        if (end > beg) {
            const uint32_t trep = (uint32_t)ti * 0x5555u;
            uint32_t fc = 0;                                  // high half: F entering the next column
            uint32_t carry = (uint32_t)h1 << 16;              // high half: H(i, j - 1)
            uint32_t sa = eh_sa + 4u * K16_MODW(fb);
            uint32_t qa = qp_sa + ((uint32_t)fb >> 3) * qp_stride;
            int code = fb + 7;
            uint4 c0 = lds128(sa), c1 = lds128(sa + 16);
            uint32_t s0, s1, s2, s3, xa;
            {
                const uint32_t x = lds16(qa) ^ trep;
                s0 = K16_SCORE(x, 0); s1 = K16_SCORE(x, 1); s2 = K16_SCORE(x, 2); s3 = K16_SCORE(x, 3);
                xa = lds16(qa + qp_stride) ^ trep;
            }
            if (lb > fb) {
                K16_FIRST(zf)
                // interior blocks, unrolled twice over two register sets
                int nmid = ((lb - fb) >> 3) - 1;
                if (nmid > 0) {
                    uint4 n0, n1;
                    uint32_t t0, t1, t2, t3, xb;
                    for (;;) {
                        K16_BLOCK(c0, c1, s0, s1, s2, s3, xa, n0, n1, t0, t1, t2, t3, xb)
                        if (--nmid == 0) { c0 = n0; c1 = n1; s0 = t0; s1 = t1; s2 = t2; s3 = t3; break; }
                        K16_BLOCK(n0, n1, t0, t1, t2, t3, xb, c0, c1, s0, s1, s2, s3, xa)
                        if (--nmid == 0) break;
                    }
                }
            }
            K16_EDGE(16 * (end - lb), zl, h1)
            if (lb == fb) zf = zl;
            my_cells += end - beg;
        } else {
            // empty window: eh[end] = {h1, 0}  (bandedSWA.cpp:213)
            const uint32_t ha = K16_HADDR(end);
            sts16(ha, (uint32_t)h1);
            sts16(ha + 8, 0u);
        }
        const int jfin = end > beg ? end : beg;
        if (jfin == qlen) {                                   // bandedSWA.cpp:214-217
            if (!(st.gscore > h1)) st.max_ie = i;
            st.gscore = st.gscore > h1 ? st.gscore : h1;
        }
        const int m = mkey >> 16;
        int mj = mkey & 0xffff;
        if (m > st.max || (m != 0 && st.max - m > zdrop_r)) {
            // (m == 0 ends the pair in bsw_row_update before mj is looked at -- and an empty window leaves
            // mkey = 0, whose "block" would lie in front of this thread's row: compute-sanitizer's racecheck
            // flagged those reads against the neighbouring thread's stores)
            // the key names a block (its last column, mj + 1 a multiple of 8): the reference's mj is
            // the last column of [mj - 7, mj] whose H equals m (bandedSWA.cpp:202-203).  H(i, c) sits
            // in hs[c + 1]; the eight halves are flagged in parallel (1 where hs >= m: inside this
            // row's sweep no H exceeds m; columns left of beg hold zeros, columns from end on are
            // masked out) and the highest flag taken.  The epilogue reads mj only under the condition above.
            const uint32_t gb = eh_sa + 4u * K16_MODW(mj - 7);            // the block [mj - 7, mj] ...
            const uint32_t ga = eh_sa + 4u * K16_MODW(mj + 1);            // ... and the first group of the next one
            const uint32_t a0 = lds32(gb), a1 = lds32(gb + 4), b0 = lds32(gb + 16), b1 = lds32(gb + 20), c0 = lds32(ga);
            const uint32_t dm = pack2(1 - m, 1 - m), one2 = 0x00010001u;
            const uint32_t fa0 = addmin_relu(a0, dm, one2), fa1 = addmin_relu(a1, dm, one2);
            const uint32_t fb0 = addmin_relu(b0, dm, one2), fb1 = addmin_relu(b1, dm, one2), fc0 = addmin_relu(c0, dm, one2);
            // bit k of the mask = column mj - 7 + k
            const uint32_t xw = mad_u(fc0, 128u, mad_u(fb1, 32u, mad_u(fb0, 8u, fa1 * 2u)));
            uint32_t mask = (xw & 0xaau) | ((xw >> 15) & 0x54u) | (fa0 >> 16);
            if (mj >= end) mask &= (1u << (end - (mj - 7))) - 1u;
            mj = mj - 7 + hibit(mask);
        }
        // row epilogue: global max / max_off / z-drop (bsw_row_update, on the register copies of the parameters)
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
        // next row's window (bandedSWA.cpp:230-233): first non-zero column of [beg, end), then the
        // last non-zero column of [beg', end]
        if (end > beg) {
            uint32_t zb = zf;
            if (lb == fb) zb &= ~(1u << (end - fb));
            int jj;
            if (zb) jj = fb + lobit(zb);
            else {
                // the first block holds no live column: look for the first one a whole block at a time (two 128-bit
                // loads and one non-zero map per 8 columns; on divergent pairs this search runs more than once per
                // row, for one or two lanes of the warp at a time, and a column-by-column loop of dependent 16-bit
                // loads cost 6 % of the kernel, profiles/r02k_sass_sweep_w100_launch0.txt)
                jj = end;
                for (int jb = fb + 8; jb < end; jb += 8) {
                    const uint32_t ba = eh_sa + 4u * K16_MODW(jb);
                    const uint4 b0 = lds128(ba), b1 = lds128(ba + 16);
                    uint32_t zm;
                    K16_ZMAP(b0.x | b0.z, b0.y | b0.w, b1.x | b1.z, b1.y | b1.w, zm)
                    if (zm) { jj = jb + lobit(zm); break; }
                }
                jj = jj < end ? jj : end;              // (columns from end on may hold stale non-zero cells)
            }
            beg = jj;
            const uint32_t ze = beg > lb ? zl & (0xffu << (beg - lb)) : zl;
            if (ze) jj = lb + hibit(ze);
            else {
                jj = beg - 1;
                for (int jb = lb - 8; jb + 7 >= beg; jb -= 8) {
                    const uint32_t ba = eh_sa + 4u * K16_MODW(jb);
                    const uint4 b0 = lds128(ba), b1 = lds128(ba + 16);
                    uint32_t zm;
                    K16_ZMAP(b0.x | b0.z, b0.y | b0.w, b1.x | b1.z, b1.y | b1.w, zm)
                    if (jb < beg) zm &= 0xffu << (beg - jb);
                    if (zm) { jj = jb + hibit(zm); break; }
                }
            }
            end = jj + 2 < qlen ? jj + 2 : qlen;
        }
        // (an empty window has m == 0 and stopped the pair above)
    }
#undef K16_MODW
#undef K16_NEXT
#undef K16_HADDR
#undef K16_SCORE
#undef K16_WORD
#undef K16_GROUP
#undef K16_KEY
#undef K16_PREFETCH
#undef K16_BLOCK
#undef K16_GE
#undef K16_ZMAP
#undef K16_FIRST
#undef K16_EDGE
}

// shared memory of one block: score table + rows (rowstride words per thread) + query plane (sized by
// the class's full query stride qstride, which equals rowstride unless the rows are circular)
BSW_HD size_t smem_bytes(int block, int rowstride, int qstride)
{
    return (size_t)TAB_BYTES + (size_t)rowstride * block * 4 + (size_t)((qstride >> 3) + 2) * block * 2;
}
BSW_HD size_t smem_bytes(int block, int qstride) { return smem_bytes(block, qstride, qstride); }

// columns of the circular row for band w (pair_sweep<.., true>): a multiple of 8, >= 2 w + 16
BSW_HD int circ_cols(int w) { return (2 * w + 16 + 7) & ~7; }

} // namespace k16

// ------------------------------------------------------------------------------------------------
// Kernel: one pair per thread; same arguments as bsw_short_kernel<BLOCK, false>.
// ------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
// qstride = words per thread row; wcols = 0, or the columns of the circular row (then qstride = wcols + 4: the
// padding keeps qstride / 4 odd, i.e. the 128-bit accesses of a quarter warp in distinct bank groups)
// perm == nullptr: results in input order; cell_counter == nullptr: a result's .w carries the pair's effective cells
// (both: the latency route under load, run_tiny)
template <int BLOCK, bool SAMEGAP, bool CIRC = false>
__global__ void __launch_bounds__(BLOCK)
bsw_short16_kernel(const int4* __restrict__ meta, const uint32_t* __restrict__ perm,
                   const uint32_t* __restrict__ qseq, const uint32_t* __restrict__ tseq,
                   int4* __restrict__ res, int first, int count, int qstride,
                   const __grid_constant__ KParams P, unsigned long long* __restrict__ cell_counter, int wcols = 0)
{
    extern __shared__ __align__(16) uint32_t k16_smem[];
    const int tid = threadIdx.x;
    for (int k = tid; k < k16::TAB_WORDS; k += BLOCK) k16_smem[k] = k16::table_word(P, k >> 5);
    __syncthreads();
    const int local = blockIdx.x * BLOCK + tid;
    long long my_cells = 0;
    if (local < count) {
        const int4 md = meta[first + local];
        if (!(md.w & BSW_META_NFLAG)) {
            const uint32_t smem_sa = (uint32_t)__cvta_generic_to_shared(k16_smem);
            const uint32_t eh_sa = smem_sa + k16::TAB_BYTES + (uint32_t)(tid * qstride) * 4u;
            const uint32_t qp_sa = smem_sa + k16::TAB_BYTES + (uint32_t)(BLOCK * qstride) * 4u + (uint32_t)tid * 2u;
            const uint32_t tab_sa = smem_sa + (uint32_t)(tid & 31) * 4u;
            PairState st;
            k16::pair_sweep<SAMEGAP, CIRC>(P, md, qseq + (uint32_t)md.x, tseq + (uint32_t)md.y, eh_sa, qp_sa, BLOCK * 2u,
                                           tab_sa, st, my_cells, (uint32_t)wcols);
            int4 r = bsw_pack_result(st);
            if (!cell_counter) r.w = (int)my_cells;
            res[perm ? perm[first + local] : (uint32_t)(first + local)] = r;
        }
    }
    if (!cell_counter) return;
    for (int off = 16; off > 0; off >>= 1) my_cells += __shfl_down_sync(0xffffffffu, my_cells, off);
    if ((tid & 31) == 0 && my_cells) atomicAdd(cell_counter, (unsigned long long)my_cells);
}
#endif

} // namespace bsw
