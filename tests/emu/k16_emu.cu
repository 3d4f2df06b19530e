// k16_emu.cu -- TEST INFRASTRUCTURE: runs the packed kernel's row sweep (k16::pair_sweep, the
// same source the GPU executes) on the CPU, with the DPX .S16x2 instructions and the shared-memory
// window emulated, so tests/test_k16_emulation.py can compare it with the oracle without a GPU.
// Built by tests/emu/build.py with nvcc as host code.
#include <vector>
#include <cstdio>
#include <algorithm>
#include "../../include/bsw.h"
#include "../../genomicsbench_b200/csrc/bsw_kernel16.cuh"

using namespace bsw;

namespace {
// same rule as the engine (bsw_engine.cu stride_for)
int stride_for(int qmax)
{
    const int need = qmax + 8;
    int q;
    if (need <= 136) q = (need + 3) / 4;
    else if (need <= 520) q = ((need + 15) & ~15) / 4;
    else q = ((need + 31) & ~31) / 4;
    if (!(q & 1)) ++q;
    return 4 * q;
}

void pack2bit(const uint8_t* s, int n, std::vector<uint32_t>& out)
{
    out.assign((size_t)(n + 15) / 16 + 1, 0u);
    for (int k = 0; k < n; ++k) out[(size_t)k >> 4] |= (uint32_t)(s[k] & 3) << (2 * (k & 15));
}
} // namespace

extern "C" {

// params: match, mismatch(+), o_del, e_del, o_ins, e_ins, zdrop, end_bonus, zmode
// returns 0, or 1 when the pair is outside the packed kernel's domain; out6 = score qle tle gtle gscore max_off
// circ != 0: circular rows of k16::circ_cols(w) columns (what the engine runs when the band is narrower than the query)
// fill: the byte shared memory holds before the pair (the GPU leaves whatever was there; pads must not matter)
int k16_emu_pair2(const int* prm, const uint8_t* q, int qlen, const uint8_t* t, int tlen, int h0, int w,
                  int tid, int block, int circ, int fill, int* out6, long long* cells, long long* overflows)
{
    KParams P{};
    P.match = prm[0]; P.mismatch_neg = -prm[1]; P.ambig = -1;
    P.o_del = prm[2]; P.e_del = prm[3]; P.o_ins = prm[4]; P.e_ins = prm[5];
    P.oe_del = P.o_del + P.e_del; P.oe_ins = P.o_ins + P.e_ins;
    P.zdrop = prm[6]; P.end_bonus = prm[7]; P.zmode = prm[8];
    P.mx = std::max(P.match, P.mismatch_neg); P.w = w; P.kone = 1;
    if (!k16::eligible(P.match, qlen, h0)) return 1;
    const int plane = stride_for(qlen);
    int qstride = plane, wcols = 0;
    if (circ && k16::circ_cols(w) + 4 < plane) { wcols = k16::circ_cols(w); qstride = wcols + 4; }
    std::vector<uint8_t> smem(k16::smem_bytes(block, qstride, plane) + 64, (uint8_t)fill);
    k16::emu_smem = smem.data();
    k16::emu_overflows = 0;
    uint32_t* tab = reinterpret_cast<uint32_t*>(smem.data());
    for (int k = 0; k < k16::TAB_WORDS; ++k) tab[k] = k16::table_word(P, k >> 5);
    std::vector<uint32_t> qw, tw;
    pack2bit(q, qlen, qw); pack2bit(t, tlen, tw);
    const int4 md = make_int4(0, 0, qlen | (tlen << 16), h0);
    const uint32_t eh_sa = k16::TAB_BYTES + (uint32_t)(tid * qstride) * 4u;
    const uint32_t qp_sa = k16::TAB_BYTES + (uint32_t)(block * qstride) * 4u + (uint32_t)tid * 2u;
    const uint32_t tab_sa = (uint32_t)(tid & 31) * 4u;
    PairState st;
    long long c = 0;
    const uint32_t qps = (uint32_t)block * 2u;
    if (wcols) {
        if (P.oe_del == P.oe_ins) k16::pair_sweep<true, true>(P, md, qw.data(), tw.data(), eh_sa, qp_sa, qps, tab_sa, st, c, (uint32_t)wcols);
        else k16::pair_sweep<false, true>(P, md, qw.data(), tw.data(), eh_sa, qp_sa, qps, tab_sa, st, c, (uint32_t)wcols);
    } else {
        if (P.oe_del == P.oe_ins) k16::pair_sweep<true, false>(P, md, qw.data(), tw.data(), eh_sa, qp_sa, qps, tab_sa, st, c);
        else k16::pair_sweep<false, false>(P, md, qw.data(), tw.data(), eh_sa, qp_sa, qps, tab_sa, st, c);
    }
    out6[0] = st.max; out6[1] = st.max_j + 1; out6[2] = st.max_i + 1; out6[3] = st.max_ie + 1;
    out6[4] = st.gscore; out6[5] = st.max_off;
    if (cells) *cells = c;
    if (overflows) *overflows = k16::emu_overflows;
    k16::emu_smem = nullptr;
    return 0;
}

int k16_emu_pair(const int* prm, const uint8_t* q, int qlen, const uint8_t* t, int tlen, int h0, int w,
                 int tid, int block, int* out6, long long* cells, long long* overflows)
{
    return k16_emu_pair2(prm, q, qlen, t, tlen, h0, w, tid, block, 0, 0xA5, out6, cells, overflows);
}

// batch over SeqPair records (one base per byte, codes 0-3); skipped[i] = 1 for pairs outside the domain
long long k16_emu_batch2(const int* prm, SeqPair* pairs, const uint8_t* ref, const uint8_t* qer, long long n, int w,
                         int circ, int fill, uint8_t* skipped, long long* overflows)
{
    long long total = 0, ovf = 0;
#pragma omp parallel for schedule(dynamic, 64) reduction(+ : total, ovf)
    for (long long i = 0; i < n; ++i) {
        SeqPair& sp = pairs[i];
        int out[6]; long long c = 0, o = 0;
        const int rc = k16_emu_pair2(prm, qer + sp.idq, sp.len2, ref + sp.idr, sp.len1, sp.h0, w,
                                     (int)(i % 64), 64, circ, fill, out, &c, &o);
        if (skipped) skipped[i] = (uint8_t)rc;
        if (rc) continue;
        sp.score = out[0]; sp.qle = out[1]; sp.tle = out[2]; sp.gtle = out[3]; sp.gscore = out[4]; sp.max_off = out[5];
        total += c; ovf += o;
    }
    if (overflows) *overflows = ovf;
    return total;
}

long long k16_emu_batch(const int* prm, SeqPair* pairs, const uint8_t* ref, const uint8_t* qer, long long n, int w,
                        uint8_t* skipped, long long* overflows)
{
    return k16_emu_batch2(prm, pairs, ref, qer, n, w, 0, 0xA5, skipped, overflows);
}

} // extern "C"
