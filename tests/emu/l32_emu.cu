// l32_emu.cu -- TEST INFRASTRUCTURE: runs the int32 ring kernel's row sweep (l32::sweep, the same source the GPU
// executes) on the CPU.  The 32 lanes of a warp are 32 coroutines (ucontext) of one host thread, scheduled round-robin
// as in w16_emu.cu: a collective is "hand in my value, yield, read everyone's".  The ring is filled with garbage before
// every pair, so a slot read before the sweep wrote it (a virgin cell the rule missed) shows up as a wrong result.
// tests/test_extend32.py compiles it with nvcc as host code (its `emu` fixture) and compares the results with the
// oracle and the golden vectors.
#include <vector>
#include <thread>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <ucontext.h>
#include "../../include/bsw.h"
#include "../../genomicsbench_b200/csrc/bsw_long32.cuh"

using namespace bsw;

namespace bsw { namespace l32 {

struct HostExchange {
    int slot[2][32];            // double-buffered: a lane may be one collective ahead of the others, never two
    int round[32] = {};
    ucontext_t ctx[32], main_ctx;
    bool done[32] = {};
};

static void hx_yield(HostExchange* hx, int lane)
{
    for (int k = 1; k <= 32; ++k) {
        const int nx = (lane + k) & 31;
        if (!hx->done[nx]) {
            if (nx != lane) swapcontext(&hx->ctx[lane], &hx->ctx[nx]);
            return;
        }
    }
    swapcontext(&hx->ctx[lane], &hx->main_ctx);
}

const int* hx_all(HostExchange* hx, int lane, int v)
{
    const int r = hx->round[lane]++ & 1;
    hx->slot[r][lane] = v;
    hx_yield(hx, lane);
    return hx->slot[r];
}

}} // namespace bsw::l32

namespace {

struct WarpEmu {
    static constexpr size_t STACK = 128 << 10;
    l32::HostExchange hx;
    std::vector<uint8_t> stacks;
    std::vector<int> ring;
    const KParams* P = nullptr;
    const uint8_t* q = nullptr; const uint8_t* t = nullptr;
    int qlen = 0, tlen = 0, h0 = 0, K = 0;
    PairState sts[32];
    long long cells[32];

    WarpEmu() : stacks(32 * STACK) {}
    static void lane_entry(unsigned lo, unsigned hi, int lane)
    {
        WarpEmu* self = reinterpret_cast<WarpEmu*>(((uintptr_t)hi << 32) | lo);
        self->lane_run(lane);
    }
    void lane_run(int lane)
    {
        l32::Warp wp;
        wp.lane = lane; wp.hx = &hx;
        long long c = 0;
        l32::sweep(*P, q, qlen, t, tlen, h0, ring.data(), ring.data() + K, K, wp, sts[lane], c);
        cells[lane] = c;
        hx.done[lane] = true;
        l32::hx_yield(&hx, lane);                        // never returns here
    }
    bool run(const KParams& prm, const uint8_t* qb, int ql, const uint8_t* tb, int tl, int h, int k, PairState& st, long long& c)
    {
        P = &prm; q = qb; t = tb; qlen = ql; tlen = tl; h0 = h; K = k;
        ring.assign((size_t)2 * K + 4, 0x5a5a5a5a);       // garbage: no slot may be read before it is written
        for (int l = 0; l < 32; ++l) {
            hx.done[l] = false; hx.round[l] = 0;
            getcontext(&hx.ctx[l]);
            hx.ctx[l].uc_stack.ss_sp = stacks.data() + (size_t)l * STACK;
            hx.ctx[l].uc_stack.ss_size = STACK;
            hx.ctx[l].uc_link = &hx.main_ctx;
            const uintptr_t p = (uintptr_t)this;
            makecontext(&hx.ctx[l], (void (*)())lane_entry, 3, (unsigned)(p & 0xffffffffu), (unsigned)(p >> 32), l);
        }
        swapcontext(&hx.main_ctx, &hx.ctx[0]);
        for (int l = 0; l < 32; ++l) if (!hx.done[l]) return false;
        for (int l = 1; l < 32; ++l) if (memcmp(&sts[l], &sts[0], sizeof(PairState)) != 0) return false;
        st = sts[0]; c = 0;
        for (int l = 0; l < 32; ++l) c += cells[l];
        return true;
    }
};

KParams make_params(const int* prm, int w)
{
    KParams P{};
    P.match = prm[0]; P.mismatch_neg = -prm[1]; P.ambig = prm[9];
    P.o_del = prm[2]; P.e_del = prm[3]; P.o_ins = prm[4]; P.e_ins = prm[5];
    P.oe_del = P.o_del + P.e_del; P.oe_ins = P.o_ins + P.e_ins;
    P.zdrop = prm[6]; P.end_bonus = prm[7]; P.zmode = prm[8];
    P.mx = std::max(std::max(P.match, P.mismatch_neg), P.ambig); P.w = w; P.kone = 1;
    return P;
}

} // namespace

extern "C" {

// params: match, mismatch(+), o_del, e_del, o_ins, e_ins, zdrop, end_bonus, zmode, ambig.  Batch over SeqPair records
// (one base per byte, codes 0-4), results in place.  ring_k > 0 forces that many ring slots (a multiple of 128 at
// least l32::ring_slots of every pair), 0 = each pair's own ring_slots.  Returns the effective cells, -1 when the lanes
// of a warp disagreed.
long long l32_emu_batch(const int* prm, SeqPair* pairs, const uint8_t* ref, const uint8_t* qer, long long n, int w, int ring_k)
{
    const KParams P = make_params(prm, w);
    const int nth = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<long long> cells((size_t)nth, 0);
    std::vector<int> bad((size_t)nth, 0);
    auto worker = [&](int t) {
        WarpEmu emu;
        for (long long i = t; i < n; i += nth) {
            SeqPair& sp = pairs[i];
            const int K = ring_k > 0 ? ring_k : l32::ring_slots(sp.len2, bsw_clamp_band(P, sp.len2));
            PairState st;
            long long c = 0;
            if (!emu.run(P, qer + sp.idq, sp.len2, ref + sp.idr, sp.len1, sp.h0, K, st, c)) {
                fprintf(stderr, "l32_emu: lanes disagree on pair %lld\n", i);
                bad[(size_t)t] = 1;
                continue;
            }
            sp.score = st.max; sp.qle = st.max_j + 1; sp.tle = st.max_i + 1; sp.gtle = st.max_ie + 1;
            sp.gscore = st.gscore; sp.max_off = st.max_off;
            cells[(size_t)t] += c;
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nth; ++t) th.emplace_back(worker, t);
    worker(0);
    for (auto& t : th) t.join();
    long long total = 0;
    for (int t = 0; t < nth; ++t) { if (bad[(size_t)t]) return -1; total += cells[(size_t)t]; }
    return total;
}

// l32::ring_slots of a query length and the band after the clamp (the tests size forced rings with it)
int l32_ring_slots(const int* prm, int qlen, int w)
{
    const KParams P = make_params(prm, w);
    return l32::ring_slots(qlen, bsw_clamp_band(P, qlen));
}

} // extern "C"
