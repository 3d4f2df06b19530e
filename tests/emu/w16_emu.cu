// w16_emu.cu -- TEST INFRASTRUCTURE: runs the warp-per-pair register kernel's row sweep (w16::warp_sweep, the
// same source the GPU executes) on the CPU.  The 32 lanes of a warp are 32 coroutines (ucontext) of one host thread,
// scheduled round-robin: a collective (shuffle, REDUX) is "hand in my value, yield, read everyone's" -- by the time a
// lane runs again all 32 have handed theirs in, because every lane executes the same sequence of collectives (the
// kernel's control flow is warp-uniform; a lane that strays deadlocks or trips the state comparison below).  The DPX
// .S16x2 instructions and the shared-memory window are emulated as in k16_emu.cu.  tests/test_w16_emulation.py
// compares the results with the oracle and the golden vectors without a GPU.  Built by tests/emu/build.py with
// nvcc as host code.
#include <vector>
#include <thread>
#include <cstdio>
#include <algorithm>
#include <ucontext.h>
#include "../../include/bsw.h"
#include "../../genomicsbench_b200/csrc/bsw_warp16.cuh"

using namespace bsw;

namespace bsw { namespace w16 {

struct HostExchange {
    int slot[2][32];            // double-buffered: a lane may be one collective ahead of the others, never two
    int round[32] = {};         // collectives a lane has entered
    ucontext_t ctx[32], main_ctx;
    bool done[32] = {};
};

// switch from `lane` to the next lane that is still running (round-robin); to the scheduler when none is
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

}} // namespace bsw::w16

namespace {

void pack2bit(const uint8_t* s, int n, std::vector<uint32_t>& out)
{
    out.assign((size_t)(n + 15) / 16 + 1, 0u);
    for (int k = 0; k < n; ++k) out[(size_t)k >> 4] |= (uint32_t)(s[k] & 3) << (2 * (k & 15));
}

KParams make_params(const int* prm, int w)
{
    KParams P{};
    P.match = prm[0]; P.mismatch_neg = -prm[1]; P.ambig = -1;
    P.o_del = prm[2]; P.e_del = prm[3]; P.o_ins = prm[4]; P.e_ins = prm[5];
    P.oe_del = P.o_del + P.e_del; P.oe_ins = P.o_ins + P.e_ins;
    P.zdrop = prm[6]; P.end_bonus = prm[7]; P.zmode = prm[8];
    P.mx = std::max(P.match, P.mismatch_neg); P.w = w; P.kone = 1;
    return P;
}

// one emulated warp, reused for the pairs of one host thread
struct WarpEmu {
    static constexpr int WARPS = 3;                      // warps of the emulated block (score words at different offsets)
    static constexpr size_t STACK = 128 << 10;
    w16::HostExchange hx;
    std::vector<uint8_t> smem, stacks;
    const KParams* P = nullptr;
    int4 md{};
    const uint32_t* qw = nullptr; const uint32_t* tw = nullptr;
    uint32_t sc_sa = 0;
    PairState sts[32];
    long long cells[32];

    explicit WarpEmu(int fill) : smem(w16::MASK_BYTES + WARPS * w16::SCORE_BYTES + 64, (uint8_t)fill), stacks(32 * STACK)
    {
        uint32_t* tab = reinterpret_cast<uint32_t*>(smem.data());
        for (int k = 0; k < w16::MASK_BYTES / 4; ++k) tab[k] = w16::mask_word((k >> 2) / 9, (k >> 2) % 9, k & 3);
    }
    static void lane_entry(unsigned lo, unsigned hi, int lane)
    {
        WarpEmu* self = reinterpret_cast<WarpEmu*>(((uintptr_t)hi << 32) | lo);
        self->lane_run(lane);
    }
    void lane_run(int lane)
    {
        w16::Warp wp;
        wp.lane = lane; wp.hx = &hx;
        long long c = 0;
        if (P->oe_del == P->oe_ins) w16::warp_sweep<true>(*P, md, qw, tw, 0u, sc_sa, wp, sts[lane], c);
        else w16::warp_sweep<false>(*P, md, qw, tw, 0u, sc_sa, wp, sts[lane], c);
        cells[lane] = c;
        hx.done[lane] = true;
        w16::hx_yield(&hx, lane);                        // never returns here
    }
    // runs one pair; false when the lanes ended with different states
    bool run(const KParams& prm, const int4 m, const uint32_t* q, const uint32_t* t, int warp_slot, PairState& st, long long& c)
    {
        P = &prm; md = m; qw = q; tw = t;
        sc_sa = (uint32_t)w16::MASK_BYTES + (uint32_t)(warp_slot % WARPS) * w16::SCORE_BYTES;
        k16::emu_smem = smem.data();
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
        k16::emu_smem = nullptr;
        for (int l = 0; l < 32; ++l) if (!hx.done[l]) return false;
        for (int l = 1; l < 32; ++l) if (memcmp(&sts[l], &sts[0], sizeof(PairState)) != 0) return false;
        st = sts[0]; c = cells[0];
        for (int l = 1; l < 32; ++l) c += cells[l];
        return true;
    }
};

} // namespace

extern "C" {

// params: match, mismatch(+), o_del, e_del, o_ins, e_ins, zdrop, end_bonus, zmode.
// batch over SeqPair records (one base per byte, codes 0-3); skipped[i] = 1 for pairs outside the kernel's domain
// (w16::scoring_ok, 16-bit scores, queries <= w16::MAX_QLEN).  fill: the byte shared memory holds before the first pair
// (pads must not matter).  Returns the effective cells, -1 when the lanes of a warp disagreed.
long long w16_emu_batch(const int* prm, SeqPair* pairs, const uint8_t* ref, const uint8_t* qer, long long n, int w,
                        int fill, uint8_t* skipped, long long* overflows)
{
    const KParams P = make_params(prm, w);
    const int nth = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<long long> cells((size_t)nth, 0), ovf((size_t)nth, 0);
    std::vector<int> bad((size_t)nth, 0);
    auto worker = [&](int t) {
        WarpEmu emu(fill);
        std::vector<uint32_t> qw, tw;
        k16::emu_overflows = 0;
        for (long long i = t; i < n; i += nth) {
            SeqPair& sp = pairs[i];
            const bool ok = w16::scoring_ok(P) && k16::eligible(P.match, sp.len2, sp.h0) && sp.len2 <= w16::MAX_QLEN;
            if (skipped) skipped[i] = ok ? 0 : 1;
            if (!ok) continue;
            pack2bit(qer + sp.idq, sp.len2, qw); pack2bit(ref + sp.idr, sp.len1, tw);
            PairState st;
            long long c = 0;
            if (!emu.run(P, make_int4(0, 0, sp.len2 | (sp.len1 << 16), sp.h0), qw.data(), tw.data(), (int)i, st, c)) {
                fprintf(stderr, "w16_emu: lanes disagree on pair %lld\n", i);
                bad[(size_t)t] = 1;
                continue;
            }
            sp.score = st.max; sp.qle = st.max_j + 1; sp.tle = st.max_i + 1; sp.gtle = st.max_ie + 1;
            sp.gscore = st.gscore; sp.max_off = st.max_off;
            cells[(size_t)t] += c;
        }
        ovf[(size_t)t] = k16::emu_overflows;
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nth; ++t) th.emplace_back(worker, t);
    worker(0);
    for (auto& t : th) t.join();
    long long total = 0, o = 0;
    for (int t = 0; t < nth; ++t) { total += cells[(size_t)t]; o += ovf[(size_t)t]; if (bad[(size_t)t]) total = -1; }
    if (overflows) *overflows = o;
    for (int t = 0; t < nth; ++t) if (bad[(size_t)t]) return -1;
    return total;
}

} // extern "C"
