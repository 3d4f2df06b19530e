// g32_emu.cu -- TEST INFRASTRUCTURE: runs bsw_global32's row sweep and backtrack (g32::sweep / g32::backtrack, the same
// source the GPU executes) on the CPU, the 32 lanes of a warp as coroutines of one host thread through l32_emu.cu's
// host exchange.  The ring and the direction matrix are filled with garbage before every alignment, so a ring slot
// read before the sweep wrote it, or a direction the backtrack reads but the sweep never stored, shows up as a wrong
// result.  tests/test_global32.py compiles it with nvcc as host code and compares the results with the golden vectors
// and the oracle.
#include "l32_emu.cu"
#include "../../genomicsbench_b200/csrc/bsw_global32.cuh"
#include "../../genomicsbench_b200/csrc/bsw_global_plan.h"

namespace {

struct G32Emu {
    static constexpr size_t STACK = 128 << 10;
    l32::HostExchange hx;
    std::vector<uint8_t> stacks;
    std::vector<int> ring;
    std::vector<uint32_t> dz;                            // direction matrix (uint32_t: aligned for the tile loads)
    std::vector<uint32_t> tile;
    const GlobalParams* P = nullptr;
    const uint8_t* q = nullptr; const uint8_t* t = nullptr;
    uint32_t* cg = nullptr;
    int qlen = 0, tlen = 0, w = 0, K = 0;
    long long pitch = 0;
    int score[32], n_op[32];

    G32Emu() : stacks(32 * STACK), tile(g32::TILE_ROWS * g32::TILE_BYTES / 4) {}
    static void lane_entry(unsigned lo, unsigned hi, int lane)
    {
        G32Emu* self = reinterpret_cast<G32Emu*>(((uintptr_t)hi << 32) | lo);
        self->lane_run(lane);
    }
    void lane_run(int lane)
    {
        l32::Warp wp;
        wp.lane = lane; wp.hx = &hx;
        uint8_t* z = reinterpret_cast<uint8_t*>(dz.data());
        score[lane] = g32::sweep(*P, q, qlen, t, tlen, w, ring.data(), ring.data() + K, K, z, pitch, wp);
        wp.sync();                                       // (the kernels' boundary)
        n_op[lane] = g32::backtrack(z, pitch, qlen, tlen, w, cg, reinterpret_cast<uint8_t*>(tile.data()), wp);
        hx.done[lane] = true;
        l32::hx_yield(&hx, lane);                        // never returns here
    }
    bool run(const GlobalParams& prm, const uint8_t* qb, int ql, const uint8_t* tb, int tl, int wv, int k, uint32_t* out,
             int& sc, int& n)
    {
        P = &prm; q = qb; t = tb; qlen = ql; tlen = tl; w = wv; K = k; cg = out;
        pitch = g32::dir_pitch(qlen, w);
        ring.assign((size_t)2 * K + 4, 0x5a5a5a5a);     // garbage: no slot may be read before it is written
        dz.assign((size_t)(pitch * tlen / 4) + 16, 0xa5a5a5a5u);
        std::fill(tile.begin(), tile.end(), 0xa5a5a5a5u);
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
        for (int l = 1; l < 32; ++l) if (score[l] != score[0] || n_op[l] != n_op[0]) return false;
        sc = score[0]; n = n_op[0];
        return true;
    }
};

} // namespace

extern "C" {

// params: o_del, e_del, o_ins, e_ins, match, mismatch (+), ambig (the order of the golden files).  Alignment i: query
// qer[idq, + len2), target ref[idr, + len1), band w[i]; its operations go to cigar[cigar_off[i] ..] (room for
// len1 + len2).  ring_k > 0 forces that many ring slots (a multiple of 128, at least l32::ring_slots of every
// alignment), 0 = each alignment's own.  Returns 0, or -1 when the lanes of a warp disagreed.
int g32_emu_batch(const int* prm, const SeqPair* pairs, const uint8_t* ref, const uint8_t* qer, long long n, const int* w,
                  int ring_k, int* score, int* n_cigar, uint32_t* cigar, const long long* cigar_off)
{
    const GlobalParams P{prm[0], prm[1], prm[2], prm[3], prm[4], -prm[5], prm[6]};
    const int nth = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<int> bad((size_t)nth, 0);
    auto worker = [&](int th) {
        G32Emu emu;
        for (long long i = th; i < n; i += nth) {
            const SeqPair& sp = pairs[i];
            const int wv = g2::eff_w(sp.len2, sp.len1, w[i]);
            const int K = ring_k > 0 ? ring_k : l32::ring_slots(sp.len2, wv);
            if (!emu.run(P, qer + sp.idq, sp.len2, ref + sp.idr, sp.len1, wv, K, cigar + cigar_off[i], score[i], n_cigar[i])) {
                fprintf(stderr, "g32_emu: lanes disagree on alignment %lld\n", i);
                bad[(size_t)th] = 1;
            }
        }
    };
    std::vector<std::thread> th;
    for (int k = 1; k < nth; ++k) th.emplace_back(worker, k);
    worker(0);
    for (auto& x : th) x.join();
    for (int k = 0; k < nth; ++k) if (bad[(size_t)k]) return -1;
    return 0;
}

// ring slots of an alignment as the kernel sizes them (the tests size forced rings with it)
int g32_ring_slots(int qlen, int tlen, int w) { return l32::ring_slots(qlen, g2::eff_w(qlen, tlen, w)); }

} // extern "C"
