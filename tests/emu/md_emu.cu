// md_emu.cu -- TEST INFRASTRUCTURE: runs bsw_reg2aln's finishing-pass sweeps (md::md_sweep, the same source the GPU
// executes) on the CPU, the 32 lanes of a warp as coroutines of one host thread through l32_emu.cu's host exchange.
// The MD buffer is filled with garbage before every region, so a byte the write sweep misses shows up.
// tests/test_reg2aln.py compiles it with nvcc as host code and compares the results with the oracle.
#include "l32_emu.cu"
#include "../../genomicsbench_b200/csrc/bsw_md.cuh"

namespace {

struct MdEmu {
    static constexpr size_t STACK = 128 << 10;
    l32::HostExchange hx;
    std::vector<uint8_t> stacks;
    const uint8_t* q = nullptr; const uint8_t* r = nullptr; const uint32_t* cg = nullptr;
    int n_cig = 0, rev = 0;
    md::MdScore S{};
    char* out = nullptr;
    md::MdCount cnt[32];

    MdEmu() : stacks(32 * STACK) {}
    static void lane_entry(unsigned lo, unsigned hi, int lane)
    {
        MdEmu* self = reinterpret_cast<MdEmu*>(((uintptr_t)hi << 32) | lo);
        self->lane_run(lane);
    }
    void lane_run(int lane)
    {
        l32::Warp wp;
        wp.lane = lane; wp.hx = &hx;
        cnt[lane] = md::md_sweep<false>(q, r, cg, n_cig, rev, S, nullptr, wp);
        wp.sync();
        const md::MdCount c2 = md::md_sweep<true>(q, r, cg, n_cig, rev, S, out, wp);
        if (c2.md_len != cnt[lane].md_len) cnt[lane].md_len = -1;
        hx.done[lane] = true;
        l32::hx_yield(&hx, lane);                        // never returns here
    }
    bool run(const uint8_t* qb, const uint8_t* rb, const uint32_t* c, int nc, int rv, const md::MdScore& sc, char* o,
             md::MdCount& res)
    {
        q = qb; r = rb; cg = c; n_cig = nc; rev = rv; S = sc; out = o;
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
        for (int l = 0; l < 32; ++l)
            if (cnt[l].md_len < 0 || cnt[l].md_len != cnt[0].md_len || cnt[l].n_mm != cnt[0].n_mm ||
                cnt[l].n_gap != cnt[0].n_gap || cnt[l].msc != cnt[0].msc) return false;
        res = cnt[0];
        return true;
    }
};

} // namespace

extern "C" {

// score: match, mismatch (+), ambig.  Region i: query q[qoff[i] ..], reference r[roff[i] ..] (both as the DP aligned them:
// reversed on the reverse strand), operations cig[coff[i] .. + n_cig[i]) before the squeeze, rev[i].  Writes
// md[md_room[i] .. + md_len[i]) (the buffer is filled with '#' by the caller), nm[i], msc[i].  Returns 0, or -1 when the
// lanes of a warp disagreed or the two sweeps' lengths differ.
int md_emu_batch(const int* score, long long n, const uint8_t* q, const long long* qoff, const uint8_t* r,
                 const long long* roff, const uint32_t* cig, const long long* coff, const int* n_cig, const int* rev,
                 char* md, const long long* md_room, int* md_len, int* nm, int* msc)
{
    const md::MdScore S{score[0], -score[1], score[2]};
    const int nth = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
    std::vector<int> bad((size_t)nth, 0);
    auto worker = [&](int th) {
        MdEmu emu;
        for (long long i = th; i < n; i += nth) {
            md::MdCount c{};
            if (!emu.run(q + qoff[i], r + roff[i], cig + coff[i], n_cig[i], rev[i], S, md + md_room[i], c)) {
                fprintf(stderr, "md_emu: lanes disagree on region %lld\n", i);
                bad[(size_t)th] = 1;
                continue;
            }
            md_len[i] = c.md_len; nm[i] = c.n_mm + c.n_gap; msc[i] = c.msc;
        }
    };
    std::vector<std::thread> th;
    for (int k = 1; k < nth; ++k) th.emplace_back(worker, k);
    worker(0);
    for (auto& x : th) x.join();
    for (int k = 0; k < nth; ++k) if (bad[(size_t)k]) return -1;
    return 0;
}

} // extern "C"
