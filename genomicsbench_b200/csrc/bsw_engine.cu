// bsw_engine.cu -- engine object, chunk pipeline and kernel launches behind the C ABI (include/bsw.h).
//
// Stands in for BandedPairWiseSW's batch wrapper smithWatermanBatchWrapper16
// (benchmarks/bsw/bandedSWA.cpp:1150-1431).  Where the reference pads to the SIMD width, sorts by
// len1, transposes AoS->SoA per 16 pairs and calls the AVX kernel, this engine cuts the batch into
// chunks of consecutive pairs and runs every chunk through a device-side pipeline:
//
//   host buffers pinned (bsw_host_alloc / bsw_host_register, "direct" route):
//     DMA of the raw SeqPair records -> bsw_scan_pairs (validate, 16-byte descriptors, summary)
//     -> DMA of the byte range the chunk's sequences span (or zero-copy reads when that range is
//     sparse) -> bsw_bucket_* (counting sort by len2|h0|len1) -> bsw_pack_pairs (2 bits/base, processing order)
//     -> bsw_short_kernel per shared-memory class -> bsw_writeback into the device copy of the
//     records -> DMA of the records back.  The host touches no payload byte.
//   pageable host buffers ("staged" route):
//     host threads stream over the chunk once, in input order: descriptors + the sequences'
//     bytes gathered into pinned staging, H2D, then the same device stages; results come back by
//     D2H and a second streaming pass writes them into the caller's records.
//
// Chunk c+1 is prepared and copied while chunk c computes and chunk c-1 drains.  Pairs that
// contain N (code 4) or whose query exceeds the short kernel's shared-memory limit are listed by
// the pack kernel and run by the byte-reading kernels before the chunk's results leave.
#include "bsw_common.h"
#include "bsw_kernels.cuh"
#include "bsw_kernel16.cuh"
#include "bsw_warp16.cuh"
#include "bsw_long32.cuh"
#include "bsw_prep.cuh"
#include "bsw_global.cuh"
#include "bsw_global2.cuh"
#include "bsw_global_plan.h"
#include "bsw_global32.cuh"
#include "bsw_md.cuh"
#include <atomic>
#include <cstdio>
#include <cstring>
#include <string>
#include <memory>
#include <deque>
#include <climits>
#include <thread>
#include <condition_variable>
#include <type_traits>
#include <cuda.h>                         // types only: the driver entry points are fetched through the runtime

using namespace bsw;

namespace {

constexpr int SHORT_BLOCK = 64;           // threads (= pairs) per block of the short kernel
constexpr int SHORT_MAX_QLEN = 824;       // eh words + query byte plane of SHORT_BLOCK threads must fit 227 KB
constexpr int WARP_BLOCK = 128;           // threads per block of the warp-per-pair register kernel (bsw_warp16.cuh): 4 pairs
// default bsw_params.warp_max_pairs: pairs a device runs one per WARP at any moment, all calls and engines of the process
// together (see WarpLease)
constexpr int WARP_MAX_PAIRS = 4096;
constexpr int NSTREAMS = 16;              // DP compute streams per device (one shared-memory class each, run concurrently)
constexpr int NSLOTS = 8;                 // chunks in flight per device (records ahead / prepare / compute / drain, + slack before a slot is reused)
constexpr int64_t CHUNK_EXTEND = 1 << 18; // largest chunk of bsw_extend (overlap vs bucketing quality)
constexpr int64_t CHUNK_MIN = 1 << 15;    // the last chunks of a batch shrink towards this (short pipeline drain)
constexpr int64_t CHUNK_STAGE = 1 << 20;  // pairs per chunk of bsw_stage (resident: best bucketing)
constexpr int BUCKET_BITS = 18;           // bins of the counting sort (1 MB table)
constexpr long long OFF_BIAS = 1ll << 30; // bias of ChunkInfo::min_* / max_* (bsw_prep.cuh)
constexpr size_t BINS_WORDS = ((size_t)1 << BUCKET_BITS) + SCAN_MAX_TILES + 8;   // bin table + tile totals + ticket
constexpr int64_t CHUNK_PCIE = 3 << 15;   // chunk of a PCIe-bound batch (98 304 pairs): DP keeps pace with the arrivals

std::string g_create_error;
std::mutex g_err_mutex;
// BSW_TIMELINE=1: bsw_extend prints, per chunk, when each pipeline stage finished on the device and
// when the host reached its enqueue / wait points (diagnostic; the events then carry timestamps)
const bool g_timeline = getenv("BSW_TIMELINE") != nullptr;

// CUDA green contexts (driver API, CUDA >= 12.4), fetched with cudaGetDriverEntryPoint so that the
// library does not link libcuda (it must load, and export its symbols, on a box without a driver).
// They split a device's SMs into a small SERVICE partition for the chunk streams (copies, scan,
// bucket, pack, write-back) and a DP partition for the extension kernels: a DP launch fills every
// SM it may use to the register / shared-memory limit with blocks that live as long as the launch,
// and no stream priority evicts running blocks -- on shared SMs the next chunk's 10-microsecond
// prep kernels waited ~0.5 ms behind it and the copy engine idled (scripts/greenctx_probe.cu,
// BSW_TIMELINE).  Used for PCIe-bound batches only; compute-bound ones keep all SMs for the DP.
struct GreenApi {
    decltype(&cuDeviceGetDevResource) get_res = nullptr;
    decltype(&cuDevSmResourceSplitByCount) split = nullptr;
    decltype(&cuDevResourceGenerateDesc) gen_desc = nullptr;
    decltype(&cuGreenCtxCreate) create = nullptr;
    decltype(&cuGreenCtxStreamCreate) stream_create = nullptr;
    decltype(&cuGreenCtxDestroy) destroy = nullptr;
    bool ok = false;
    GreenApi()
    {
        auto get = [](const char* name, auto& fn) {
            void* p = nullptr;
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !p) {
                cudaGetLastError();
                return false;
            }
            fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(p);
            return true;
        };
        ok = get("cuDeviceGetDevResource", get_res) && get("cuDevSmResourceSplitByCount", split) &&
             get("cuDevResourceGenerateDesc", gen_desc) && get("cuGreenCtxCreate", create) &&
             get("cuGreenCtxStreamCreate", stream_create) && get("cuGreenCtxDestroy", destroy);
    }
};
const GreenApi& green_api() { static GreenApi g; return g; }

struct Launch {
    int first, count;     // range in the chunk's processing order
    int qstride;          // shared-memory row words per thread
    int block;            // threads (= pairs) per block: 64, or 32 where that keeps more warps resident
    int wcols = 0;        // packed kernel: columns of the circular row (then qstride = wcols + 4), 0 = the row holds the whole query
    int plane = 0;        // packed kernel: query stride that sizes the 2-bit query plane (= qstride unless circular)
    bool warp = false;    // the warp-per-pair register kernel (queries <= w16::MAX_QLEN)
};

template <class T>
struct Buf {              // grow-only device buffer with an optional pinned-host twin
    T* d = nullptr; T* h = nullptr; size_t cap = 0; size_t hcap = 0;
};

struct Slot {
    // buffers
    Buf<uint8_t> raw_pairs;               // device copy of the caller's records (direct route)
    Buf<int4> desc, meta, res;            // per pair: byte-offset descriptor, word-offset descriptor, result
    Buf<uint32_t> perm, rank, bins, nlist, llist, qpk, tpk, scratch;
    Buf<uint8_t> qraw, rraw;              // sequence bytes (device; pinned twin = staging of the staged route)
    ChunkInfo* d_info = nullptr; ChunkInfo* h_info = nullptr;
    ChunkInfo* h_info_dev = nullptr;      // device-side address of h_info (mapped page-locked memory)
    // speculative sequence copies of the direct route (direct_begin): absolute byte range per side
    bool spec[2] = {false, false};        // [0] query, [1] reference
    long long spec_lo[2] = {0, 0}, spec_hi[2] = {0, 0};
    unsigned int* d_queue = nullptr;
    cudaStream_t st{};                    // the stream the chunk in this slot runs on: st_plain or st_svc
    cudaStream_t st_plain{}, st_svc{};    // whole device (high priority) / service partition
    cudaEvent_t ev_rec{}, ev_seqd{};      // direct route: records / speculative sequence copy arrived (recorded on the H2D stream)
    bool bins_zeroed = false;             // the bin table was cleared at open()
    bool fork_recorded = false;           // ev_fork already marks the end of the prep kernels
    cudaEvent_t ev_tl[5] = {};            // BSW_TIMELINE: after zero / count / scan / scatter / pack
    cudaEvent_t ev_info{}, ev_dp{}, ev_out{}, ev_fork{}, ev_k0{}, ev_k1{}, ev_seq{}, ev_lists{};
    double host_t[6] = {};                // timeline: host clock at open / info / launched / dp seen / out enqueued / retired
    // chunk state
    int64_t a = 0; int n = 0;             // pairs [a, a + n) of the batch
    bool direct = false;
    bool out_records = false;             // direct route: results leave inside the records' device copy (one DMA, no host pass); else 16 B per pair + a host pass
    bool packed = false;                  // packed route (bsw_extend_packed): desc holds bsw_pair_desc records, results leave as OutScore
    bool src2bit = false;                 // the chunk's sequences arrived as 2-bit words (packed route, or packed by the staged route's host pass)
    Buf<uint8_t> tinybuf;                 // latency route: one block {queue word | descriptors | query bytes | reference bytes}
    Buf<uint8_t> rawq, rawr;              // staged route: RAW side buffer (pairs with N, long queries), page-locked twin + device copy
    bool use16 = true;                    // this chunk's short pairs run the packed 16-bit kernel
    const uint8_t* q2src = nullptr;       // packed route: device copy of the chunk's 2-bit words (query / reference) ...
    const uint8_t* r2src = nullptr;
    const uint32_t* dp_q = nullptr;       // 2-bit words the DP kernels read (the packed copies, or q2src / r2src in place)
    const uint32_t* dp_t = nullptr;
    unsigned int q_lo = 0, r_lo = 0;      // ... and the batch word offset of its first word
    Buf<uint8_t> outbuf;                  // packed route: OutScore records on their way out
    bool tiny = false;                    // latency route: every pair goes to the warp-per-pair kernel (run_pipeline)
    bool warp_ok = false;                 // the whole call is small enough for the warp-per-pair kernel (tail chunks of a large call are not)
    bool seq_on_device = false;           // both sequence buffers are device copies with >= 64 bytes of slack behind them
    const uint8_t* qbase = nullptr;       // device-visible address of descriptor offset 0 (query / reference)
    const uint8_t* rbase = nullptr;
    ChunkInfo info;                       // host copy used for planning
    std::vector<Launch> plan;
    int n_sorted = 0;                     // short pairs (in perm)
    unsigned n_nlist = 0, n_llist = 0; int qmax_n = 0;
    int long_stride = 0, long_blocks = 0;
};

struct DevCtx {
    int dev = 0;
    int sms = 148;
    cudaStream_t cs[NSTREAMS] = {};       // DP streams over the whole device (low priority)
    cudaStream_t cs_part[NSTREAMS] = {};  // DP streams of the DP partition
    cudaStream_t h2d{};                   // every host-to-device copy of the direct route, in chunk order (see direct_begin)
    CUgreenCtx g_svc = nullptr, g_dp = nullptr;
    int svc_sms = 0, dp_sms = 0;          // 0: no partitions on this device
    cudaEvent_t ev_join[NSTREAMS] = {};
    cudaEvent_t ev_t0{}, ev_t1{};         // device timeline of bsw_run_staged
    std::deque<Slot> slots;
    unsigned long long* d_cells = nullptr;
    unsigned long long* h_cells = nullptr;
    bool attr_set = false;
    // packed route: buffers of the batch that stay resident for the whole call (RAW sequences; every 2-bit word
    // when the batch is not ordered) and the event that marks their arrival
    Buf<uint8_t> rawq, rawr, allq, allr;
    cudaEvent_t ev_res{};
};

// What a call processes: the reference's layout (SeqPair records + one byte per base, results in place) or a
// packed batch (include/bsw.h: bsw_packed_batch) with a separate result array.
struct Job {
    SeqPair* pairs = nullptr; const uint8_t* seq_ref = nullptr; const uint8_t* seq_qer = nullptr;
    const bsw_packed_batch* pb = nullptr; void* out = nullptr; bool out16 = false;
    bool force_staged = false;            // page-locked buffers, but sequences spread over more than the direct route's 2^30-byte reach
};
constexpr int BSW_RETRY_STAGED = -100;    // internal: the direct route met such a chunk; the call is run again on the staged route

struct GlobalBufs;                        // bsw_global.inl
struct X32Bufs;                           // bsw_extend32.inl
struct G32Bufs;                           // bsw_global32.inl
struct MdBufs;                            // bsw_reg2aln.inl
struct ChainBufs;                         // bsw_chain.inl
struct AsyncQueue;                        // bsw_async.inl

} // namespace

struct ChainLanes;                        // bsw_chain.inl

struct bsw_engine {
    bsw_params p;
    KParams kp;
    std::deque<DevCtx> devs;
    std::unique_ptr<ThreadPool> pool;
    std::string err;
    bsw_stats stats;
    int short_max = SHORT_MAX_QLEN;       // longest query the short kernel takes
    bool use16 = true;                    // short pairs run the packed 16-bit kernel (bsw_kernel16.cuh)
    // staged batch (bsw_stage / bsw_run_staged / bsw_fetch)
    bool staged = false, ran = false;
    int64_t n = 0;
    int32_t w = 0;
    std::vector<std::pair<int, int>> staged_chunks;   // (device, slot) per chunk, batch order
    GlobalBufs* gbufs = nullptr;          // device buffers of bsw_global
    ChainBufs* cbufs = nullptr;           // page-locked staging of bsw_extend_chains
    bool cells_counted = false;           // the last run summed its effective cells itself (latency route): no device counters to collect
    ChainLanes* clanes = nullptr;         // child engines of bsw_extend_chains' lanes
    AsyncQueue* aq = nullptr;             // queue + worker of bsw_extend_async
    X32Bufs* x32bufs = nullptr;           // chunk buffers of bsw_extend32
    G32Bufs* g32bufs = nullptr;           // chunk buffers of bsw_global32
    MdBufs* mdbufs = nullptr;             // chunk buffers of bsw_reg2aln's finishing pass
    std::once_flag aq_once;
};

namespace {

// A call on an engine with several devices runs one host thread per device (run_sharded): each thread collects its
// statistics and its error text in its own Shard and points these at them; everywhere else they stay null and the
// engine's own members are used.
thread_local bsw_stats* t_stats = nullptr;
thread_local std::string* t_err = nullptr;
inline bsw_stats& stats_of(bsw_engine* eng) { return t_stats ? *t_stats : eng->stats; }
inline std::string& err_of(bsw_engine* eng) { return t_err ? *t_err : eng->err; }

#define CUDA_TRY(call)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            err_of(eng) = std::string(#call) + ": " + cudaGetErrorString(e_);                   \
            return BSW_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

template <class T>
int ensure(bsw_engine* eng, Buf<T>& b, size_t need, bool host = false)
{
    if (need > b.cap) {
        const size_t cap = std::max(need + need / 4, (size_t)1024);
        if (b.d) cudaFree(b.d);
        b.d = nullptr; b.cap = 0;
        CUDA_TRY(cudaMalloc((void**)&b.d, cap * sizeof(T)));
        b.cap = cap;
    }
    if (host && need > b.hcap) {
        const size_t cap = std::max(need + need / 4, (size_t)1024);
        if (b.h) cudaFreeHost(b.h);
        b.h = nullptr; b.hcap = 0;
        CUDA_TRY(cudaHostAlloc((void**)&b.h, cap * sizeof(T), cudaHostAllocDefault));
        b.hcap = cap;
    }
    return BSW_OK;
}

template <class T>
void release(Buf<T>& b)
{
    if (b.d) cudaFree(b.d);
    if (b.h) cudaFreeHost(b.h);
    b.d = nullptr; b.h = nullptr; b.cap = b.hcap = 0;
}

// One chunk in flight on the engine's first device (bsw_global, bsw_extend32, bsw_global32): its stream, the events around its
// kernels and the items of the call it holds.  The entry points add their own buffers on top.
struct ChunkSlot {
    cudaStream_t st{};
    cudaEvent_t e0{}, e1{};
    int64_t first = 0, m = 0;             // items [first, first + m) of the call
    ChunkSlot() = default; ChunkSlot(const ChunkSlot&) = delete;     // owns its stream and events
    ~ChunkSlot()
    {
        if (st) cudaStreamDestroy(st);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
    }
    int open(bsw_engine* eng)             // stream and events, created on first use
    {
        if (!st) {
            CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
            CUDA_TRY(cudaEventCreate(&e0));
            CUDA_TRY(cudaEventCreate(&e1));
        }
        return BSW_OK;
    }
    void add_kernel_ms(bsw_stats& S) const
    {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess) S.ms_kernel += (double)ms;
    }
};

// Runs n items through two alternating slots: launch(k, first) prepares the chunk from item `first` on in slot k (and
// sets its m) and enqueues its device work, finish(k) waits for slot k and moves its results out.  The host prepares
// chunk j + 1 while the device runs chunk j; the slots drain in submission order.  An error returns only after the
// device is synchronised, so that no copy still runs into a slot's or the caller's buffers.
template <class SlotT, class LaunchFn, class FinishFn>
int run_chunks(SlotT (&slot)[2], int64_t n, LaunchFn&& launch, FinishFn&& finish)
{
    bool pending[2] = {false, false};
    int cur = 0;
    for (int64_t next = 0; next < n || pending[0] || pending[1]; cur ^= 1) {
        if (pending[cur]) {
            if (int rc = finish(cur)) { cudaDeviceSynchronize(); return rc; }
            pending[cur] = false;
        }
        if (next < n) {
            if (int rc = launch(cur, next)) { cudaDeviceSynchronize(); return rc; }
            pending[cur] = true;
            next += slot[cur].m;
        }
    }
    return BSW_OK;
}

// Frees an entry point's chunk slots (their destructors release their buffers) on the device they ran on.
template <class BufsT>
void free_chunk_bufs(bsw_engine* eng, BufsT*& b)
{
    if (!b) return;
    if (!eng->devs.empty()) cudaSetDevice(eng->devs[0].dev);
    delete b;
    b = nullptr;
}

// Shared-memory words per thread (S).  S >= qlen + 8 (prefetched group, bsw_kernels.cuh), S / 4
// odd (the 128-bit row accesses of a quarter warp then fall into 8 distinct bank groups).  Steps
// of 8 words where occupancy is most sensitive to them, coarser for long queries (one launch per
// step present in a chunk).
inline int stride_for(int qmax, bool fine = false)
{
    const int need = qmax + 8;
    if (need > SHORT_MAX_QLEN + 8) return -1;
    int q;                                        // S / 4
    if (need <= 136 || (fine && need <= 520)) q = (need + 3) / 4;
    else if (need <= 520) q = ((need + 15) & ~15) / 4;
    else q = ((need + 31) & ~31) / 4;
    if (!(q & 1)) ++q;
    return 4 * q;
}

// Block size of the packed kernel for a shared-memory class: a block's footprint (rows + query plane + 2 KB
// score table + 1 KB the SM reserves) only fits the SM's 228 KB a whole number of times, and for some
// classes 32-thread blocks leave less of it unused than 64-thread ones -- one more resident warp where
// there are only four to seven.  BSW_SHORT_BLOCK=64 / 32 in the environment forces one size.
inline int short16_block(int qstride, int plane, bool circ)
{
    static const int forced = getenv("BSW_SHORT_BLOCK") ? atoi(getenv("BSW_SHORT_BLOCK")) : 0;
    if (forced == 32 || forced == 64) return forced;
    const int sm_bytes = 228 * 1024;
    const int rb = circ ? 12 : 14;                    // register limit in blocks of 64: 71 registers, 77 with circular rows
    const int w64 = std::min((int)(sm_bytes / (k16::smem_bytes(64, qstride, plane) + 1024)), rb) * 2;
    const int w32 = std::min((int)(sm_bytes / (k16::smem_bytes(32, qstride, plane) + 1024)), 2 * rb);
    return w32 > w64 ? 32 : 64;
}

// dynamic shared memory of one short-kernel block: eh words + the 2-bit query byte plane
inline size_t short_smem_bytes(int qstride)
{
    return (size_t)qstride * SHORT_BLOCK * sizeof(uint32_t) + (size_t)((qstride + 3) / 4) * SHORT_BLOCK;
}

inline int bits_for(uint32_t range)      // bits needed to hold values 0..range
{
    int b = 0;
    while (range) { ++b; range >>= 1; }
    return b;
}

// May a call of n pairs run its short pairs (queries <= w16::MAX_QLEN) one per warp?  One thread sweeps a 151-bp pair in
// ~0.4 ms whatever the batch, so a call that leaves most schedulers without a warp is bound by that latency; the
// warp-per-pair register kernel (bsw_warp16.cuh) sweeps it in ~0.14 ms, at ~10 x the issue slots per cell.  That pays
// while the GPU has issue slots to spare: measured (profiles/r03c_warp_probe.json, r03d_latency_ab.txt) up to ~4 000
// 151-bp pairs in flight on the device -- one call of that size, or eight of the driver's 512-pair calls; beyond that
// the issue rate bounds them all and the thread-per-pair kernel serves more pairs per second.  So the pairs on the
// warp kernel are a per-device budget (bsw_params.warp_max_pairs; -1: never), shared by every call and engine of
// the process: a call takes its share for as long as it runs, or runs thread-per-pair.
std::atomic<int64_t> g_warp_pairs[64];           // per CUDA device: pairs of running calls that took the warp kernel

struct WarpLease {
    int dev = -1;
    int64_t n = 0;
    WarpLease() = default;
    WarpLease(const WarpLease&) = delete;
    WarpLease& operator=(const WarpLease&) = delete;
    ~WarpLease() { release(); }
    bool acquire(const bsw_engine* eng, int cuda_dev, int64_t pairs, bool use16, int32_t limit_param)
    {
        if (!use16 || limit_param < 0 || pairs <= 0 || cuda_dev < 0 || cuda_dev >= 64) return false;
        if (!w16::scoring_ok(eng->kp)) return false;
        const int64_t limit = limit_param > 0 ? limit_param : WARP_MAX_PAIRS;
        std::atomic<int64_t>& g = g_warp_pairs[cuda_dev];
        int64_t cur = g.load(std::memory_order_relaxed);
        do {
            if (cur + pairs > limit) return false;
        } while (!g.compare_exchange_weak(cur, cur + pairs, std::memory_order_relaxed));
        dev = cuda_dev; n = pairs;
        return true;
    }
    void release()
    {
        if (dev >= 0) g_warp_pairs[dev].fetch_sub(n, std::memory_order_relaxed);
        dev = -1; n = 0;
    }
};

// the static part of the rule, for a batch that stays resident (bsw_stage): no lease is held between its runs
bool warp_fits(const bsw_engine* eng, int64_t n)
{
    if (!eng->use16 || eng->p.warp_max_pairs < 0 || n <= 0 || !w16::scoring_ok(eng->kp)) return false;
    return n <= (eng->p.warp_max_pairs > 0 ? eng->p.warp_max_pairs : WARP_MAX_PAIRS);
}

int set_kernel_attrs(bsw_engine* eng, DevCtx& c)
{
    if (c.attr_set) return BSW_OK;
    const int maxsm = 227 * 1024;
    CUDA_TRY(cudaFuncSetAttribute(bsw_short_kernel<SHORT_BLOCK, false>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    CUDA_TRY(cudaFuncSetAttribute(bsw_short_kernel<SHORT_BLOCK, true>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    CUDA_TRY(cudaFuncSetAttribute(bsw_short16_kernel<64, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    CUDA_TRY(cudaFuncSetAttribute(bsw_short16_kernel<64, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    CUDA_TRY(cudaFuncSetAttribute(bsw_short16_kernel<32, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    CUDA_TRY(cudaFuncSetAttribute(bsw_short16_kernel<32, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    CUDA_TRY(cudaFuncSetAttribute(bsw_short16_kernel<64, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    CUDA_TRY(cudaFuncSetAttribute(bsw_short16_kernel<64, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    CUDA_TRY(cudaFuncSetAttribute(bsw_short16_kernel<32, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    CUDA_TRY(cudaFuncSetAttribute(bsw_short16_kernel<32, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, maxsm));
    c.attr_set = true;
    return BSW_OK;
}

// Splits the device into a service partition and a DP partition (see GreenApi).  Best effort: on
// any failure the device simply runs unpartitioned.  BSW_SERVICE_SMS overrides the service size
// (0 disables the split).
void setup_partitions(DevCtx& c)
{
    const GreenApi& G = green_api();
    int want = 32;
    if (const char* e = getenv("BSW_SERVICE_SMS")) want = atoi(e);
    if (!G.ok || want <= 0 || want * 2 > c.sms) return;
    cudaFree(0);                                            // the primary context must exist
    CUdevResource all{}, svc{}, rest{};
    if (G.get_res((CUdevice)c.dev, &all, CU_DEV_RESOURCE_TYPE_SM) != CUDA_SUCCESS) return;
    unsigned nb = 1;
    if (G.split(&svc, &nb, &all, &rest, 0, (unsigned)want) != CUDA_SUCCESS || nb != 1 || rest.sm.smCount == 0) return;
    CUdevResourceDesc d_svc{}, d_rest{};
    if (G.gen_desc(&d_svc, &svc, 1) != CUDA_SUCCESS || G.gen_desc(&d_rest, &rest, 1) != CUDA_SUCCESS) return;
    CUgreenCtx g_svc = nullptr, g_dp = nullptr;
    if (G.create(&g_svc, d_svc, (CUdevice)c.dev, CU_GREEN_CTX_DEFAULT_STREAM) != CUDA_SUCCESS) return;
    if (G.create(&g_dp, d_rest, (CUdevice)c.dev, CU_GREEN_CTX_DEFAULT_STREAM) != CUDA_SUCCESS) { G.destroy(g_svc); return; }
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    for (int k = 0; k < NSTREAMS; ++k) {
        CUstream cu = nullptr;
        if (G.stream_create(&cu, g_dp, CU_STREAM_NON_BLOCKING, prio_lo) != CUDA_SUCCESS) {
            for (int j = 0; j < k; ++j) { cudaStreamDestroy(c.cs_part[j]); c.cs_part[j] = nullptr; }
            G.destroy(g_svc); G.destroy(g_dp);
            return;
        }
        c.cs_part[k] = (cudaStream_t)cu;
    }
    c.g_svc = g_svc; c.g_dp = g_dp;
    c.svc_sms = (int)svc.sm.smCount; c.dp_sms = (int)rest.sm.smCount;
}

int validate_params(const bsw_params* p, std::string& why)
{
    auto bad = [&](const char* m) { why = m; return BSW_ERR_PARAM; };
    if (p->e_del < 1 || p->e_ins < 1) return bad("e_del / e_ins must be >= 1");
    if (p->o_del < 0 || p->o_ins < 0) return bad("o_del / o_ins must be >= 0");
    if (p->o_del + p->e_del > 16000 || p->o_ins + p->e_ins > 16000) return bad("gap penalties too large");
    if (p->match < 1 || p->match > 127) return bad("match must be in 1..127");
    if (p->mismatch < 0 || p->mismatch > 127) return bad("mismatch penalty must be in 0..127");
    if (p->ambig > p->match || p->ambig < -127) return bad("ambig must be in -127..match");
    if (p->zdrop_mode == BSW_ZDROP_VECTOR && (p->zdrop < 1 || p->zdrop > 32767))
        return bad("zdrop must be in 1..32767 (32767 = off); the reference's vector z-drop is not 'off' for <= 0");
    if (p->zdrop_mode != BSW_ZDROP_VECTOR && p->zdrop_mode != BSW_ZDROP_SCALAR) return bad("zdrop_mode");
    if (p->zdrop > 32767) return bad("zdrop must be <= 32767");
    if (p->end_bonus < 0 || p->end_bonus > 16000) return bad("end_bonus out of range");
    if (p->n_devices < 0 || p->n_devices > 16) return bad("n_devices must be in 0..16");
    if (p->long_min_qlen < 0) return bad("long_min_qlen must be >= 0");
    if (p->short_variant != BSW_SHORT_PACKED16 && p->short_variant != BSW_SHORT_WIDE32) return bad("short_variant");
    if (p->tiny_batch < 0) return bad("tiny_batch must be >= 0");
    if (p->warp_max_pairs < -1) return bad("warp_max_pairs must be >= -1");
    return BSW_OK;
}

void init_info(ChunkInfo& I)
{
    memset(&I, 0, sizeof(I));
    I.min_r = I.min_q = ~0ull;
    I.mn[0] = I.mn[1] = I.mn[2] = INT_MAX;
}

// true when the pointer is pinned / registered host memory the device can DMA and map
bool is_pinned(const void* p)
{
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

int slot_create(bsw_engine* eng, DevCtx& c, Slot& s)
{
    // The chunk streams (copies, prep kernels, write-back) outrank the DP streams: a DP launch
    // queues thousands of blocks, and at equal priority the small kernels of the NEXT chunks would
    // wait behind that backlog, starving the copy engine of work (seen in the BSW_TIMELINE trace).
    int prio_lo = 0, prio_hi = 0;
    CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    CUDA_TRY(cudaStreamCreateWithPriority(&s.st_plain, cudaStreamNonBlocking, prio_hi));
    if (c.svc_sms > 0) {
        CUstream cu = nullptr;
        if (green_api().stream_create(&cu, c.g_svc, CU_STREAM_NON_BLOCKING, prio_hi) != CUDA_SUCCESS) {
            err_of(eng) = "cuGreenCtxStreamCreate failed";
            return BSW_ERR_CUDA;
        }
        s.st_svc = (cudaStream_t)cu;
    }
    s.st = s.st_plain;
    for (cudaEvent_t* e : {&s.ev_info, &s.ev_dp, &s.ev_out, &s.ev_fork, &s.ev_seq, &s.ev_lists, &s.ev_rec, &s.ev_seqd})
        CUDA_TRY(cudaEventCreateWithFlags(e, g_timeline ? cudaEventDefault : cudaEventDisableTiming));
    if (g_timeline) for (cudaEvent_t& e : s.ev_tl) CUDA_TRY(cudaEventCreate(&e));
    CUDA_TRY(cudaEventCreate(&s.ev_k0));
    CUDA_TRY(cudaEventCreate(&s.ev_k1));
    CUDA_TRY(cudaMalloc((void**)&s.d_info, sizeof(ChunkInfo)));
    CUDA_TRY(cudaHostAlloc((void**)&s.h_info, sizeof(ChunkInfo), cudaHostAllocMapped));
    CUDA_TRY(cudaHostGetDevicePointer((void**)&s.h_info_dev, s.h_info, 0));
    CUDA_TRY(cudaMalloc((void**)&s.d_queue, sizeof(unsigned int)));
    return BSW_OK;
}

void slot_destroy(Slot& s)
{
    if (s.st_plain) cudaStreamDestroy(s.st_plain);
    if (s.st_svc) cudaStreamDestroy(s.st_svc);
    for (cudaEvent_t e : {s.ev_info, s.ev_dp, s.ev_out, s.ev_fork, s.ev_k0, s.ev_k1, s.ev_seq, s.ev_lists, s.ev_rec, s.ev_seqd})
        if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s.ev_tl) if (e) cudaEventDestroy(e);
    release(s.raw_pairs); release(s.desc); release(s.meta); release(s.res); release(s.perm); release(s.rank);
    release(s.bins); release(s.nlist); release(s.llist); release(s.qpk); release(s.tpk); release(s.scratch);
    release(s.qraw); release(s.rraw); release(s.outbuf); release(s.rawq); release(s.rawr); release(s.tinybuf);
    if (s.d_info) cudaFree(s.d_info);
    if (s.h_info) cudaFreeHost(s.h_info);
    if (s.d_queue) cudaFree(s.d_queue);
}

int get_slot(bsw_engine* eng, DevCtx& c, int k, Slot** out)
{
    while ((int)c.slots.size() <= k) {
        c.slots.emplace_back();
        if (int rc = slot_create(eng, c, c.slots.back())) return rc;
    }
    *out = &c.slots[(size_t)k];
    return BSW_OK;
}

inline int grid_for(const DevCtx& c, int n, int per_block)
{
    return std::max(1, std::min((n + per_block - 1) / per_block, c.sms * 32));
}

// ------------------------------------------------------------------------------------------
// stage A, direct route: records DMA + scan; the summary comes back through ev_info
// ------------------------------------------------------------------------------------------
int direct_begin(bsw_engine* eng, DevCtx& c, Slot& s, const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer)
{
    const size_t bytes = (size_t)s.n * sizeof(SeqPair);
    if (int rc = ensure(eng, s.raw_pairs, bytes)) return rc;
    if (int rc = ensure(eng, s.desc, (size_t)s.n)) return rc;
    // Host-to-device copies of all chunks go through ONE stream, in chunk order: copies issued on
    // several streams share the link, so with the next chunks' copies already queued every chunk
    // would arrive late; in FIFO order chunk k is complete before chunk k + 1 takes bandwidth.
    if (int rc = ensure(eng, s.bins, BINS_WORDS)) return rc;
    bsw_info_init<<<1, PREP_BLOCK, 0, s.st>>>(s.d_info);
    bsw_zero_words<<<64, PREP_BLOCK, 0, s.st>>>(reinterpret_cast<uint4*>(s.bins.d), (int)(BINS_WORDS / 4));
    s.bins_zeroed = true;
    CUDA_TRY(cudaMemcpyAsync(s.raw_pairs.d, pairs + s.a, bytes, cudaMemcpyHostToDevice, c.h2d));
    CUDA_TRY(cudaEventRecord(s.ev_rec, c.h2d));
    CUDA_TRY(cudaStreamWaitEvent(s.st, s.ev_rec, 0));
    const long long base0_r = pairs[s.a].idr, base0_q = pairs[s.a].idq;     // one record read by the host
    bsw_scan_pairs<<<grid_for(c, s.n, 8 * PREP_BLOCK), PREP_BLOCK, 0, s.st>>>(
        reinterpret_cast<const SeqPair*>(s.raw_pairs.d), s.n, base0_r, base0_q, eng->p.match, eng->short_max,
        s.desc.d, s.d_info);
    bsw_info_publish<<<1, PREP_BLOCK, 0, s.st>>>(s.d_info, s.h_info_dev);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(s.ev_info, s.st));
    stats_of(eng).h2d_bytes += (int64_t)bytes;
    stats_of(eng).kernel_launches += 4;

    // Speculative sequence copy.  The byte range the chunk's sequences span is only known after the
    // scan, and waiting for it would leave the copy engine idle for a host round trip per chunk.
    // Batches are normally laid out in record order (the reference loader, main_banded.cpp:131-185,
    // appends sequence after sequence), so the range from the first record's offset to the last
    // record's end is copied right away; direct_sequences() checks the scanned range against it and
    // copies again in the rare case the guess does not cover it.
    const SeqPair& f = pairs[s.a];
    const SeqPair& l = pairs[s.a + s.n - 1];
    double est_q = 0, est_r = 0;                                            // bases per pair, sampled
    const int step = std::max(1, s.n / 61);
    int ns = 0;
    for (int i = 0; i < s.n; i += step, ++ns) { est_q += pairs[s.a + i].len2; est_r += pairs[s.a + i].len1; }
    est_q = est_q / ns * s.n; est_r = est_r / ns * s.n;
    struct Side { const uint8_t* host; long long lo, hi; double est; Buf<uint8_t>* buf; };
    Side sides[2] = {{seq_qer, std::min(f.idq, l.idq), std::max(f.idq + f.len2, l.idq + l.len2), est_q, &s.qraw},
                     {seq_ref, std::min(f.idr, l.idr), std::max(f.idr + f.len1, l.idr + l.len1), est_r, &s.rraw}};
    for (int k = 0; k < 2; ++k) {
        Side& sd = sides[k];
        s.spec[k] = false;
        if (sd.lo < 0 || sd.hi <= sd.lo || f.len1 < 1 || f.len2 < 1 || l.len1 < 1 || l.len2 < 1 ||
            f.len1 > 32767 || f.len2 > 32767 || l.len1 > 32767 || l.len2 > 32767) continue;     // out of domain: the scan reports it
        const long long lo_al = sd.lo & ~15ll;                              // keep the source's 16-byte phase
        const double span = (double)(sd.hi - lo_al);
        if (span > 2.0 * sd.est + (double)(1 << 20) || span > 3.0e9) continue;   // sparse (or not in record order): wait for the scan
        if (int rc = ensure(eng, *sd.buf, (size_t)(sd.hi - lo_al) + 64)) return rc;
        CUDA_TRY(cudaMemcpyAsync(sd.buf->d, sd.host + lo_al, (size_t)(sd.hi - lo_al), cudaMemcpyHostToDevice, c.h2d));
        s.spec[k] = true; s.spec_lo[k] = lo_al; s.spec_hi[k] = sd.hi;
        stats_of(eng).h2d_bytes += sd.hi - lo_al;
    }
    CUDA_TRY(cudaEventRecord(s.ev_seqd, c.h2d));
    return BSW_OK;
}

// stage B, direct route: sequences on the device -- the speculative copy when it covers the scanned
// range, else a DMA of that range (dense) or mapped reads (sparse)
int direct_sequences(bsw_engine* eng, Slot& s, const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer)
{
    CUDA_TRY(cudaEventSynchronize(s.ev_info));
    s.info = *s.h_info;
    if (s.info.bad) return BSW_ERR_DOMAIN;
    if (s.info.far) return BSW_RETRY_STAGED;
    const long long base0_r = pairs[s.a].idr, base0_q = pairs[s.a].idq;
    struct Side { const uint8_t* host; long long base0; unsigned long long mn, mx, bases; Buf<uint8_t>* buf; const uint8_t** out; };
    Side sides[2] = {{seq_qer, base0_q, s.info.min_q, s.info.max_q, s.info.qbases, &s.qraw, &s.qbase},
                     {seq_ref, base0_r, s.info.min_r, s.info.max_r, s.info.tbases, &s.rraw, &s.rbase}};
    s.seq_on_device = true;
    for (int k = 0; k < 2; ++k) {
        Side& sd = sides[k];
        const long long lo = sd.base0 + ((long long)sd.mn - OFF_BIAS);       // absolute byte offsets [lo, hi)
        const long long hi = sd.base0 + ((long long)sd.mx - OFF_BIAS);
        if (s.spec[k] && lo >= s.spec_lo[k] && hi <= s.spec_hi[k]) {
            *sd.out = sd.buf->d + (sd.base0 - s.spec_lo[k]);
            continue;
        }
        const unsigned long long span = (unsigned long long)(hi - lo);
        const bool dense = span <= 2 * sd.bases + (1ull << 20);
        if (dense) {
            const long long lo_al = lo & ~15ll;                             // keep the source's 16-byte phase
            const size_t bytes = (size_t)(hi - lo_al);
            if (int rc = ensure(eng, *sd.buf, bytes + 64)) return rc;
            CUDA_TRY(cudaMemcpyAsync(sd.buf->d, sd.host + lo_al, bytes, cudaMemcpyHostToDevice, s.st));
            *sd.out = sd.buf->d + (sd.base0 - lo_al);
            stats_of(eng).h2d_bytes += (int64_t)bytes;
        } else {
            void* dp = nullptr;
            CUDA_TRY(cudaHostGetDevicePointer(&dp, const_cast<uint8_t*>(sd.host), 0));
            *sd.out = static_cast<const uint8_t*>(dp) + sd.base0;
            s.seq_on_device = false;                                        // host memory read in place: it may end with the last base
            stats_of(eng).h2d_bytes += (int64_t)sd.bases;
        }
    }
    // (the chunk stream never overtakes its own speculative copies, used or not: the buffers are its own)
    CUDA_TRY(cudaStreamWaitEvent(s.st, s.ev_seqd, 0));
    if (g_timeline) CUDA_TRY(cudaEventRecord(s.ev_seq, s.st));
    return BSW_OK;
}

// ------------------------------------------------------------------------------------------
// stage A, packed route: descriptors + the chunk's 2-bit words DMA'd as the loader packed them, scan
// ------------------------------------------------------------------------------------------
inline unsigned int words_of(int len) { return (unsigned int)(len + 15) >> 4; }

// buffers of a packed batch that every chunk of the call addresses absolutely: the RAW sequences, and all 2-bit
// words when the batch does not promise ascending offsets
int packed_resident(bsw_engine* eng, DevCtx& c, const bsw_packed_batch& B)
{
    CUDA_TRY(cudaSetDevice(c.dev));
    if (B.raw_q_bytes > 0 || B.raw_r_bytes > 0) {
        if (int rc = ensure(eng, c.rawq, (size_t)B.raw_q_bytes + 64)) return rc;
        if (int rc = ensure(eng, c.rawr, (size_t)B.raw_r_bytes + 64)) return rc;
        CUDA_TRY(cudaMemcpyAsync(c.rawq.d, B.raw_q, (size_t)B.raw_q_bytes, cudaMemcpyHostToDevice, c.h2d));
        CUDA_TRY(cudaMemcpyAsync(c.rawr.d, B.raw_r, (size_t)B.raw_r_bytes, cudaMemcpyHostToDevice, c.h2d));
        stats_of(eng).h2d_bytes += B.raw_q_bytes + B.raw_r_bytes;
    }
    if (!B.ordered) {
        if (int rc = ensure(eng, c.allq, (size_t)B.q2_words * 4 + 64)) return rc;
        if (int rc = ensure(eng, c.allr, (size_t)B.r2_words * 4 + 64)) return rc;
        CUDA_TRY(cudaMemcpyAsync(c.allq.d, B.q2, (size_t)B.q2_words * 4, cudaMemcpyHostToDevice, c.h2d));
        CUDA_TRY(cudaMemcpyAsync(c.allr.d, B.r2, (size_t)B.r2_words * 4, cudaMemcpyHostToDevice, c.h2d));
        stats_of(eng).h2d_bytes += (B.q2_words + B.r2_words) * 4;
    }
    CUDA_TRY(cudaEventRecord(c.ev_res, c.h2d));
    return BSW_OK;
}

int packed_begin(bsw_engine* eng, DevCtx& c, Slot& s, const bsw_packed_batch& B)
{
    const bsw_pair_desc* D = B.desc + s.a;
    if (int rc = ensure(eng, s.desc, (size_t)s.n)) return rc;
    if (int rc = ensure(eng, s.bins, BINS_WORDS)) return rc;
    bsw_info_init<<<1, PREP_BLOCK, 0, s.st>>>(s.d_info);
    bsw_zero_words<<<64, PREP_BLOCK, 0, s.st>>>(reinterpret_cast<uint4*>(s.bins.d), (int)(BINS_WORDS / 4));
    s.bins_zeroed = true;
    CUDA_TRY(cudaMemcpyAsync(s.desc.d, D, sizeof(bsw_pair_desc) * (size_t)s.n, cudaMemcpyHostToDevice, c.h2d));
    CUDA_TRY(cudaEventRecord(s.ev_rec, c.h2d));
    CUDA_TRY(cudaStreamWaitEvent(s.st, s.ev_rec, 0));
    stats_of(eng).h2d_bytes += (int64_t)sizeof(bsw_pair_desc) * s.n;
    PackedRange R{};
    R.rawq = (unsigned int)B.raw_q_bytes; R.rawr = (unsigned int)B.raw_r_bytes;
    if (!B.ordered) {
        R.qlo = 0; R.qhi = (unsigned int)B.q2_words; R.rlo = 0; R.rhi = (unsigned int)B.r2_words;
        s.q2src = c.allq.d; s.r2src = c.allr.d;
    } else {
        // ascending offsets: the chunk's words are the range from its first to its last 2-bit pair
        int f = 0, l = s.n - 1;
        while (f < s.n && (D[f].flags & BSW_PAIR_RAW)) ++f;
        while (l > f && (D[l].flags & BSW_PAIR_RAW)) --l;
        if (f < s.n) {
            R.qlo = D[f].q_off; R.qhi = D[l].q_off + words_of(D[l].len2);
            R.rlo = D[f].r_off; R.rhi = D[l].r_off + words_of(D[l].len1);
            if (R.qhi < R.qlo || R.rhi < R.rlo || (int64_t)R.qhi > B.q2_words || (int64_t)R.rhi > B.r2_words) {
                err_of(eng) = "bsw_extend_packed: batch.ordered is set but the offsets do not ascend inside the buffers";
                return BSW_ERR_PARAM;
            }
        }
        const size_t qb = (size_t)(R.qhi - R.qlo) * 4, rb = (size_t)(R.rhi - R.rlo) * 4;
        if (int rc = ensure(eng, s.qraw, qb + 64)) return rc;
        if (int rc = ensure(eng, s.rraw, rb + 64)) return rc;
        if (qb) CUDA_TRY(cudaMemcpyAsync(s.qraw.d, B.q2 + R.qlo, qb, cudaMemcpyHostToDevice, c.h2d));
        if (rb) CUDA_TRY(cudaMemcpyAsync(s.rraw.d, B.r2 + R.rlo, rb, cudaMemcpyHostToDevice, c.h2d));
        s.q2src = s.qraw.d; s.r2src = s.rraw.d;
        stats_of(eng).h2d_bytes += (int64_t)(qb + rb);
    }
    s.q_lo = R.qlo; s.r_lo = R.rlo;
    CUDA_TRY(cudaEventRecord(s.ev_seqd, c.h2d));
    bsw_scan_packed<<<grid_for(c, s.n, 8 * PREP_BLOCK), PREP_BLOCK, 0, s.st>>>(s.desc.d, s.n, R, eng->p.match, eng->short_max,
                                                                               eng->use16 ? 1 : 0, s.d_info);
    bsw_info_publish<<<1, PREP_BLOCK, 0, s.st>>>(s.d_info, s.h_info_dev);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(s.ev_info, s.st));
    stats_of(eng).kernel_launches += 4;
    return BSW_OK;
}

// stage B, packed route: the summary is on the host; the byte kernels read the resident RAW sequences
int packed_info(bsw_engine* eng, DevCtx& c, Slot& s)
{
    CUDA_TRY(cudaEventSynchronize(s.ev_info));
    s.info = *s.h_info;
    if (s.info.bad) return BSW_ERR_DOMAIN;
    s.qbase = c.rawq.d; s.rbase = c.rawr.d;
    s.seq_on_device = true;
    CUDA_TRY(cudaStreamWaitEvent(s.st, s.ev_seqd, 0));
    CUDA_TRY(cudaStreamWaitEvent(s.st, c.ev_res, 0));
    if (g_timeline) CUDA_TRY(cudaEventRecord(s.ev_seq, s.st));
    return BSW_OK;
}

// ------------------------------------------------------------------------------------------
// stage A+B, staged route: one streaming host pass builds descriptors + gathers the bytes
// ------------------------------------------------------------------------------------------
int staged_prepare_bytes(bsw_engine* eng, Slot& s, const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer);

// Pageable host buffers: the one streaming pass over the caller's memory packs the sequences to 2 bits per base on
// the way into page-locked staging (the host-side packer of the packed route, bsw_common.h), so the chunk crosses PCIe
// at ~46 B per short pair instead of 138 and the device needs no pack kernel: it is handed to the 2-bit source path
// of the packed route (descriptors with word offsets, DP kernels read the words in place).  Pairs that contain N, and
// queries for the warp-per-pair kernel, keep one byte per base (RAW) in a side buffer.  The latency route (tiny: every
// pair on the byte-reading warp-per-pair kernel) keeps the byte form of the pass.
int staged_prepare(bsw_engine* eng, Slot& s, const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer)
{
    static const bool bytes_only = getenv("BSW_STAGED_BYTES") && atoi(getenv("BSW_STAGED_BYTES")) != 0;   // A/B: round-1 form
    if (s.tiny || bytes_only) return staged_prepare_bytes(eng, s, pairs, seq_ref, seq_qer);
    const double t0 = now_ms();
    const SeqPair* P = pairs + s.a;
    const int n = s.n;
    const int match = eng->p.match, short_max = eng->short_max;
    const bool use16 = eng->use16;
    const int BLK = std::max(256, std::min(4096, n / (2 * eng->pool->size())));
    const int nblk = (n + BLK - 1) / BLK;
    struct Sum { uint64_t qw = 0, rw = 0, rq = 0, rr = 0; };       // 2-bit words; RAW bytes of the long queries
    std::vector<Sum> sums((size_t)nblk + 1);
    std::vector<ChunkInfo> part((size_t)eng->pool->size());
    for (ChunkInfo& I : part) init_info(I);
    // pass 1 (records only): validate, summary, word / byte totals per block
    eng->pool->run(nblk, [&](int64_t b, int t) {
        ChunkInfo& I = part[(size_t)t];
        Sum sm;
        const int lo = (int)b * BLK, hi = std::min(n, lo + BLK);
        for (int k = lo; k < hi; ++k) {
            const SeqPair& sp = P[k];
            if (sp.len1 < 1 || sp.len1 > 32767 || sp.len2 < 1 || sp.len2 > 32767 || sp.h0 < 0 ||
                (int64_t)sp.h0 + (int64_t)sp.len2 * match > 32767 || sp.idr < 0 || sp.idq < 0) { I.bad++; continue; }
            I.nominal += (unsigned long long)sp.len1 * (unsigned long long)sp.len2;
            I.hist[std::min(sp.len2, LEN_HIST - 1)]++;
            I.qmax_all = std::max(I.qmax_all, sp.len2);
            if (sp.len2 <= short_max) {
                sm.qw += (uint64_t)((sp.len2 + 15) >> 4); sm.rw += (uint64_t)((sp.len1 + 15) >> 4);
                I.n_short++;
                I.mn[0] = std::min(I.mn[0], sp.len2); I.mx[0] = std::max(I.mx[0], sp.len2);
                I.mn[1] = std::min(I.mn[1], sp.h0);   I.mx[1] = std::max(I.mx[1], sp.h0);
                I.mn[2] = std::min(I.mn[2], sp.len1); I.mx[2] = std::max(I.mx[2], sp.len1);
                if (use16 && !k16::eligible(match, sp.len2, sp.h0)) I.n_wide++;
            } else {
                sm.rq += (uint64_t)sp.len2; sm.rr += (uint64_t)sp.len1;
            }
        }
        sums[(size_t)b + 1] = sm;
    });
    ChunkInfo& I = s.info;
    init_info(I);
    for (const ChunkInfo& p : part) {
        I.bad += p.bad; I.nominal += p.nominal; I.n_short += p.n_short; I.n_wide += p.n_wide;
        I.qmax_all = std::max(I.qmax_all, p.qmax_all);
        for (int f = 0; f < 3; ++f) { I.mn[f] = std::min(I.mn[f], p.mn[f]); I.mx[f] = std::max(I.mx[f], p.mx[f]); }
        for (int k = 0; k < LEN_HIST; ++k) I.hist[k] += p.hist[k];
    }
    if (I.bad) return BSW_ERR_DOMAIN;
    for (int b = 0; b < nblk; ++b) {
        sums[(size_t)b + 1].qw += sums[(size_t)b].qw; sums[(size_t)b + 1].rw += sums[(size_t)b].rw;
        sums[(size_t)b + 1].rq += sums[(size_t)b].rq; sums[(size_t)b + 1].rr += sums[(size_t)b].rr;
    }
    const Sum tot = sums[(size_t)nblk];
    I.qbases = tot.qw * 16; I.tbases = tot.rw * 16;              // (they size the word arrays of device_prepare)
    if (tot.qw > 0x3fffffffull || tot.rw > 0x3fffffffull || tot.rq > 0x3fffffffull || tot.rr > 0x3fffffffull) {
        err_of(eng) = "chunk too large for 32-bit offsets";
        return BSW_ERR_PARAM;
    }
    if (int rc = ensure(eng, s.desc, (size_t)n, true)) return rc;
    if (int rc = ensure(eng, s.qraw, (size_t)tot.qw * 4 + 64, true)) return rc;
    if (int rc = ensure(eng, s.rraw, (size_t)tot.rw * 4 + 64, true)) return rc;
    uint32_t* const q2 = reinterpret_cast<uint32_t*>(s.qraw.h);
    uint32_t* const r2 = reinterpret_cast<uint32_t*>(s.rraw.h);
    // pass 2 (sequences, read once): pack, descriptors; pairs with N are remembered
    std::vector<std::vector<int>> with_n((size_t)eng->pool->size());
    eng->pool->run(nblk, [&](int64_t b, int t) {
        Sum o = sums[(size_t)b];
        const int lo = (int)b * BLK, hi = std::min(n, lo + BLK);
        for (int k = lo; k < hi; ++k) {
            const SeqPair& sp = P[k];
            if (k + 4 < hi) {
                __builtin_prefetch(seq_qer + P[k + 4].idq, 0, 0);
                __builtin_prefetch(seq_ref + P[k + 4].idr, 0, 0);
                __builtin_prefetch(seq_ref + P[k + 4].idr + 64, 0, 0);
            }
            if (sp.len2 <= short_max) {
                const bool nq = pack_seq(seq_qer + sp.idq, sp.len2, q2 + o.qw);
                const bool nr = pack_seq(seq_ref + sp.idr, sp.len1, r2 + o.rw);
                s.desc.h[k] = make_int4((int)o.qw, (int)o.rw, sp.len2 | (sp.len1 << 16), sp.h0);
                if (nq || nr) with_n[(size_t)t].push_back(k);
                o.qw += (uint64_t)((sp.len2 + 15) >> 4); o.rw += (uint64_t)((sp.len1 + 15) >> 4);
            } else {
                s.desc.h[k] = make_int4((int)o.rq, (int)o.rr, sp.len2 | (sp.len1 << 16), sp.h0 | (BSW_PAIR_RAW << 16));
                o.rq += (uint64_t)sp.len2; o.rr += (uint64_t)sp.len1;
            }
        }
    });
    // RAW side buffer: the long queries (offsets from pass 1), then the pairs with N
    uint64_t rq = tot.rq, rr = tot.rr;
    for (const std::vector<int>& v : with_n) for (int k : v) { rq += (uint64_t)P[k].len2; rr += (uint64_t)P[k].len1; }
    if (rq > 0x3fffffffull || rr > 0x3fffffffull) { err_of(eng) = "chunk too large for 32-bit offsets"; return BSW_ERR_PARAM; }
    if (int rc = ensure(eng, s.rawq, (size_t)rq + 64, true)) return rc;
    if (int rc = ensure(eng, s.rawr, (size_t)rr + 64, true)) return rc;
    if (tot.rq > 0)
        eng->pool->run(nblk, [&](int64_t b, int) {
            const int lo = (int)b * BLK, hi = std::min(n, lo + BLK);
            for (int k = lo; k < hi; ++k) {
                const SeqPair& sp = P[k];
                if (sp.len2 <= short_max) continue;
                memcpy(s.rawq.h + s.desc.h[k].x, seq_qer + sp.idq, (size_t)sp.len2);
                memcpy(s.rawr.h + s.desc.h[k].y, seq_ref + sp.idr, (size_t)sp.len1);
            }
        });
    {
        uint64_t oq = tot.rq, orr = tot.rr;
        for (const std::vector<int>& v : with_n)
            for (int k : v) {
                const SeqPair& sp = P[k];
                memcpy(s.rawq.h + oq, seq_qer + sp.idq, (size_t)sp.len2);
                memcpy(s.rawr.h + orr, seq_ref + sp.idr, (size_t)sp.len1);
                s.desc.h[k] = make_int4((int)oq, (int)orr, sp.len2 | (sp.len1 << 16), sp.h0 | (BSW_PAIR_RAW << 16));
                oq += (uint64_t)sp.len2; orr += (uint64_t)sp.len1;
            }
    }
    memset(s.rawq.h + rq, 0, 64); memset(s.rawr.h + rr, 0, 64);
    stats_of(eng).ms_pack += now_ms() - t0;
    // H2D
    bsw_info_init<<<1, PREP_BLOCK, 0, s.st>>>(s.d_info);
    stats_of(eng).kernel_launches++;
    CUDA_TRY(cudaMemcpyAsync(s.desc.d, s.desc.h, sizeof(int4) * (size_t)n, cudaMemcpyHostToDevice, s.st));
    if (tot.qw) CUDA_TRY(cudaMemcpyAsync(s.qraw.d, s.qraw.h, (size_t)tot.qw * 4, cudaMemcpyHostToDevice, s.st));
    if (tot.rw) CUDA_TRY(cudaMemcpyAsync(s.rraw.d, s.rraw.h, (size_t)tot.rw * 4, cudaMemcpyHostToDevice, s.st));
    if (rq + rr > 0) {
        CUDA_TRY(cudaMemcpyAsync(s.rawq.d, s.rawq.h, (size_t)rq + 64, cudaMemcpyHostToDevice, s.st));
        CUDA_TRY(cudaMemcpyAsync(s.rawr.d, s.rawr.h, (size_t)rr + 64, cudaMemcpyHostToDevice, s.st));
    }
    s.src2bit = true;
    s.q2src = s.qraw.d; s.r2src = s.rraw.d; s.q_lo = 0; s.r_lo = 0;
    s.qbase = s.rawq.d; s.rbase = s.rawr.d;
    s.seq_on_device = true;
    stats_of(eng).h2d_bytes += (int64_t)(sizeof(int4) * (size_t)n + (tot.qw + tot.rw) * 4 + (rq + rr ? rq + rr + 128 : 0));
    return BSW_OK;
}

// the byte form of the pass (latency route): descriptors + the sequences' bytes gathered into pinned staging
int staged_prepare_bytes(bsw_engine* eng, Slot& s, const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer)
{
    const double t0 = now_ms();
    const SeqPair* P = pairs + s.a;
    const int n = s.n;
    const int match = eng->p.match, short_max = eng->short_max;
    // pass 1: validate + byte totals per block of pairs (4096, fewer for small chunks so that every pool thread gets
    // a share: a 4096-pair call spent 0.18 of its 0.76 ms in a single-threaded gather)
    const int BLK = std::max(256, std::min(4096, n / (2 * eng->pool->size())));
    const int nblk = (n + BLK - 1) / BLK;
    std::vector<uint64_t> qsum((size_t)nblk + 1, 0), rsum((size_t)nblk + 1, 0);
    std::vector<ChunkInfo> part((size_t)eng->pool->size());
    for (ChunkInfo& I : part) init_info(I);
    eng->pool->run(nblk, [&](int64_t b, int t) {
        ChunkInfo& I = part[(size_t)t];
        uint64_t q = 0, r = 0;
        const int lo = (int)b * BLK, hi = std::min(n, lo + BLK);
        for (int k = lo; k < hi; ++k) {
            const SeqPair& sp = P[k];
            if (sp.len1 < 1 || sp.len1 > 32767 || sp.len2 < 1 || sp.len2 > 32767 || sp.h0 < 0 ||
                (int64_t)sp.h0 + (int64_t)sp.len2 * match > 32767 || sp.idr < 0 || sp.idq < 0) { I.bad++; continue; }
            q += (uint64_t)sp.len2; r += (uint64_t)sp.len1;
            I.nominal += (unsigned long long)sp.len1 * (unsigned long long)sp.len2;
            I.hist[std::min(sp.len2, LEN_HIST - 1)]++;
            I.qmax_all = std::max(I.qmax_all, sp.len2);
            I.qbases += (unsigned long long)sp.len2; I.tbases += (unsigned long long)sp.len1;
            if (sp.len2 <= short_max) {
                I.n_short++;
                I.mn[0] = std::min(I.mn[0], sp.len2); I.mx[0] = std::max(I.mx[0], sp.len2);
                I.mn[1] = std::min(I.mn[1], sp.h0);   I.mx[1] = std::max(I.mx[1], sp.h0);
                I.mn[2] = std::min(I.mn[2], sp.len1); I.mx[2] = std::max(I.mx[2], sp.len1);
            }
        }
        qsum[(size_t)b + 1] = q; rsum[(size_t)b + 1] = r;
    });
    ChunkInfo& I = s.info;
    init_info(I);
    for (const ChunkInfo& p : part) {
        I.bad += p.bad; I.nominal += p.nominal; I.n_short += p.n_short; I.qbases += p.qbases; I.tbases += p.tbases;
        I.qmax_all = std::max(I.qmax_all, p.qmax_all);
        for (int f = 0; f < 3; ++f) { I.mn[f] = std::min(I.mn[f], p.mn[f]); I.mx[f] = std::max(I.mx[f], p.mx[f]); }
        for (int k = 0; k < LEN_HIST; ++k) I.hist[k] += p.hist[k];
    }
    if (I.bad) return BSW_ERR_DOMAIN;
    for (int b = 0; b < nblk; ++b) { qsum[(size_t)b + 1] += qsum[(size_t)b]; rsum[(size_t)b + 1] += rsum[(size_t)b]; }
    const uint64_t qtot = qsum[(size_t)nblk], rtot = rsum[(size_t)nblk];
    if (qtot > 0x3fffffffull || rtot > 0x3fffffffull) { err_of(eng) = "chunk too large for 32-bit byte offsets"; return BSW_ERR_PARAM; }
    if (int rc = ensure(eng, s.desc, (size_t)n, true)) return rc;
    if (int rc = ensure(eng, s.qraw, (size_t)qtot + 64, true)) return rc;
    if (int rc = ensure(eng, s.rraw, (size_t)rtot + 64, true)) return rc;
    // pass 2: gather the bytes, write descriptors (offsets into the staging buffers)
    eng->pool->run(nblk, [&](int64_t b, int) {
        uint64_t q = qsum[(size_t)b], r = rsum[(size_t)b];
        const int lo = (int)b * BLK, hi = std::min(n, lo + BLK);
        for (int k = lo; k < hi; ++k) {
            const SeqPair& sp = P[k];
            if (k + 4 < hi) {
                __builtin_prefetch(seq_qer + P[k + 4].idq, 0, 0);
                __builtin_prefetch(seq_ref + P[k + 4].idr, 0, 0);
                __builtin_prefetch(seq_ref + P[k + 4].idr + 64, 0, 0);
            }
            memcpy(s.qraw.h + q, seq_qer + sp.idq, (size_t)sp.len2);
            memcpy(s.rraw.h + r, seq_ref + sp.idr, (size_t)sp.len1);
            s.desc.h[k] = make_int4((int)q, (int)r, sp.len2 | (sp.len1 << 16), sp.h0);
            q += (uint64_t)sp.len2; r += (uint64_t)sp.len1;
        }
    });
    memset(s.qraw.h + qtot, 0, 64); memset(s.rraw.h + rtot, 0, 64);
    stats_of(eng).ms_pack += now_ms() - t0;
    // H2D
    bsw_info_init<<<1, PREP_BLOCK, 0, s.st>>>(s.d_info);
    stats_of(eng).kernel_launches++;
    CUDA_TRY(cudaMemcpyAsync(s.desc.d, s.desc.h, sizeof(int4) * (size_t)n, cudaMemcpyHostToDevice, s.st));
    CUDA_TRY(cudaMemcpyAsync(s.qraw.d, s.qraw.h, (size_t)qtot + 64, cudaMemcpyHostToDevice, s.st));
    CUDA_TRY(cudaMemcpyAsync(s.rraw.d, s.rraw.h, (size_t)rtot + 64, cudaMemcpyHostToDevice, s.st));
    s.qbase = s.qraw.d; s.rbase = s.rraw.d;
    s.seq_on_device = true;
    stats_of(eng).h2d_bytes += (int64_t)(sizeof(int4) * (size_t)n + qtot + rtot + 128);
    return BSW_OK;
}

// ------------------------------------------------------------------------------------------
// stage C (both routes): bucket, pack in processing order, launch plan
// ------------------------------------------------------------------------------------------
#define TL_MARK(K) do { if (g_timeline) CUDA_TRY(cudaEventRecord(s.ev_tl[K], s.st)); } while (0)
int device_prepare(bsw_engine* eng, DevCtx& c, Slot& s)
{
    ChunkInfo& I = s.info;
    const int n = s.n;
    // Latency route (a batch too small to fill the machine one pair per thread, e.g. the reference
    // driver's -b 512): no bucketing, no packing -- every pair is listed for the warp-per-pair kernel,
    // whose rows live in shared memory; a pair then takes ~0.1 ms instead of ~0.35 ms.
    if (s.tiny) I.n_short = 0;
    s.n_sorted = I.n_short;
    // (packed route: 2-bit pairs outside the 16-bit kernel's score domain cannot fall back to the byte kernel --
    // the chunk then runs the 32-bit kernel as a whole)
    s.use16 = eng->use16 && !(s.src2bit && I.n_wide > 0);
    const size_t qwords = (size_t)(I.qbases / 16) + (size_t)I.n_short + 8;
    const size_t twords = (size_t)(I.tbases / 16) + (size_t)I.n_short + 8;
    if (int rc = ensure(eng, s.meta, (size_t)n)) return rc;
    if (int rc = ensure(eng, s.res, (size_t)n, !s.out_records)) return rc;
    if (int rc = ensure(eng, s.qpk, qwords)) return rc;
    if (int rc = ensure(eng, s.tpk, twords)) return rc;
    if (int rc = ensure(eng, s.perm, (size_t)n)) return rc;
    if (int rc = ensure(eng, s.rank, (size_t)n)) return rc;
    if (int rc = ensure(eng, s.nlist, (size_t)n)) return rc;
    if (int rc = ensure(eng, s.llist, (size_t)n)) return rc;
    s.plan.clear();
    {
        BucketKey K;
        K.mn2 = I.n_short ? I.mn[0] : 0; K.mnh = I.n_short ? I.mn[1] : 0; K.mn1 = I.n_short ? I.mn[2] : 0;
        const int b_l2 = I.n_short ? bits_for((uint32_t)(I.mx[0] - I.mn[0])) : 0;        // <= 10: never shortened
        const int w_h0 = I.n_short ? bits_for((uint32_t)(I.mx[1] - I.mn[1])) : 0;
        const int w_l1 = I.n_short ? bits_for((uint32_t)(I.mx[2] - I.mn[2])) : 0;
        // key = len2 | h0 | len1 cut to the bin table's BUCKET_BITS.  BSW_KEY_MODE (experiments): 0 = drop the low bits
        // of the last field only (h0 exact, len1 coarse), 1 = len2 | len1 | h0 the same way, 2 = len2 | len1 | h0 with
        // the dropped bits shared between both fields
        // (measured, r02j_keymode.log: the orders differ by <= 2 %; 2 is never behind: short8 2.205 -> 2.167 ms, sweep w = 500 22.00 -> 21.58 ms)
        static const int key_mode = getenv("BSW_KEY_MODE") ? atoi(getenv("BSW_KEY_MODE")) : 2;
        const int room = std::max(0, BUCKET_BITS - b_l2);
        K.l1_first = key_mode != 0;
        if (key_mode == 2) {
            int k_l1 = std::min(w_l1, (room * 3 + 4) / 5), k_h0 = std::min(w_h0, room - k_l1);
            k_l1 = std::min(w_l1, room - k_h0);
            K.b_l1 = k_l1; K.b_h0 = k_h0;
        } else if (key_mode == 1) {
            K.b_l1 = std::min(w_l1, room); K.b_h0 = std::min(w_h0, room - K.b_l1);
        } else {
            K.b_h0 = std::min(w_h0, room); K.b_l1 = std::min(w_l1, room - K.b_h0);
        }
        K.s_h0 = w_h0 - K.b_h0; K.s_l1 = w_l1 - K.b_l1;
        const int total = b_l2 + K.b_h0 + K.b_l1;
        K.short_max = s.tiny ? 0 : eng->short_max;
        const int nbins = 1 << total;
        const int ntiles = (nbins + SCAN_TILE - 1) / SCAN_TILE;           // <= 256
        const size_t nb_pad = (size_t)ntiles * SCAN_TILE;                  // whole tiles, so the scan needs no edge cases
        if (int rc = ensure(eng, s.bins, BINS_WORDS)) return rc;            // bins, tile totals, ticket counter
        uint32_t* totals = s.bins.d + nb_pad;
        unsigned int* ticket = totals + SCAN_MAX_TILES;
        if (!s.bins_zeroed) {                                                // (direct route: cleared at open())
            bsw_zero_words<<<64, PREP_BLOCK, 0, s.st>>>(reinterpret_cast<uint4*>(s.bins.d), (int)(BINS_WORDS / 4));
            stats_of(eng).kernel_launches++;
        }
        s.bins_zeroed = false;
        TL_MARK(0);
        bsw_bucket_count<<<grid_for(c, n, 2 * PREP_BLOCK), PREP_BLOCK, 0, s.st>>>(s.desc.d, n, K, s.bins.d, s.rank.d, s.llist.d, s.d_info);
        stats_of(eng).kernel_launches++;
        TL_MARK(1);
        if (I.n_short > 0) {
            bsw_bucket_scan<<<ntiles, PREP_BLOCK, 0, s.st>>>(s.bins.d, nbins, totals, ticket);
            TL_MARK(2);
            static const bool gather = getenv("BSW_PACKED_GATHER") && atoi(getenv("BSW_PACKED_GATHER")) != 0;   // A/B: re-lay the words in processing order
            if (s.src2bit && !gather) {
                // packed route: the DP kernels read the 2-bit words where the host's DMA left them
                bsw_bucket_scatter<true><<<grid_for(c, n, 2 * PREP_BLOCK), PREP_BLOCK, 0, s.st>>>(
                    s.desc.d, n, K, s.bins.d, totals, s.rank.d, s.perm.d, s.meta.d, s.nlist.d, s.d_info, s.q_lo, s.r_lo);
                TL_MARK(3);
                s.dp_q = reinterpret_cast<const uint32_t*>(s.q2src); s.dp_t = reinterpret_cast<const uint32_t*>(s.r2src);
                stats_of(eng).kernel_launches += 2;
            } else {
                bsw_bucket_scatter<false><<<grid_for(c, n, 2 * PREP_BLOCK), PREP_BLOCK, 0, s.st>>>(s.desc.d, n, K, s.bins.d, totals, s.rank.d, s.perm.d);
                TL_MARK(3);
                // 2-bit packing in processing order
                if (s.src2bit)
                    bsw_pack_pairs<true><<<grid_for(c, I.n_short, PREP_BLOCK), PREP_BLOCK, 0, s.st>>>(
                        s.desc.d, s.perm.d, I.n_short, s.q2src, s.r2src, s.meta.d, s.qpk.d, s.tpk.d, s.nlist.d, s.d_info, 0, 1,
                        s.q_lo, s.r_lo);
                else
                    bsw_pack_pairs<false><<<grid_for(c, I.n_short, PREP_BLOCK), PREP_BLOCK, 0, s.st>>>(
                        s.desc.d, s.perm.d, I.n_short, s.qbase, s.rbase, s.meta.d, s.qpk.d, s.tpk.d, s.nlist.d, s.d_info,
                        s.use16 ? eng->p.match : 0, s.seq_on_device ? 1 : 0);
                s.dp_q = s.qpk.d; s.dp_t = s.tpk.d;
                stats_of(eng).kernel_launches += 3;
            }
            TL_MARK(4);
            // launch plan: the processing order ascends in len2, so the shared-memory classes are
            // prefix ranges of it, read off the len2 histogram
            static const bool circ_ok = !(getenv("BSW_CIRC") && atoi(getenv("BSW_CIRC")) == 0);   // BSW_CIRC=0: rows always hold the whole query
            int pos = 0;
            for (int l = I.mn[0]; l <= std::min(I.mx[0], eng->short_max); ++l) {
                const int cnt = (int)I.hist[l];
                if (!cnt) continue;
                int qs = stride_for(l, s.use16);
                int wc = 0;
                const int plane = qs;
                if (s.use16 && circ_ok && eng->kp.w <= 4096 && (k16::circ_cols(eng->kp.w) + 4) * 10 <= qs * 7) {
                    // the band is much narrower than the query: circular rows of the band's width (bsw_kernel16.cuh);
                    // every longer class then shares one row stride and merges into one launch.  Only where the
                    // rows shrink by 30 % or more: the wrap costs ~6 registers and a few instructions per block,
                    // and measured at w = 100 / qlen <= 300 (rows 26 % smaller at best) it gains nothing
                    // (long16 5 % slower), while at w = 32 it is worth +32 % (scripts/sweep_points.py)
                    wc = k16::circ_cols(eng->kp.w);
                    qs = wc + 4;
                }
                if (!s.plan.empty() && s.plan.back().qstride == qs && s.plan.back().wcols == wc) {
                    s.plan.back().count += cnt;
                    s.plan.back().plane = std::max(s.plan.back().plane, plane);
                } else {
                    Launch L{pos, cnt, qs, SHORT_BLOCK};
                    L.wcols = wc; L.plane = plane;
                    s.plan.push_back(L);
                }
                pos += cnt;
            }
            if (s.use16) for (Launch& L : s.plan) L.block = short16_block(L.qstride, L.plane, L.wcols != 0);
            // a call too small to fill the machine one pair per thread: the classes with queries <= w16::MAX_QLEN (a prefix
            // of the processing order) become one launch of the warp-per-pair register kernel
            if (s.use16 && s.warp_ok && pos > 0 && I.mn[0] <= w16::MAX_QLEN) {
                int cnt = 0;
                for (int l = I.mn[0]; l <= std::min(I.mx[0], w16::MAX_QLEN); ++l) cnt += (int)I.hist[l];
                size_t k = 0;
                while (k < s.plan.size() && s.plan[k].first + s.plan[k].count <= cnt) ++k;
                if (k < s.plan.size() && s.plan[k].first < cnt) {            // a merged class straddles the limit: cut it
                    s.plan[k].count -= cnt - s.plan[k].first;
                    s.plan[k].first = cnt;
                }
                s.plan.erase(s.plan.begin(), s.plan.begin() + (std::ptrdiff_t)k);
                Launch L{0, cnt, 0, WARP_BLOCK};
                L.warp = true;
                s.plan.insert(s.plan.begin(), L);
            }
        }
    }
    CUDA_TRY(cudaGetLastError());
    // the pack kernel's counters (pairs for the byte kernels) travel back with the chunk
    // the DP launches fork here, ahead of the summary's trip to the host (a PCIe write that queues
    // behind the result traffic)
    CUDA_TRY(cudaEventRecord(s.ev_fork, s.st));
    s.fork_recorded = true;
    bsw_info_publish<<<1, PREP_BLOCK, 0, s.st>>>(s.d_info, s.h_info_dev);
    CUDA_TRY(cudaGetLastError());
    stats_of(eng).kernel_launches++;
    CUDA_TRY(cudaEventRecord(s.ev_lists, s.st));
    return BSW_OK;
}

void launch_warp(bsw_engine* eng, cudaStream_t st, const int4* meta, const uint32_t* perm, const uint32_t* qseq,
                 const uint32_t* tseq, int4* res, int first, int count, unsigned long long* cells)
{
    constexpr int PAIRS = WARP_BLOCK / 32;
    const int grid = (count + PAIRS - 1) / PAIRS;
    const size_t smem = w16::MASK_BYTES + (size_t)PAIRS * w16::SCORE_BYTES;
    if (eng->kp.oe_del == eng->kp.oe_ins)
        bsw_warp16_kernel<WARP_BLOCK, true><<<grid, WARP_BLOCK, smem, st>>>(meta, perm, qseq, tseq, res, first, count, eng->kp, cells);
    else
        bsw_warp16_kernel<WARP_BLOCK, false><<<grid, WARP_BLOCK, smem, st>>>(meta, perm, qseq, tseq, res, first, count, eng->kp, cells);
}

// DP launches of a chunk: fan out over the device's compute streams (those of the DP partition
// when the batch runs partitioned), longest class first
int launch_dp(bsw_engine* eng, DevCtx& c, Slot& s, bool partitioned = false)
{
    cudaStream_t* cs = partitioned ? c.cs_part : c.cs;
    if (!s.fork_recorded) CUDA_TRY(cudaEventRecord(s.ev_fork, s.st));
    s.fork_recorded = false;
    if (s.plan.empty()) return BSW_OK;
    const int nl = (int)s.plan.size();
    const int used = std::min(nl, NSTREAMS);
    for (int k = 0; k < used; ++k) CUDA_TRY(cudaStreamWaitEvent(cs[k], s.ev_fork, 0));
    int li = 0;
    for (int k = nl - 1; k >= 0; --k, ++li) {
        const Launch& L = s.plan[(size_t)k];
        cudaStream_t st = cs[li % NSTREAMS];
        const int grid = (L.count + L.block - 1) / L.block;
        if (L.warp) {
            launch_warp(eng, st, s.meta.d, s.perm.d, s.dp_q, s.dp_t, s.res.d, L.first, L.count, c.d_cells);
        } else if (s.use16) {
            const bool sg = eng->kp.oe_del == eng->kp.oe_ins;
            const size_t smem = k16::smem_bytes(L.block, L.qstride, L.plane);
#define BSW_LAUNCH16(B, SG, CIRC)                                                                                     \
            bsw_short16_kernel<B, SG, CIRC><<<grid, B, smem, st>>>(s.meta.d, s.perm.d, s.dp_q, s.dp_t, s.res.d, L.first,     \
                                                                   L.count, L.qstride, eng->kp, c.d_cells, L.wcols)
            const int variant = (L.block == 32 ? 4 : 0) | (sg ? 2 : 0) | (L.wcols ? 1 : 0);
            switch (variant) {
                case 0: BSW_LAUNCH16(64, false, false); break;
                case 1: BSW_LAUNCH16(64, false, true); break;
                case 2: BSW_LAUNCH16(64, true, false); break;
                case 3: BSW_LAUNCH16(64, true, true); break;
                case 4: BSW_LAUNCH16(32, false, false); break;
                case 5: BSW_LAUNCH16(32, false, true); break;
                case 6: BSW_LAUNCH16(32, true, false); break;
                default: BSW_LAUNCH16(32, true, true); break;
            }
#undef BSW_LAUNCH16
        } else {
            bsw_short_kernel<SHORT_BLOCK, false><<<grid, SHORT_BLOCK, short_smem_bytes(L.qstride), st>>>(
                s.meta.d, s.perm.d, s.dp_q, s.dp_t, s.res.d, L.first, L.count, L.qstride, eng->kp, c.d_cells);
        }
        stats_of(eng).kernel_launches++;
    }
    CUDA_TRY(cudaGetLastError());
    for (int k = 0; k < used; ++k) {
        CUDA_TRY(cudaEventRecord(c.ev_join[k], cs[k]));
        CUDA_TRY(cudaStreamWaitEvent(s.st, c.ev_join[k], 0));
    }
    return BSW_OK;
}

// byte-reading kernels for the pairs the pack kernel listed (N-containing / long); counts known
int launch_bytes(bsw_engine* eng, DevCtx& c, Slot& s)
{
    if (s.n_nlist > 0) {
        const int qstride = stride_for(s.qmax_n);
        const int grid = (int)((s.n_nlist + SHORT_BLOCK - 1) / SHORT_BLOCK);
        bsw_short_kernel<SHORT_BLOCK, true><<<grid, SHORT_BLOCK, short_smem_bytes(qstride), s.st>>>(
            s.desc.d, s.nlist.d, reinterpret_cast<const uint32_t*>(s.qbase), reinterpret_cast<const uint32_t*>(s.rbase),
            s.res.d, 0, (int)s.n_nlist, qstride, eng->kp, c.d_cells);
        stats_of(eng).kernel_launches++;
    }
    if (s.n_llist > 0) {
        s.long_stride = (s.info.qmax_all + 12) & ~3;
        int64_t blocks = std::min<int64_t>(((int64_t)s.n_llist + LONG_WARPS - 1) / LONG_WARPS, (int64_t)c.sms * 8);
        const int64_t cap_words = (int64_t)(256ll << 20) / 4;       // <= 256 MB of eh rows
        blocks = std::max<int64_t>(1, std::min(blocks, cap_words / ((int64_t)s.long_stride * LONG_WARPS)));
        s.long_blocks = (int)blocks;
        const size_t row_bytes = (size_t)LONG_WARPS * (size_t)s.long_stride * sizeof(uint32_t);
        CUDA_TRY(cudaMemsetAsync(s.d_queue, 0, sizeof(unsigned int), s.st));
        if (row_bytes <= 48 * 1024) {                    // rows in shared memory (queries up to ~3000)
            bsw_long_kernel<true><<<s.long_blocks, LONG_WARPS * 32, row_bytes, s.st>>>(
                s.desc.d, s.llist.d, s.qbase, s.rbase, s.res.d, (int)s.n_llist, eng->kp, nullptr, s.long_stride,
                s.d_queue, c.d_cells);
        } else {
            if (int rc = ensure(eng, s.scratch, (size_t)blocks * LONG_WARPS * (size_t)s.long_stride)) return rc;
            bsw_long_kernel<false><<<s.long_blocks, LONG_WARPS * 32, 0, s.st>>>(
                s.desc.d, s.llist.d, s.qbase, s.rbase, s.res.d, (int)s.n_llist, eng->kp, s.scratch.d, s.long_stride,
                s.d_queue, c.d_cells);
        }
        stats_of(eng).kernel_launches++;
    }
    CUDA_TRY(cudaGetLastError());
    return BSW_OK;
}

// results of a chunk leave the device: straight into the caller's records (direct) or D2H
int output_chunk(bsw_engine* eng, DevCtx& c, Slot& s, const Job& job)
{
    SeqPair* const pairs = job.pairs;
    if (s.packed) {
        // the six result fields alone: 16 bytes per pair as the kernels leave them, or OutScore records (24 bytes)
        if (job.out16) {
            CUDA_TRY(cudaMemcpyAsync(static_cast<bsw_score16*>(job.out) + s.a, s.res.d, sizeof(int4) * (size_t)s.n, cudaMemcpyDeviceToHost, s.st));
            stats_of(eng).d2h_bytes += (int64_t)sizeof(int4) * s.n;
        } else {
            if (int rc = ensure(eng, s.outbuf, sizeof(OutScore) * (size_t)s.n)) return rc;
            bsw_out_scores<<<grid_for(c, s.n, 2 * PREP_BLOCK), PREP_BLOCK, 0, s.st>>>(s.res.d, s.n, reinterpret_cast<int2*>(s.outbuf.d));
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaMemcpyAsync(static_cast<OutScore*>(job.out) + s.a, s.outbuf.d, sizeof(OutScore) * (size_t)s.n, cudaMemcpyDeviceToHost, s.st));
            stats_of(eng).kernel_launches++;
            stats_of(eng).d2h_bytes += (int64_t)sizeof(OutScore) * s.n;
        }
    } else if (s.out_records) {
        // results go into the device copy of the records, which then returns by one DMA (the
        // input fields come back as they left; per-field writes over PCIe would be 4-byte TLPs)
        bsw_writeback<<<grid_for(c, s.n, 2 * PREP_BLOCK), PREP_BLOCK, 0, s.st>>>(s.res.d, s.n, reinterpret_cast<SeqPair*>(s.raw_pairs.d));
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaMemcpyAsync(pairs + s.a, s.raw_pairs.d, (size_t)s.n * sizeof(SeqPair), cudaMemcpyDeviceToHost, s.st));
        stats_of(eng).kernel_launches++;
        stats_of(eng).d2h_bytes += (int64_t)s.n * (int64_t)sizeof(SeqPair);
    } else {
        CUDA_TRY(cudaMemcpyAsync(s.res.h, s.res.d, sizeof(int4) * (size_t)s.n, cudaMemcpyDeviceToHost, s.st));
        stats_of(eng).d2h_bytes += (int64_t)sizeof(int4) * s.n;
    }
    CUDA_TRY(cudaEventRecord(s.ev_out, s.st));
    return BSW_OK;
}

inline void write_result(SeqPair& sp, const int4 v)
{
    sp.score = (int16_t)(v.x & 0xffff);  sp.qle = (int16_t)(v.x >> 16);
    sp.tle = (int16_t)(v.y & 0xffff);    sp.gtle = (int16_t)(v.y >> 16);
    sp.gscore = (int16_t)(v.z & 0xffff); sp.max_off = (int16_t)(v.z >> 16);
}

// staged route: second streaming pass, results into the caller's records
void unpack_chunk(bsw_engine* eng, Slot& s, SeqPair* pairs)
{
    if (s.out_records || s.packed) return;
    const double t0 = now_ms();
    SeqPair* P = pairs + s.a;
    const int4* r = s.res.h;
    eng->pool->for_range(s.n, 8192, [&](int64_t b, int64_t e, int) {
        for (int64_t k = b; k < e; ++k) write_result(P[k], r[k]);
    });
    stats_of(eng).ms_scatter += now_ms() - t0;
}

// after ev_lists: the pack kernel's counters are on the host
void read_lists(Slot& s)
{
    s.n_nlist = s.h_info->n_nlist; s.n_llist = s.h_info->n_llist; s.qmax_n = s.h_info->qmax_n;
}

int begin_batch(bsw_engine* eng, const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer,
                int64_t n, int32_t w)
{
    eng->err.clear();
    eng->staged = false; eng->ran = false;
    if (n < 0 || w < 0 || (n > 0 && (!pairs || !seq_ref || !seq_qer))) { eng->err = "bad arguments"; return BSW_ERR_PARAM; }
    if (n > 0x7fffffff) { eng->err = "more than 2^31-1 pairs per call"; return BSW_ERR_PARAM; }
    bsw_stats& S = eng->stats;
    memset(&S, 0, sizeof(S));
    S.pairs = n;
    eng->n = n; eng->w = w; eng->kp.w = w;
    return BSW_OK;
}

const char* kDomainMsg =
    "pair outside the domain: need 1<=len1,len2<=32767, h0>=0, h0+len2*match<=32767, offsets>=0 "
    "(bandedSWA.h:84, SURVEY 8b); result fields of the batch are unspecified";

struct ChunkRef { int dev; int slot; };

// The latency route: a call too small to fill the machine one pair per thread (bsw_params.tiny_batch; the reference
// driver's habit is 512 pairs per call, scripts/run-cpu.sh:30).  One host pass validates the pairs and gathers
// descriptors and sequence bytes into ONE page-locked block, whose first word is the kernel's work-queue counter
// (the copy that brings the data also zeroes it); one copy in, the warp-per-pair kernel on every pair (rows in shared
// memory), one copy out, one synchronisation: 4 CUDA calls per call instead of ~15, which is what bounds T driver
// threads (the runtime serialises API calls per process).  Returns 1 when the call does not fit this route.
int run_tiny(bsw_engine* eng, const Job& job, int dev_index, int64_t a0, int64_t n64)
{
    DevCtx& c = eng->devs[(size_t)dev_index];
    bsw_stats& S = stats_of(eng);
    const int n = (int)n64;
    const SeqPair* P = job.pairs + a0;
    const int match = eng->p.match;
    uint64_t qtot = 0, rtot = 0, nominal = 0;
    int qmax = 0;
    for (int k = 0; k < n; ++k) {
        const SeqPair& sp = P[k];
        if (sp.len1 < 1 || sp.len1 > 32767 || sp.len2 < 1 || sp.len2 > 32767 || sp.h0 < 0 ||
            (int64_t)sp.h0 + (int64_t)sp.len2 * match > 32767 || sp.idr < 0 || sp.idq < 0) {
            err_of(eng) = kDomainMsg;
            return BSW_ERR_DOMAIN;
        }
        qtot += (uint64_t)sp.len2; rtot += (uint64_t)sp.len1;
        nominal += (uint64_t)sp.len1 * (uint64_t)sp.len2;
        qmax = std::max(qmax, sp.len2);
    }
    const int long_stride = (qmax + 12) & ~3;
    const size_t row_bytes = (size_t)LONG_WARPS * (size_t)long_stride * sizeof(uint32_t);
    if (row_bytes > 48 * 1024 || qtot + rtot > (64u << 20)) return 1;      // very long queries: the general route
    CUDA_TRY(cudaSetDevice(c.dev));
    Slot* sp0 = nullptr;
    if (int rc = get_slot(eng, c, 0, &sp0)) return rc;
    Slot& s = *sp0;
    // Queries of at most 255 bases: the warp-per-pair register kernel (bsw_warp16.cuh) on 2-bit words packed by the host
    // pass.  A call with an N or a pair outside the 16-bit score domain keeps the byte route below.
    if (qmax <= w16::MAX_QLEN && eng->use16 && eng->p.warp_max_pairs >= 0 && w16::scoring_ok(eng->kp)) {
        if (int rc = set_kernel_attrs(eng, c)) return rc;
        const size_t off_desc = 64, off_q = off_desc + sizeof(int4) * (size_t)n;
        const size_t qwords = (size_t)(qtot / 16) + (size_t)n + 4, twords = (size_t)(rtot / 16) + (size_t)n + 4;
        const size_t off_t = off_q + 4 * qwords;
        if (int rc = ensure(eng, s.tinybuf, off_t + 4 * twords, true)) return rc;
        if (int rc = ensure(eng, s.res, (size_t)n, true)) return rc;
        uint8_t* const hb = s.tinybuf.h;
        int4* const hd = reinterpret_cast<int4*>(hb + off_desc);
        uint32_t* const hq = reinterpret_cast<uint32_t*>(hb + off_q);
        uint32_t* const ht = reinterpret_cast<uint32_t*>(hb + off_t);
        uint32_t q = 0, r = 0;
        bool plain = true;
        for (int k = 0; k < n && plain; ++k) {
            const SeqPair& sp = P[k];
            if (!k16::eligible(match, sp.len2, sp.h0)) { plain = false; break; }
            if (pack_seq(job.seq_qer + sp.idq, sp.len2, hq + q) | pack_seq(job.seq_ref + sp.idr, sp.len1, ht + r)) { plain = false; break; }
            hd[k] = make_int4((int)q, (int)r, sp.len2 | (sp.len1 << 16), sp.h0);
            q += (uint32_t)(sp.len2 + 15) >> 4; r += (uint32_t)(sp.len1 + 15) >> 4;
        }
        if (plain) {
            cudaStream_t st = s.st_plain;
            const size_t h2d = off_t + 4 * (size_t)r;
            CUDA_TRY(cudaMemcpyAsync(s.tinybuf.d, hb, h2d, cudaMemcpyHostToDevice, st));
            const int4* const d_desc = reinterpret_cast<const int4*>(s.tinybuf.d + off_desc);
            const uint32_t* const d_q = reinterpret_cast<const uint32_t*>(s.tinybuf.d + off_q);
            const uint32_t* const d_t = reinterpret_cast<const uint32_t*>(s.tinybuf.d + off_t);
            // a warp per pair while the device's budget of such pairs lasts (WarpLease), else the thread-per-pair kernel on
            // the same words: 0.4 ms per call instead of 0.14, but next to no load on a GPU whose issue rate is the bound
            WarpLease lease;
            if (!lease.acquire(eng, c.dev, n, eng->use16, eng->p.warp_max_pairs)) {
                const int qs = stride_for(qmax, true);
                const int block = short16_block(qs, qs, false);
                const int grid = (n + block - 1) / block;
                const size_t smem = k16::smem_bytes(block, qs, qs);
                const bool sg = eng->kp.oe_del == eng->kp.oe_ins;
#define BSW_LAUNCH16T(B, SG) bsw_short16_kernel<B, SG, false><<<grid, B, smem, st>>>(d_desc, nullptr, d_q, d_t, s.res.d, 0, n, qs, eng->kp, nullptr, 0)
                if (block == 32) { if (sg) BSW_LAUNCH16T(32, true); else BSW_LAUNCH16T(32, false); }
                else { if (sg) BSW_LAUNCH16T(64, true); else BSW_LAUNCH16T(64, false); }
#undef BSW_LAUNCH16T
            } else {
                launch_warp(eng, st, d_desc, nullptr, d_q, d_t, s.res.d, 0, n, nullptr);
            }
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaMemcpyAsync(s.res.h, s.res.d, sizeof(int4) * (size_t)n, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            SeqPair* out = job.pairs + a0;
            int64_t cells = 0;
            for (int k = 0; k < n; ++k) { write_result(out[k], s.res.h[k]); cells += s.res.h[k].w; }
            S.cells_nominal += (int64_t)nominal; S.cells_effective += cells; S.kernel_launches += 1; S.n_short += n;
            S.h2d_bytes += (int64_t)h2d; S.d2h_bytes += (int64_t)sizeof(int4) * n;
            return BSW_OK;
        }
    }
    const size_t off_desc = 64, off_q = off_desc + sizeof(int4) * (size_t)n;
    const size_t off_r = (off_q + qtot + 64 + 15) & ~(size_t)15, total = off_r + rtot + 64;
    if (int rc = ensure(eng, s.tinybuf, total, true)) return rc;
    if (int rc = ensure(eng, s.res, (size_t)n, true)) return rc;
    uint8_t* const hb = s.tinybuf.h;
    memset(hb, 0, 64);                                                      // the queue counter (and padding)
    int4* const hd = reinterpret_cast<int4*>(hb + off_desc);
    uint64_t q = 0, r = 0;
    for (int k = 0; k < n; ++k) {
        const SeqPair& sp = P[k];
        memcpy(hb + off_q + q, job.seq_qer + sp.idq, (size_t)sp.len2);
        memcpy(hb + off_r + r, job.seq_ref + sp.idr, (size_t)sp.len1);
        hd[k] = make_int4((int)q, (int)r, sp.len2 | (sp.len1 << 16), sp.h0);
        q += (uint64_t)sp.len2; r += (uint64_t)sp.len1;
    }
    memset(hb + off_q + qtot, 0, 64); memset(hb + off_r + rtot, 0, 64);
    cudaStream_t st = s.st_plain;
    CUDA_TRY(cudaMemcpyAsync(s.tinybuf.d, hb, total, cudaMemcpyHostToDevice, st));
    const int blocks = std::max(1, std::min((n + LONG_WARPS - 1) / LONG_WARPS, c.sms * 8));
    bsw_long_kernel<true><<<blocks, LONG_WARPS * 32, row_bytes, st>>>(
        reinterpret_cast<const int4*>(s.tinybuf.d + off_desc), nullptr, s.tinybuf.d + off_q, s.tinybuf.d + off_r, s.res.d, n, eng->kp,
        nullptr, long_stride, reinterpret_cast<unsigned int*>(s.tinybuf.d), nullptr);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(s.res.h, s.res.d, sizeof(int4) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    SeqPair* out = job.pairs + a0;
    int64_t cells = 0;
    for (int k = 0; k < n; ++k) { write_result(out[k], s.res.h[k]); cells += s.res.h[k].w; }
    S.cells_nominal += (int64_t)nominal; S.cells_effective += cells; S.kernel_launches += 1; S.n_long += n;
    S.h2d_bytes += (int64_t)total; S.d2h_bytes += (int64_t)sizeof(int4) * n;
    return BSW_OK;
}

// Runs the chunks of the batch through the pipeline.  keep == true: stop before the DP launches
// and keep every chunk resident in its own slot (bsw_stage).
//
// The call's pairs [a0, a0 + n) run on the devices [dev_lo, dev_lo + ndev) of the engine, chunks dealt round-robin
// (run_sharded gives every device its own contiguous, cost-balanced range and its own host thread; bsw_stage deals
// one range over all devices).
int run_pipeline(bsw_engine* eng, const Job& job, int dev_lo, int ndev, int64_t a0, int64_t n, int64_t chunk_pairs, bool keep)
{
    bsw_stats& S = stats_of(eng);
    SeqPair* const pairs = job.pairs;
    const uint8_t* const seq_ref = job.seq_ref;
    const uint8_t* const seq_qer = job.seq_qer;
    const bool packed = job.pb != nullptr;
    const bool direct = packed || (!job.force_staged && is_pinned(pairs) && is_pinned(seq_ref) && is_pinned(seq_qer));
    // direct route, way out: the records' device copy with the six fields filled in (72 B per pair, no host pass), or
    // BSW_DIRECT_OUT=results: the 16-byte results + the staged route's host pass into the caller's records
    static const bool out_records = !(getenv("BSW_DIRECT_OUT") && std::string(getenv("BSW_DIRECT_OUT")) == "results");
    // PCIe-bound or compute-bound?  A sample of the records gives DP time (nominal cells at the
    // resident kernel rate) against transfer time (record + sequence bytes at PCIe rate) per pair.
    // PCIe-bound batches run partitioned: chunk streams on the service SMs, DP on the rest.
    bool partitioned = false, pcie_bound = false;
    if (!keep && n >= 4 * CHUNK_MIN) {
        double cells = 0, bytes = 0;
        const int64_t step = std::max<int64_t>(1, n / 509);
        for (int64_t i = a0; i < a0 + n; i += step) {
            if (packed) {
                const bsw_pair_desc& d = job.pb->desc[i];
                cells += (double)d.len1 * (double)d.len2;
                bytes += (double)sizeof(bsw_pair_desc) + ((d.flags & BSW_PAIR_RAW) ? (double)d.len1 + d.len2 : 0.25 * ((double)d.len1 + d.len2));
            } else {
                cells += (double)pairs[i].len1 * (double)pairs[i].len2;
                bytes += (double)sizeof(SeqPair) + (double)pairs[i].len1 + (double)pairs[i].len2;
            }
        }
        pcie_bound = partitioned = cells / 2.0e9 < 0.7 * (bytes / 50e6);
        for (int d = dev_lo; d < dev_lo + ndev; ++d) partitioned = partitioned && eng->devs[(size_t)d].svc_sms > 0;
    }
    S.partitioned = partitioned ? 1 : 0;
    const bool tiny = !keep && !packed && eng->p.tiny_batch > 0 && n <= eng->p.tiny_batch;
    // short pairs one per warp (bsw_warp16.cuh)?  A call on one device takes its pairs out of the device's budget for as
    // long as it runs; a resident batch (its runs come later) and a batch dealt over several devices go by size alone
    WarpLease warp_lease;
    const bool warp_pairs = (keep || ndev != 1) ? warp_fits(eng, n)
        : warp_lease.acquire(eng, eng->devs[(size_t)dev_lo].dev, n, eng->use16, eng->p.warp_max_pairs);

    // chunk boundaries: a small first chunk (the first DP starts after a short H2D), full-size
    // chunks, then -- where transfers or the host bound the batch -- a geometric ramp-down so that the
    // work left after the last H2D (its DP and its D2H) is small.  PCIe-bound batches use smaller full-size chunks, sized so that the DP of one
    // chunk finishes while the next arrives; compute-bound ones ramp up to large chunks (fewer
    // launch tails, better bucketing).
    // (pageable buffers: the host passes are the bottleneck and want large chunks for their thread pool)
    const bool small_chunks = pcie_bound && direct;
    static const int64_t env_chunk = getenv("BSW_CHUNK") ? atoll(getenv("BSW_CHUNK")) : 0;          // experiments
    static const int env_rampdown = getenv("BSW_RAMPDOWN") ? atoi(getenv("BSW_RAMPDOWN")) : -1;
    const int64_t big = small_chunks ? CHUNK_PCIE : (env_chunk > 0 && !keep ? env_chunk : chunk_pairs);
    const int64_t tail_min = small_chunks ? CHUNK_MIN / 2 : CHUNK_MIN;    // the last chunk's latency is all tail
    // (a compute-bound batch on pinned buffers has all its data on the device long before the DP is done:
    // small last chunks only add launches with few blocks -- scripts/chunk_probe.py: large mix 23.1 -> 21.9 ms)
    const bool rampdown = env_rampdown >= 0 ? env_rampdown != 0 : (small_chunks || !direct);
    std::vector<int64_t> cut{a0};
    static const int64_t env_first = getenv("BSW_FIRST_CHUNK") ? atoll(getenv("BSW_FIRST_CHUNK")) : 0;
    // (packed route, compute-bound: the whole batch arrives in a fraction of its DP time, and 64 k pairs -- half of what
    // the SMs hold at once -- start the DP 0.15 ms earlier than they cost in launch tails: 3.07 -> 2.93 ms per 1 M short pairs)
    int64_t ramp = keep ? big : (env_first > 0 && !small_chunks ? env_first : (packed && !small_chunks ? 2 * CHUNK_MIN : CHUNK_MIN));
    for (int64_t rem = n; rem > 0;) {
        int64_t sz;
        if (ramp < big && rem > 4 * ramp) { sz = ramp; ramp = small_chunks ? big : ramp * 2; }
        else if (keep || rem > 2 * big) sz = std::min(rem, big);
        else if (rampdown && rem > 2 * tail_min) sz = std::min(rem, ((rem + 1) / 2 + 4095) & ~(int64_t)4095);
        else sz = rem;
        cut.push_back(cut.back() + sz);
        rem -= sz;
    }
    const int64_t nchunks = (int64_t)cut.size() - 1;
    std::vector<ChunkRef> refs((size_t)nchunks);
    const double tl_host0 = now_ms();
    std::vector<std::string> tl_lines;
    if (keep) eng->staged_chunks.clear();
    for (int d = dev_lo; d < dev_lo + ndev; ++d) {
        DevCtx& c = eng->devs[(size_t)d];
        CUDA_TRY(cudaSetDevice(c.dev));
        if (int rc = set_kernel_attrs(eng, c)) return rc;
        if (packed) if (int rc = packed_resident(eng, c, *job.pb)) return rc;
    }
    DevCtx& tl_dev = eng->devs[(size_t)dev_lo];                   // BSW_TIMELINE: the device whose events are printed
    auto slot_of = [&](int64_t k) -> Slot& { return eng->devs[(size_t)refs[(size_t)k].dev].slots[(size_t)refs[(size_t)k].slot]; };
    auto dev_of = [&](int64_t k) -> DevCtx& { return eng->devs[(size_t)refs[(size_t)k].dev]; };

    // open: bind chunk k to its device and slot; on the direct route start its records DMA + scan
    auto open = [&](int64_t k) -> int {
        const int d = dev_lo + (int)(k % ndev);
        const int sl = keep ? (int)(k / ndev) : (int)((k / ndev) % NSLOTS);
        refs[(size_t)k] = ChunkRef{d, sl};
        DevCtx& c = eng->devs[(size_t)d];
        CUDA_TRY(cudaSetDevice(c.dev));
        Slot* sp = nullptr;
        if (int rc = get_slot(eng, c, sl, &sp)) return rc;
        Slot& s = *sp;
        s.a = cut[(size_t)k]; s.n = (int)(cut[(size_t)k + 1] - cut[(size_t)k]);
        s.direct = direct;
        s.out_records = direct && !packed && out_records;
        s.packed = packed;
        s.src2bit = packed;                                   // (the staged route sets it in its host pass)
        s.tiny = tiny;
        s.warp_ok = warp_pairs;
        s.st = partitioned ? s.st_svc : s.st_plain;
        if (g_timeline) { if (k == 0) CUDA_TRY(cudaEventRecord(tl_dev.ev_t0, s.st)); s.host_t[0] = now_ms() - tl_host0; }
        CUDA_TRY(cudaEventRecord(s.ev_k0, s.st));
        if (packed) return packed_begin(eng, c, s, *job.pb);
        if (direct) return direct_begin(eng, c, s, pairs, seq_ref, seq_qer);
        return BSW_OK;
    };
    // finish: the chunk's DP is enqueued; learn the byte-kernel lists, run them, send results out
    auto finish = [&](int64_t k) -> int {
        DevCtx& c = dev_of(k); Slot& s = slot_of(k);
        CUDA_TRY(cudaSetDevice(c.dev));
        // only the pack kernel's counters are needed here, not the DP: the byte kernels and the
        // results' way out are stream-ordered behind the DP launches, the host does not wait for them
        CUDA_TRY(cudaEventSynchronize(s.ev_lists));
        if (g_timeline) s.host_t[3] = now_ms() - tl_host0;
        read_lists(s);
        S.n_short += s.n_sorted - (int)s.n_nlist; S.n_long += (int)s.n_llist;
        if (int rc = launch_bytes(eng, c, s)) return rc;
        CUDA_TRY(cudaEventRecord(s.ev_k1, s.st));
        const int rc = output_chunk(eng, c, s, job);
        if (g_timeline) s.host_t[4] = now_ms() - tl_host0;
        return rc;
    };
    auto retire = [&](int64_t k) -> int {
        DevCtx& c = dev_of(k); Slot& s = slot_of(k);
        CUDA_TRY(cudaSetDevice(c.dev));
        CUDA_TRY(cudaEventSynchronize(s.ev_out));
        unpack_chunk(eng, s, pairs);
        float ms = 0;
        if (cudaEventElapsedTime(&ms, s.ev_k0, s.ev_k1) == cudaSuccess) S.ms_kernel += (double)ms;
        if (g_timeline && ndev == 1) {
            s.host_t[5] = now_ms() - tl_host0;
            char line[512];
            float t[7] = {};
            cudaEvent_t evs[7] = {s.ev_k0, s.ev_info, s.ev_seq, s.ev_fork, s.ev_dp, s.ev_k1, s.ev_out};
            for (int e = 0; e < 7; ++e)
                if (cudaEventElapsedTime(&t[e], tl_dev.ev_t0, evs[e]) != cudaSuccess) { t[e] = -1; cudaGetLastError(); }
            snprintf(line, sizeof(line),
                     "chunk %2d n=%7d | dev: open %6.3f rec+scan %6.3f seq %6.3f prep %6.3f dp %6.3f bytes %6.3f out %6.3f"
                     " | host: open %6.3f info %6.3f launched %6.3f dp-seen %6.3f out-enq %6.3f retired %6.3f",
                     (int)k, s.n, t[0], t[1], t[2], t[3], t[4], t[5], t[6],
                     s.host_t[0], s.host_t[1], s.host_t[2], s.host_t[3], s.host_t[4], s.host_t[5]);
            tl_lines.emplace_back(line);
            float p[5] = {};
            for (int e = 0; e < 5; ++e)
                if (cudaEventElapsedTime(&p[e], tl_dev.ev_t0, s.ev_tl[e]) != cudaSuccess) { p[e] = -1; cudaGetLastError(); }
            snprintf(line, sizeof(line), "          prep detail: zero %6.3f count %6.3f scan %6.3f scatter %6.3f pack %6.3f fork %6.3f",
                     p[0], p[1], p[2], p[3], p[4], t[3]);
            tl_lines.emplace_back(line);
        }
        return BSW_OK;
    };

    // Per iteration k: records (and the speculative sequence copy) of chunk k + 3 ndev go out (direct
    // route) so the copy engine never waits for the host; chunk k gets its prep kernels and DP launches; chunk
    // k - ndev drains (byte kernels, results out).  Chunks retire (results on the host; staged route:
    // second host pass) as soon as their D2H has completed, without blocking -- the host only waits
    // for a chunk when the slot it occupies is needed again, NSLOTS chunks later, so that a DP that
    // runs long never keeps the host from feeding the copy engine.
    const int lag = ndev;
    const int ahead = direct && !keep ? 3 * ndev : ndev;     // chunks opened (records + speculative sequence copy) ahead of k
    int64_t next_retire = 0;
    for (int64_t k = 0; k < std::min<int64_t>(ahead, nchunks); ++k) if (int rc = open(k)) return rc;
    for (int64_t k = 0; k < nchunks + lag; ++k) {
        if (k + ahead < nchunks) {
            if (!keep)
                while (next_retire <= k + ahead - (int64_t)NSLOTS * ndev) if (int rc = retire(next_retire++)) return rc;
            if (int rc = open(k + ahead)) return rc;
        }
        if (k < nchunks) {
            DevCtx& c = dev_of(k); Slot& s = slot_of(k);
            CUDA_TRY(cudaSetDevice(c.dev));
            int rc = packed ? packed_info(eng, c, s)
                   : direct ? direct_sequences(eng, s, pairs, seq_ref, seq_qer) : staged_prepare(eng, s, pairs, seq_ref, seq_qer);
            if (rc) { if (rc == BSW_ERR_DOMAIN) err_of(eng) = kDomainMsg; return rc; }
            S.cells_nominal += (int64_t)s.info.nominal;
            if ((rc = device_prepare(eng, c, s))) return rc;
            if (g_timeline) s.host_t[1] = now_ms() - tl_host0;      // (after the wait for the summary + planning)
            if (!keep && (rc = launch_dp(eng, c, s, partitioned))) return rc;
            CUDA_TRY(cudaEventRecord(s.ev_dp, s.st));
            if (g_timeline) s.host_t[2] = now_ms() - tl_host0;
            if (keep) s.fork_recorded = false;                     // bsw_run_staged forks behind its own start event
            if (keep) eng->staged_chunks.emplace_back(refs[(size_t)k].dev, refs[(size_t)k].slot);
        }
        if (keep) continue;
        if (k - lag >= 0 && k - lag < nchunks) if (int rc = finish(k - lag)) return rc;
        while (next_retire < k - lag) {                   // finished chunks whose results have arrived
            Slot& s = slot_of(next_retire);
            CUDA_TRY(cudaSetDevice(dev_of(next_retire).dev));
            const cudaError_t q = cudaEventQuery(s.ev_out);
            if (q == cudaErrorNotReady) break;
            CUDA_TRY(q);
            if (int rc = retire(next_retire++)) return rc;
        }
    }
    if (!keep) while (next_retire < nchunks) if (int rc = retire(next_retire++)) return rc;
    if (g_timeline && !keep) {
        fprintf(stderr, "bsw timeline (ms; device times relative to the first chunk's open, host times to the call):\n");
        for (const std::string& l : tl_lines) fprintf(stderr, "  %s\n", l.c_str());
    }
    if (keep) {
        for (int64_t k = 0; k < nchunks; ++k) {
            DevCtx& c = dev_of(k); Slot& s = slot_of(k);
            CUDA_TRY(cudaSetDevice(c.dev));
            CUDA_TRY(cudaEventSynchronize(s.ev_dp));
            read_lists(s);
            S.n_short += s.n_sorted - (int)s.n_nlist; S.n_long += (int)s.n_llist;
        }
    }
    return BSW_OK;
}

int zero_cells(bsw_engine* eng)
{
    for (DevCtx& c : eng->devs) {
        CUDA_TRY(cudaSetDevice(c.dev));
        CUDA_TRY(cudaMemsetAsync(c.d_cells, 0, sizeof(unsigned long long), c.cs[0]));
        CUDA_TRY(cudaStreamSynchronize(c.cs[0]));
    }
    return BSW_OK;
}

// Estimated DP cost of a pair: rows x min(columns, band) + a fixed per-pair part (SURVEY 8(e))
inline double pair_cost(int len1, int len2, int w)
{
    return (double)len1 * (double)std::min(len2, 2 * w + 1) + 64.0;
}

// The multi-GPU partitioner on the hot path (replaces the OpenMP batch loop, main_banded.cpp:279-291): the call's
// pairs are cut, in input order, into one contiguous range per device with equal estimated DP cost
// (sum of len1 * min(len2, 2w + 1), read off a sample of the records), each range runs through the chunk pipeline of
// its own device on its own host thread, and every chunk's results land at its pairs' input positions.  Contiguous
// ranges keep the host side free of any gather / scatter pass and every copy a plain DMA; the length bucketing
// happens per chunk on the device.  BSW_MULTI=deal in the environment restores the single-thread round-robin
// dealing of chunks over the devices (kept for A/B measurements, scripts/multi_probe.py).
int run_sharded(bsw_engine* eng, const Job& job, int64_t n, int64_t chunk_pairs)
{
    const int ndev = (int)eng->devs.size();
    eng->cells_counted = false;
    if (!job.pb && eng->p.tiny_batch > 0 && n <= eng->p.tiny_batch) {
        static const bool fused = !(getenv("BSW_TINY_FUSED") && atoi(getenv("BSW_TINY_FUSED")) == 0);     // A/B: 0 = the chunk pipeline's latency route
        if (fused) {
            const int rc = run_tiny(eng, job, 0, 0, n);
            if (rc != 1) { eng->stats.shards = 1; eng->cells_counted = true; return rc; }      // (the results carried their cell counts)
        }
    }
    if (int rc = zero_cells(eng)) return rc;
    static const bool deal = getenv("BSW_MULTI") && std::string(getenv("BSW_MULTI")) == "deal";
    eng->stats.shards = 1;
    if (ndev == 1 || deal) return run_pipeline(eng, job, 0, ndev, 0, n, chunk_pairs, false);
    if (n < (int64_t)ndev * CHUNK_MIN) return run_pipeline(eng, job, 0, 1, 0, n, chunk_pairs, false);   // too small to split
    eng->stats.shards = ndev;
    // cost curve from a sample (every step-th pair), cut at equal cost
    const int64_t step = std::max<int64_t>(1, n / 8192);
    const int64_t ns = (n + step - 1) / step;
    std::vector<double> cum((size_t)ns + 1, 0.0);
    for (int64_t k = 0; k < ns; ++k) {
        const int64_t i = k * step;
        int l1, l2;
        if (job.pb) { l1 = job.pb->desc[i].len1; l2 = job.pb->desc[i].len2; }
        else { l1 = job.pairs[i].len1; l2 = job.pairs[i].len2; }
        l1 = std::min(std::max(l1, 1), 32767); l2 = std::min(std::max(l2, 1), 32767);
        cum[(size_t)k + 1] = cum[(size_t)k] + pair_cost(l1, l2, eng->w);
    }
    std::vector<int64_t> begin((size_t)ndev + 1, 0);
    begin[(size_t)ndev] = n;
    for (int g = 1; g < ndev; ++g) {
        const double target = cum[(size_t)ns] * (double)g / (double)ndev;
        const int64_t k = std::lower_bound(cum.begin(), cum.end(), target) - cum.begin();
        begin[(size_t)g] = std::min(n, std::max(begin[(size_t)g - 1], (k * step) & ~(int64_t)63));
    }
    struct Shard { bsw_stats stats; std::string err; int rc = BSW_OK; };
    std::vector<Shard> shards((size_t)ndev);
    auto work = [&](int g) {
        Shard& sh = shards[(size_t)g];
        memset(&sh.stats, 0, sizeof(sh.stats));
        t_stats = &sh.stats; t_err = &sh.err;
        const int64_t a = begin[(size_t)g], m = begin[(size_t)g + 1] - a;
        if (m > 0) sh.rc = run_pipeline(eng, job, g, 1, a, m, chunk_pairs, false);
        if (sh.rc != BSW_OK) { cudaSetDevice(eng->devs[(size_t)g].dev); cudaDeviceSynchronize(); }
        t_stats = nullptr; t_err = nullptr;
    };
    std::vector<std::thread> threads;
    for (int g = 1; g < ndev; ++g) threads.emplace_back(work, g);
    work(0);
    for (std::thread& t : threads) t.join();
    bsw_stats& S = eng->stats;
    int rc = BSW_OK;
    double ms_kernel = 0;
    for (const Shard& sh : shards) {
        if (sh.rc != BSW_OK && rc == BSW_OK) { rc = sh.rc; eng->err = sh.err; }
        S.cells_nominal += sh.stats.cells_nominal; S.kernel_launches += sh.stats.kernel_launches;
        S.h2d_bytes += sh.stats.h2d_bytes; S.d2h_bytes += sh.stats.d2h_bytes;
        S.ms_pack += sh.stats.ms_pack; S.ms_scatter += sh.stats.ms_scatter;
        S.n_short += sh.stats.n_short; S.n_long += sh.stats.n_long;
        S.partitioned |= sh.stats.partitioned;
        ms_kernel = std::max(ms_kernel, sh.stats.ms_kernel);      // the devices run side by side
    }
    S.ms_kernel += ms_kernel;
    return rc;
}

int collect_cells(bsw_engine* eng)
{
    for (DevCtx& c : eng->devs) {
        CUDA_TRY(cudaSetDevice(c.dev));
        CUDA_TRY(cudaMemcpy(c.h_cells, c.d_cells, sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        eng->stats.cells_effective += (int64_t)*c.h_cells;
    }
    return BSW_OK;
}

void quiesce(bsw_engine* eng)
{
    for (DevCtx& c : eng->devs) { cudaSetDevice(c.dev); cudaDeviceSynchronize(); }
}

} // namespace

extern "C" {

const char* bsw_version(void) { return "bsw_b200 0.3 sm_100a"; }

void bsw_default_params(bsw_params* p)
{
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->o_del = p->o_ins = 6; p->e_del = p->e_ins = 1;   // main_banded.cpp:51-52
    p->zdrop = 100; p->end_bonus = 5;                   // main_banded.cpp:250
    p->match = 1; p->mismatch = 4; p->ambig = -1;       // main_banded.cpp:49-50,53
    p->zdrop_mode = BSW_ZDROP_VECTOR;
}

const char* bsw_last_error(const bsw_engine* eng)
{
    if (eng) return eng->err.c_str();
    std::lock_guard<std::mutex> g(g_err_mutex);
    static thread_local std::string copy;
    copy = g_create_error;
    return copy.c_str();
}

bsw_engine* bsw_create(const bsw_params* params, int* err)
{
    auto fail = [&](int code, const std::string& msg) -> bsw_engine* {
        { std::lock_guard<std::mutex> g(g_err_mutex); g_create_error = msg; }
        if (err) *err = code;
        return nullptr;
    };
    if (!params) return fail(BSW_ERR_PARAM, "params == NULL");
    std::string why;
    if (validate_params(params, why) != BSW_OK) return fail(BSW_ERR_PARAM, why);

    // One hardware queue per stream the pipeline keeps busy (6 chunk streams + 16 DP streams + the
    // H2D stream): with the default of 8 connections, streams share queues and a prep kernel of one
    // chunk waits behind another chunk's result copy.  Only effective if this is the process's
    // first CUDA call; a caller that initialises CUDA earlier exports the variable itself.
    // (set once per process: engines may be created from concurrent threads -- the C++ class creates its engine
    // lazily inside the driver's OpenMP region -- and setenv is not thread-safe)
    static std::once_flag env_once;
    std::call_once(env_once, [] { setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0); });
    int ndev_avail = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev_avail);
    if (ce != cudaSuccess || ndev_avail < 1)
        return fail(BSW_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(ce) +
                                  " (this engine has no CPU fallback)");
    bsw_engine* eng = new bsw_engine();
    eng->p = *params;
    KParams& k = eng->kp;
    k.match = params->match; k.mismatch_neg = -params->mismatch; k.ambig = params->ambig;
    k.o_del = params->o_del; k.e_del = params->e_del; k.o_ins = params->o_ins; k.e_ins = params->e_ins;
    k.oe_del = k.o_del + k.e_del; k.oe_ins = k.o_ins + k.e_ins;
    k.zdrop = params->zdrop; k.end_bonus = params->end_bonus; k.zmode = params->zdrop_mode;
    k.mx = std::max(std::max(k.match, k.mismatch_neg), k.ambig);
    k.w = 0; k.kone = 1;
    eng->pool.reset(new ThreadPool(auto_threads(params->host_threads)));
    eng->use16 = params->short_variant == BSW_SHORT_PACKED16;
    eng->short_max = params->long_min_qlen > 0 ? std::min(params->long_min_qlen - 1, SHORT_MAX_QLEN) : SHORT_MAX_QLEN;
    memset(&eng->stats, 0, sizeof(eng->stats));

    std::vector<int> ids;
    if (params->n_devices == 0) { int cur = 0; cudaGetDevice(&cur); ids.push_back(cur); }
    else for (int i = 0; i < params->n_devices; ++i) ids.push_back(params->devices[i]);
    for (int id : ids)
        if (id < 0 || id >= ndev_avail) { bsw_destroy(eng); return fail(BSW_ERR_PARAM, "device ordinal out of range"); }
    eng->devs.resize(ids.size());
    for (size_t i = 0; i < ids.size(); ++i) {
        DevCtx& c = eng->devs[i];
        c.dev = ids[i];
        bool ok = cudaSetDevice(c.dev) == cudaSuccess;
        cudaDeviceProp prop{};
        ok = ok && cudaGetDeviceProperties(&prop, c.dev) == cudaSuccess;
        if (ok && prop.major != 10) {
            bsw_destroy(eng);                                  // releases the streams / events of the devices set up so far
            return fail(BSW_ERR_CUDA, std::string("device ") + prop.name +
                                      " is not sm_100: this library carries sm_100a code only");
        }
        c.sms = prop.multiProcessorCount;
        for (int s = 0; ok && s < NSTREAMS; ++s) {
            int prio_lo = 0, prio_hi = 0;
            cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
            ok = cudaStreamCreateWithPriority(&c.cs[s], cudaStreamNonBlocking, prio_lo) == cudaSuccess;
            ok = ok && cudaEventCreateWithFlags(&c.ev_join[s], cudaEventDisableTiming) == cudaSuccess;
        }
        if (ok) {
            int prio_lo = 0, prio_hi = 0;
            cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
            ok = cudaStreamCreateWithPriority(&c.h2d, cudaStreamNonBlocking, prio_hi) == cudaSuccess;
        }
        if (ok) setup_partitions(c);
        ok = ok && cudaEventCreate(&c.ev_t0) == cudaSuccess && cudaEventCreate(&c.ev_t1) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&c.ev_res, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventRecord(c.ev_res, c.h2d) == cudaSuccess;
        ok = ok && cudaMalloc((void**)&c.d_cells, sizeof(unsigned long long)) == cudaSuccess;
        ok = ok && cudaHostAlloc((void**)&c.h_cells, sizeof(unsigned long long), cudaHostAllocDefault) == cudaSuccess;
        if (!ok) {
            std::string m = std::string("device setup failed: ") + cudaGetErrorString(cudaGetLastError());
            bsw_destroy(eng);
            return fail(BSW_ERR_CUDA, m);
        }
    }
    if (err) *err = BSW_OK;
    return eng;
}

static void bsw_global_release(bsw_engine* eng);      // bsw_global.inl
static void bsw_chain_release(bsw_engine* eng);       // bsw_chain.inl
static void bsw_async_release(bsw_engine* eng);       // bsw_async.inl
static void bsw_extend32_release(bsw_engine* eng);    // bsw_extend32.inl
static void bsw_global32_release(bsw_engine* eng);    // bsw_global32.inl
static void bsw_reg2aln_release(bsw_engine* eng);     // bsw_reg2aln.inl

void bsw_destroy(bsw_engine* eng)
{
    if (!eng) return;
    bsw_async_release(eng);
    bsw_global_release(eng);
    bsw_chain_release(eng);
    bsw_extend32_release(eng);
    bsw_global32_release(eng);
    bsw_reg2aln_release(eng);
    for (DevCtx& c : eng->devs) {
        cudaSetDevice(c.dev);
        cudaDeviceSynchronize();
        for (Slot& s : c.slots) slot_destroy(s);
        for (int s = 0; s < NSTREAMS; ++s) {
            if (c.cs[s]) cudaStreamDestroy(c.cs[s]);
            if (c.cs_part[s]) cudaStreamDestroy(c.cs_part[s]);
            if (c.ev_join[s]) cudaEventDestroy(c.ev_join[s]);
        }
        if (c.h2d) cudaStreamDestroy(c.h2d);
        if (c.g_svc) green_api().destroy(c.g_svc);
        if (c.g_dp) green_api().destroy(c.g_dp);
        if (c.ev_t0) cudaEventDestroy(c.ev_t0);
        if (c.ev_t1) cudaEventDestroy(c.ev_t1);
        if (c.ev_res) cudaEventDestroy(c.ev_res);
        release(c.rawq); release(c.rawr); release(c.allq); release(c.allr);
        if (c.d_cells) cudaFree(c.d_cells);
        if (c.h_cells) cudaFreeHost(c.h_cells);
    }
    delete eng;
}

int bsw_get_stats(const bsw_engine* eng, bsw_stats* out)
{
    if (!eng || !out) return BSW_ERR_PARAM;
    *out = eng->stats;
    return BSW_OK;
}

// ------------------------------------------------------------------------------------------
// the hot path: host buffers in, results in place
// ------------------------------------------------------------------------------------------
int bsw_extend(bsw_engine* eng, SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer,
               int64_t n, int32_t w)
{
    if (!eng) return BSW_ERR_PARAM;
    const double t_begin = now_ms();
    if (int rc = begin_batch(eng, pairs, seq_ref, seq_qer, n, w)) return rc;
    if (n == 0) return BSW_OK;
    Job job;
    job.pairs = pairs; job.seq_ref = seq_ref; job.seq_qer = seq_qer;
    int rc = run_sharded(eng, job, n, CHUNK_EXTEND);
    if (rc == BSW_RETRY_STAGED) {
        // page-locked buffers whose pairs address sequences 2^30 bytes or more apart inside one chunk (shuffled pair
        // order over large buffers): the staged route gathers the bytes on the host and has no such limit
        quiesce(eng);
        bsw_stats& S = eng->stats;
        memset(&S, 0, sizeof(S));
        S.pairs = n;
        eng->err.clear();
        job.force_staged = true;
        rc = run_sharded(eng, job, n, CHUNK_EXTEND);
    }
    if (rc != BSW_OK) { quiesce(eng); return rc; }
    if (!eng->cells_counted) if (int rc2 = collect_cells(eng)) return rc2;
    eng->stats.ms_total = now_ms() - t_begin;
    return BSW_OK;
}

// ------------------------------------------------------------------------------------------
// the hot path for a loader that emits the packed layout: 2 bits per base + 16-byte descriptors in,
// the six result fields out
// ------------------------------------------------------------------------------------------
static int extend_packed(bsw_engine* eng, const bsw_packed_batch* b, int32_t w, void* out, bool out16)
{
    if (!eng) return BSW_ERR_PARAM;
    const double t_begin = now_ms();
    eng->err.clear();
    eng->staged = false; eng->ran = false;
    if (!b || b->n_pairs < 0 || w < 0 || (b->n_pairs > 0 && (!b->desc || !out)) ||
        b->q2_words < 0 || b->r2_words < 0 || b->raw_q_bytes < 0 || b->raw_r_bytes < 0 ||
        (b->q2_words > 0 && !b->q2) || (b->r2_words > 0 && !b->r2) || (b->raw_q_bytes > 0 && !b->raw_q) ||
        (b->raw_r_bytes > 0 && !b->raw_r)) {
        eng->err = "bsw_extend_packed: bad arguments";
        return BSW_ERR_PARAM;
    }
    if (b->n_pairs > 0x7fffffff || b->q2_words > 0xffffffffll || b->r2_words > 0xffffffffll ||
        b->raw_q_bytes > 0x7fffffffll || b->raw_r_bytes > 0x7fffffffll) {
        eng->err = "bsw_extend_packed: batch too large (2^31-1 pairs, 2^32-1 words, 2^31-1 RAW bytes per side)";
        return BSW_ERR_PARAM;
    }
    bsw_stats& S = eng->stats;
    memset(&S, 0, sizeof(S));
    S.pairs = b->n_pairs;
    eng->n = b->n_pairs; eng->w = w; eng->kp.w = w;
    if (b->n_pairs == 0) return BSW_OK;
    Job job;
    job.pb = b; job.out = out; job.out16 = out16;
    const int rc = run_sharded(eng, job, b->n_pairs, CHUNK_EXTEND);
    if (rc != BSW_OK) {
        if (rc == BSW_ERR_DOMAIN)
            eng->err = "bsw_extend_packed: descriptor outside the domain: need 1<=len1,len2<=32767, h0>=0, h0+len2*match<=32767, "
                       "offsets inside the batch's buffers, and queries the engine routes to the byte-reading kernels "
                       "(longer than BSW_PACKED_MAX_QLEN or bsw_params.long_min_qlen) stored RAW";
        quiesce(eng);
        return rc;
    }
    if (int rc2 = collect_cells(eng)) return rc2;
    eng->stats.ms_total = now_ms() - t_begin;
    return BSW_OK;
}

int bsw_extend_packed(bsw_engine* eng, const bsw_packed_batch* batch, int32_t w, OutScore* out)
{
    return extend_packed(eng, batch, w, out, false);
}

int bsw_extend_packed16(bsw_engine* eng, const bsw_packed_batch* batch, int32_t w, bsw_score16* out)
{
    return extend_packed(eng, batch, w, out, true);
}

// ------------------------------------------------------------------------------------------
// band-doubling retry (tools/bwa/bwamem.c:723-753, :770-800), batched: the pairs that neither
// repeated their score nor stayed within 3/4 of the band are gathered and re-run with w << t
// ------------------------------------------------------------------------------------------
typedef int (*ExtendFn)(bsw_engine*, SeqPair*, const uint8_t*, const uint8_t*, int64_t, int32_t);

// the retry loop over one extension entry point (bsw_extend, or bsw_extend32 for bsw_extend_chains' long flanks);
// arguments validated by the caller
static int extend_retry_with(ExtendFn extend, bsw_engine* eng, SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer,
                             int64_t n, int32_t w, int32_t max_try, const int32_t* prev_score, int32_t* band_used)
{
    if (int rc = extend(eng, pairs, seq_ref, seq_qer, n, w)) return rc;
    bsw_stats total = eng->stats;
    std::vector<int64_t> active, next;
    std::vector<int32_t> prev;
    std::vector<SeqPair> sub;
    for (int64_t i = 0; i < n; ++i) {
        if (band_used) band_used[i] = w;
        const int32_t p0 = prev_score ? prev_score[i] : -1;
        if (!(pairs[i].score == p0 || pairs[i].max_off < (w >> 1) + (w >> 2))) { active.push_back(i); prev.push_back(pairs[i].score); }
    }
    for (int t = 1; t < max_try && !active.empty(); ++t) {
        const int32_t wt = w << t;
        sub.resize(active.size());
        for (size_t k = 0; k < active.size(); ++k) sub[k] = pairs[active[k]];
        if (int rc = extend(eng, sub.data(), seq_ref, seq_qer, (int64_t)sub.size(), wt)) return rc;
        total.cells_effective += eng->stats.cells_effective; total.kernel_launches += eng->stats.kernel_launches;
        total.h2d_bytes += eng->stats.h2d_bytes; total.d2h_bytes += eng->stats.d2h_bytes;
        total.ms_kernel += eng->stats.ms_kernel; total.ms_pack += eng->stats.ms_pack; total.ms_scatter += eng->stats.ms_scatter;
        next.clear();
        std::vector<int32_t> nprev;
        for (size_t k = 0; k < active.size(); ++k) {
            const int64_t i = active[k];
            SeqPair& d = pairs[i]; const SeqPair& r = sub[k];
            d.score = r.score; d.tle = r.tle; d.gtle = r.gtle; d.qle = r.qle; d.gscore = r.gscore; d.max_off = r.max_off;
            if (band_used) band_used[i] = wt;
            if (!(r.score == prev[k] || r.max_off < (wt >> 1) + (wt >> 2))) { next.push_back(i); nprev.push_back(r.score); }
        }
        active.swap(next); prev.swap(nprev);
    }
    total.ms_total = 0;
    total.pairs = n;
    eng->stats = total;
    eng->n = n;
    return BSW_OK;
}

int bsw_extend_retry(bsw_engine* eng, SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer,
                     int64_t n, int32_t w, int32_t max_try, const int32_t* prev_score, int32_t* band_used)
{
    if (!eng) return BSW_ERR_PARAM;
    if (max_try < 1 || max_try > 8 || w < 0 || ((int64_t)w << (max_try - 1)) > 0x3fffffff) {
        eng->err = "bsw_extend_retry: max_try must be in 1..8 and w << (max_try - 1) must fit";
        return BSW_ERR_PARAM;
    }
    return extend_retry_with(bsw_extend, eng, pairs, seq_ref, seq_qer, n, w, max_try, prev_score, band_used);
}

#include "bsw_extend32.inl"
#include "bsw_chain.inl"
#include "bsw_global.inl"
#include "bsw_global32.inl"
#include "bsw_reg2aln.inl"
#include "bsw_async.inl"

// ------------------------------------------------------------------------------------------
// resident form: stage (host -> HBM, packed + bucketed), run (DP kernels only, repeatable),
// fetch (results -> SeqPair[])
// ------------------------------------------------------------------------------------------
int bsw_stage(bsw_engine* eng, const SeqPair* pairs, const uint8_t* seq_ref, const uint8_t* seq_qer,
              int64_t n, int32_t w)
{
    if (!eng) return BSW_ERR_PARAM;
    const double t_begin = now_ms();
    if (int rc = begin_batch(eng, pairs, seq_ref, seq_qer, n, w)) return rc;
    eng->staged_chunks.clear();
    if (n > 0) {
        if (int rc = zero_cells(eng)) return rc;
        Job job;
        job.pairs = const_cast<SeqPair*>(pairs); job.seq_ref = seq_ref; job.seq_qer = seq_qer;
        static const int64_t env_stage = getenv("BSW_STAGE_CHUNK") ? atoll(getenv("BSW_STAGE_CHUNK")) : 0;     // experiments
        int rc = run_pipeline(eng, job, 0, (int)eng->devs.size(), 0, n, env_stage > 0 ? env_stage : CHUNK_STAGE, true);
        if (rc == BSW_RETRY_STAGED) {
            quiesce(eng);
            job.force_staged = true;
            eng->stats.cells_nominal = 0; eng->stats.h2d_bytes = 0; eng->stats.kernel_launches = 0;
            rc = run_pipeline(eng, job, 0, (int)eng->devs.size(), 0, n, env_stage > 0 ? env_stage : CHUNK_STAGE, true);
        }
        if (rc != BSW_OK) { quiesce(eng); return rc; }
    }
    eng->staged = true;
    eng->stats.ms_total = now_ms() - t_begin;
    return BSW_OK;
}

int bsw_run_staged(bsw_engine* eng)
{
    if (!eng) return BSW_ERR_PARAM;
    if (!eng->staged) { eng->err = "bsw_run_staged before bsw_stage"; return BSW_ERR_STATE; }
    bsw_stats& S = eng->stats;
    S.kernel_launches = 0; S.ms_kernel = 0; S.cells_effective = 0;
    // device timeline per GPU: ev_t0 on cs[0] -> every chunk's launches -> joined back -> ev_t1
    for (DevCtx& c : eng->devs) {
        CUDA_TRY(cudaSetDevice(c.dev));
        CUDA_TRY(cudaMemsetAsync(c.d_cells, 0, sizeof(unsigned long long), c.cs[0]));
        CUDA_TRY(cudaStreamSynchronize(c.cs[0]));
        CUDA_TRY(cudaEventRecord(c.ev_t0, c.cs[0]));
    }
    for (auto& ds : eng->staged_chunks) {
        DevCtx& c = eng->devs[(size_t)ds.first]; Slot& s = c.slots[(size_t)ds.second];
        CUDA_TRY(cudaSetDevice(c.dev));
        CUDA_TRY(cudaStreamWaitEvent(s.st, c.ev_t0, 0));
        if (int rc = launch_dp(eng, c, s)) return rc;
        if (int rc = launch_bytes(eng, c, s)) return rc;
        CUDA_TRY(cudaEventRecord(s.ev_k1, s.st));
        CUDA_TRY(cudaStreamWaitEvent(c.cs[0], s.ev_k1, 0));
    }
    for (DevCtx& c : eng->devs) {
        CUDA_TRY(cudaSetDevice(c.dev));
        CUDA_TRY(cudaEventRecord(c.ev_t1, c.cs[0]));
    }
    for (DevCtx& c : eng->devs) {
        CUDA_TRY(cudaSetDevice(c.dev));
        CUDA_TRY(cudaEventSynchronize(c.ev_t1));
        float ms = 0; CUDA_TRY(cudaEventElapsedTime(&ms, c.ev_t0, c.ev_t1));
        S.ms_kernel = std::max(S.ms_kernel, (double)ms);
    }
    if (int rc = collect_cells(eng)) return rc;
    eng->ran = true;
    return BSW_OK;
}

int bsw_fetch(bsw_engine* eng, SeqPair* pairs, int64_t n)
{
    if (!eng) return BSW_ERR_PARAM;
    if (!eng->ran) { eng->err = "bsw_fetch before bsw_run_staged"; return BSW_ERR_STATE; }
    if (n != eng->n || (n > 0 && !pairs)) { eng->err = "bsw_fetch: pair count differs from the staged batch"; return BSW_ERR_PARAM; }
    bsw_stats& S = eng->stats;
    S.d2h_bytes = 0; S.ms_d2h = 0; S.ms_scatter = 0;
    const bool pinned_out = n > 0 && is_pinned(pairs);
    for (auto& ds : eng->staged_chunks) {
        DevCtx& c = eng->devs[(size_t)ds.first]; Slot& s = c.slots[(size_t)ds.second];
        CUDA_TRY(cudaSetDevice(c.dev));
        s.out_records = pinned_out && s.direct && s.out_records;      // the record DMA needs the chunk's device copy
        if (!s.out_records) if (int rc = ensure(eng, s.res, (size_t)s.n, true)) return rc;
        Job job;
        job.pairs = pairs;
        if (int rc = output_chunk(eng, c, s, job)) return rc;
    }
    for (auto& ds : eng->staged_chunks) {
        DevCtx& c = eng->devs[(size_t)ds.first]; Slot& s = c.slots[(size_t)ds.second];
        CUDA_TRY(cudaSetDevice(c.dev));
        CUDA_TRY(cudaEventSynchronize(s.ev_out));
        unpack_chunk(eng, s, pairs);
    }
    return BSW_OK;
}

// ------------------------------------------------------------------------------------------
// pinned host memory for callers without a CUDA toolchain
// ------------------------------------------------------------------------------------------
void* bsw_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocMapped) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void bsw_host_free(void* p) { if (p) cudaFreeHost(p); }

int bsw_host_register(void* p, size_t bytes)
{
    if (!p || !bytes) return BSW_ERR_PARAM;
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped) != cudaSuccess) {
        cudaGetLastError();
        return BSW_ERR_CUDA;
    }
    return BSW_OK;
}

int bsw_host_unregister(void* p)
{
    if (!p) return BSW_ERR_PARAM;
    if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return BSW_ERR_CUDA; }
    return BSW_OK;
}

double bsw_measure_int_peak(bsw_engine* eng)
{
    if (!eng || eng->devs.empty()) return 0.0;
    DevCtx& c = eng->devs[0];
    if (cudaSetDevice(c.dev) != cudaSuccess) return 0.0;
    const int threads = 256, blocks = c.sms * 8, iters = 4096;
    int* d_out = nullptr;
    if (cudaMalloc((void**)&d_out, sizeof(int) * (size_t)threads * blocks) != cudaSuccess) return 0.0;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0, c.cs[0]);
        bsw_int_peak_kernel<<<blocks, threads, 0, c.cs[0]>>>(d_out, iters, 12345 + rep);
        cudaEventRecord(e1, c.cs[0]);
        if (cudaStreamSynchronize(c.cs[0]) != cudaSuccess) { best = 0.0; break; }
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
        const double ops = (double)threads * blocks * (double)iters * 64.0;
        if (rep > 0 && ms > 0) best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d_out);
    return best;
}

} // extern "C"
