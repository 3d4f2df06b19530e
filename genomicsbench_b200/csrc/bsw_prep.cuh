// bsw_prep.cuh -- device-side batch preparation of the bsw engine (sm_100a).
//
// Stands in for the host-side batch wrapper of the reference, smithWatermanBatchWrapper16
// (benchmarks/bsw/bandedSWA.cpp:1150-1431: pad, sortPairsLen :368-403, AoS->SoA transpose,
// sortPairsId :405-420), re-thought for a GPU behind PCIe: the host only streams bytes (or
// nothing at all when the caller's buffers are pinned), and these kernels
//   bsw_scan_pairs   read the caller's 72-byte SeqPair records, validate the domain, emit the
//                    16-byte descriptor per pair and the chunk summary the host plans with
//   bsw_bucket_*     counting sort of the chunk by (len2, h0, len1) -> processing order perm[];
//                    lists the pairs too long for the short kernel
//   bsw_pack_pairs   2-bit pack query / reference bytes (16 bases per word) in processing order,
//                    flag and list the pairs with N (and those outside the packed kernel's domain)
//   bsw_writeback    unpack the 16-byte results into the caller's SeqPair records (input order)
//
// Every kernel here runs in blocks of PREP_BLOCK = 64 threads with little shared memory: they are
// launched on high-priority streams while DP kernels of earlier chunks fill the SMs to their
// register / shared-memory limit, and a block this small fits into the room ONE retiring DP block
// frees (a 256- or 1024-thread block would wait for the DP backlog to drain; BSW_TIMELINE showed
// the next chunk's preparation stuck behind it for half a millisecond).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/bsw.h"
#include "bsw_kernels.cuh"
#include "bsw_kernel16.cuh"

namespace bsw {

constexpr int LEN_HIST = 1024;        // len2 histogram bins 0..1022, 1023 = everything longer
constexpr int PREP_BLOCK = 64;        // threads per block of the prep kernels

// Chunk summary: written by bsw_scan_pairs / bsw_pack_pairs (or by the host pass for pageable
// buffers), read by the host to size buffers and to plan the launches.
struct ChunkInfo {
    unsigned long long min_r, max_r, min_q, max_q;   // byte extents [min, max) of the sequences, relative to base0
    unsigned long long nominal;                      // sum len1 * len2
    unsigned long long qbases, tbases;               // sum len2 / sum len1 of the chunk
    int mn[3], mx[3];                                // ranges of len2, h0, len1 (short pairs)
    int bad;                                         // pairs outside the domain
    int n_short;                                     // pairs with len2 <= short_max
    unsigned int n_nlist, n_llist;                   // pairs with N (short) / long pairs, listed for the byte kernels
    unsigned int qcursor, tcursor;                   // packed words handed out
    int qmax_n;                                      // longest query among the N pairs
    int qmax_all;                                    // longest query of the chunk
    int n_wide;                                      // packed route: 2-bit pairs outside the 16-bit kernel's score domain
    int far;                                         // direct route: valid pairs whose sequences lie 2^30 bytes or more from the chunk's first pair
    int pad_[2];
    unsigned int hist[LEN_HIST];                     // pairs per len2
};
static_assert(sizeof(ChunkInfo) % 16 == 0, "bsw_info_publish copies 16-byte words");

// The chunk summary is reset and handed to the host by two tiny kernels instead of copy-engine
// transfers: a 4 KB cudaMemcpyAsync queues behind the megabytes of sequence / result traffic of the
// other chunks (BSW_TIMELINE showed the DP launches of a chunk waiting 0.5 ms for it), stores from an
// SM into mapped page-locked memory do not.
__global__ void __launch_bounds__(PREP_BLOCK)
bsw_info_init(ChunkInfo* __restrict__ info)
{
    uint32_t* w = reinterpret_cast<uint32_t*>(info);
    for (int k = threadIdx.x; k < (int)(sizeof(ChunkInfo) / 4); k += blockDim.x) w[k] = 0u;
    __syncthreads();
    if (threadIdx.x == 0) {
        info->min_r = info->min_q = ~0ull;
        info->mn[0] = info->mn[1] = info->mn[2] = 0x7fffffff;
    }
}

// zeroes the bin table (same reason: a cudaMemsetAsync may be served by a copy engine that is busy)
__global__ void __launch_bounds__(PREP_BLOCK)
bsw_zero_words(uint4* __restrict__ p, int n16)
{
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n16; k += gridDim.x * blockDim.x) p[k] = make_uint4(0, 0, 0, 0);
}

__global__ void __launch_bounds__(PREP_BLOCK)
bsw_info_publish(const ChunkInfo* __restrict__ info, ChunkInfo* __restrict__ host_mapped)
{
    const uint4* src = reinterpret_cast<const uint4*>(info);
    uint4* dst = reinterpret_cast<uint4*>(host_mapped);
    for (int k = threadIdx.x; k < (int)(sizeof(ChunkInfo) / 16); k += blockDim.x) dst[k] = __ldcg(src + k);
    __threadfence_system();
}

__device__ __forceinline__ unsigned long long bsw_umin64(unsigned long long a, unsigned long long b) { return a < b ? a : b; }
__device__ __forceinline__ unsigned long long bsw_umax64(unsigned long long a, unsigned long long b) { return a > b ? a : b; }

// desc[i] = {query byte offset, reference byte offset (both relative to base0_q / base0_r, as
// signed 32-bit), len2 | len1 << 16, h0}.  info must be zeroed except mn[] = INT_MAX, min_* = ~0.
__global__ void __launch_bounds__(PREP_BLOCK)
bsw_scan_pairs(const SeqPair* __restrict__ pairs, int n, long long base0_r, long long base0_q,
               int match, int short_max, int4* __restrict__ desc, ChunkInfo* __restrict__ info)
{
    __shared__ unsigned int s_hist[LEN_HIST];
    __shared__ unsigned long long s_u64[7];       // min_r max_r min_q max_q nominal qbases tbases
    __shared__ int s_i[9];                        // mn[3] mx[3] bad n_short qmax_all
    for (int k = threadIdx.x; k < LEN_HIST; k += blockDim.x) s_hist[k] = 0;
    if (threadIdx.x < 7) s_u64[threadIdx.x] = (threadIdx.x == 0 || threadIdx.x == 2) ? ~0ull : 0ull;
    if (threadIdx.x < 9) s_i[threadIdx.x] = threadIdx.x < 3 ? 0x7fffffff : 0;
    __syncthreads();
    unsigned long long min_r = ~0ull, max_r = 0, min_q = ~0ull, max_q = 0, nominal = 0, qb = 0, tb = 0;
    int mn0 = 0x7fffffff, mn1 = 0x7fffffff, mn2 = 0x7fffffff, mx0 = 0, mx1 = 0, mx2 = 0, bad = 0, nshort = 0, qall = 0, far = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        // 72-byte record: idr@0 idq@8 len1@24 len2@28 h0@32 (bandedSWA.h:91-100)
        const long long* p64 = reinterpret_cast<const long long*>(pairs + i);
        const int* p32 = reinterpret_cast<const int*>(pairs + i);
        const long long idr = p64[0], idq = p64[1];
        const int len1 = p32[6], len2 = p32[7], h0 = p32[8];
        const long long dr = idr - base0_r, dq = idq - base0_q;
        const bool valid = len1 >= 1 && len1 <= 32767 && len2 >= 1 && len2 <= 32767 && h0 >= 0 &&
                           (long long)h0 + (long long)len2 * match <= 32767 && idr >= 0 && idq >= 0;
        const bool near = dr > -(1ll << 30) && dr < (1ll << 30) && dq > -(1ll << 30) && dq < (1ll << 30);
        if (!valid || !near) {
            // (a valid pair too far away for the 32-bit chunk-relative offsets: the call is re-run on the staged route)
            if (valid) far = 1; else bad = 1;
            desc[i] = make_int4(0, 0, 1 | (1 << 16), 1);
            continue;
        }
        desc[i] = make_int4((int)dq, (int)dr, len2 | (len1 << 16), h0);
        nominal += (unsigned long long)len1 * (unsigned long long)len2;
        const unsigned long long ur = (unsigned long long)(dr + (1ll << 30)), uq = (unsigned long long)(dq + (1ll << 30));
        min_r = bsw_umin64(min_r, ur); max_r = bsw_umax64(max_r, ur + len1);
        min_q = bsw_umin64(min_q, uq); max_q = bsw_umax64(max_q, uq + len2);
        atomicAdd(&s_hist[min(len2, LEN_HIST - 1)], 1u);
        qall = max(qall, len2);
        qb += len2; tb += len1;
        if (len2 <= short_max) {
            ++nshort;
            mn0 = min(mn0, len2); mx0 = max(mx0, len2);
            mn1 = min(mn1, h0);   mx1 = max(mx1, h0);
            mn2 = min(mn2, len1); mx2 = max(mx2, len1);
        }
    }
    // warp reductions first (shuffles), then one shared-memory atomic per warp and value: 64-bit
    // min / max atomics in shared memory are CAS loops, 256 threads on one address serialise badly
    const unsigned FULL = 0xffffffffu;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        min_r = bsw_umin64(min_r, __shfl_xor_sync(FULL, min_r, o)); max_r = bsw_umax64(max_r, __shfl_xor_sync(FULL, max_r, o));
        min_q = bsw_umin64(min_q, __shfl_xor_sync(FULL, min_q, o)); max_q = bsw_umax64(max_q, __shfl_xor_sync(FULL, max_q, o));
        nominal += __shfl_xor_sync(FULL, nominal, o); qb += __shfl_xor_sync(FULL, qb, o); tb += __shfl_xor_sync(FULL, tb, o);
    }
    mn0 = __reduce_min_sync(FULL, mn0); mn1 = __reduce_min_sync(FULL, mn1); mn2 = __reduce_min_sync(FULL, mn2);
    mx0 = __reduce_max_sync(FULL, mx0); mx1 = __reduce_max_sync(FULL, mx1); mx2 = __reduce_max_sync(FULL, mx2);
    bad = __reduce_max_sync(FULL, bad); nshort = __reduce_add_sync(FULL, nshort); qall = __reduce_max_sync(FULL, qall);
    far = __reduce_max_sync(FULL, far);
    if (far && (threadIdx.x & 31) == 0) atomicAdd(&info->far, 1);
    if ((threadIdx.x & 31) == 0) {
        atomicMin(&s_u64[0], min_r); atomicMax(&s_u64[1], max_r);
        atomicMin(&s_u64[2], min_q); atomicMax(&s_u64[3], max_q);
        atomicAdd(&s_u64[4], nominal); atomicAdd(&s_u64[5], qb); atomicAdd(&s_u64[6], tb);
        atomicMin(&s_i[0], mn0); atomicMin(&s_i[1], mn1); atomicMin(&s_i[2], mn2);
        atomicMax(&s_i[3], mx0); atomicMax(&s_i[4], mx1); atomicMax(&s_i[5], mx2);
        if (bad) atomicAdd(&s_i[6], 1);
        atomicAdd(&s_i[7], nshort);
        atomicMax(&s_i[8], qall);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < LEN_HIST; k += blockDim.x)
        if (s_hist[k]) atomicAdd(&info->hist[k], s_hist[k]);
    if (threadIdx.x == 0) {
        atomicMin(&info->min_r, s_u64[0]); atomicMax(&info->max_r, s_u64[1]);
        atomicMin(&info->min_q, s_u64[2]); atomicMax(&info->max_q, s_u64[3]);
        atomicAdd(&info->nominal, s_u64[4]); atomicAdd(&info->qbases, s_u64[5]); atomicAdd(&info->tbases, s_u64[6]);
        atomicMin(&info->mn[0], s_i[0]); atomicMin(&info->mn[1], s_i[1]); atomicMin(&info->mn[2], s_i[2]);
        atomicMax(&info->mx[0], s_i[3]); atomicMax(&info->mx[1], s_i[4]); atomicMax(&info->mx[2], s_i[5]);
        if (s_i[6]) atomicAdd(&info->bad, s_i[6]);
        atomicAdd(&info->n_short, s_i[7]);
        atomicMax(&info->qmax_all, s_i[8]);
    }
}

// Packed route (bsw_extend_packed): the chunk's descriptors arrive in the host format of include/bsw.h
// (bsw_pair_desc = {q_off, r_off, len2 | len1 << 16, h0 | flags << 16} read as one int4), offsets absolute in the
// batch's buffers.  Validates them against the word ranges [qlo, qhi) / [rlo, rhi) that were copied for this chunk
// (RAW pairs: against the byte sizes of the raw buffers, resident as a whole) and builds the same summary as
// bsw_scan_pairs.  qbases / tbases count 16 bases per packed word (they size the gathered word arrays).
struct PackedRange {
    unsigned int qlo, qhi, rlo, rhi;          // words
    unsigned int rawq, rawr;                  // bytes
};

__global__ void __launch_bounds__(PREP_BLOCK)
bsw_scan_packed(const int4* __restrict__ desc, int n, const __grid_constant__ PackedRange R, int match, int short_max,
                int packed16, ChunkInfo* __restrict__ info)
{
    __shared__ unsigned int s_hist[LEN_HIST];
    for (int k = threadIdx.x; k < LEN_HIST; k += blockDim.x) s_hist[k] = 0;
    __syncthreads();
    unsigned long long nominal = 0, qb = 0, tb = 0;
    int mn0 = 0x7fffffff, mn1 = 0x7fffffff, mn2 = 0x7fffffff, mx0 = 0, mx1 = 0, mx2 = 0, bad = 0, nshort = 0, qall = 0, nwide = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int4 d = desc[i];
        const int len2 = d.z & 0xffff, len1 = (d.z >> 16) & 0xffff, h0 = d.w & 0xffff;
        const bool raw = ((d.w >> 16) & BSW_PAIR_RAW) != 0;
        const unsigned int qo = (unsigned int)d.x, ro = (unsigned int)d.y;
        bool ok = len1 >= 1 && len1 <= 32767 && len2 >= 1 && len2 <= 32767 && h0 >= 0 && h0 + len2 * match <= 32767;
        if (raw) ok = ok && (unsigned long long)qo + len2 <= R.rawq && (unsigned long long)ro + len1 <= R.rawr;
        else ok = ok && len2 <= short_max && qo >= R.qlo && (unsigned long long)qo + ((len2 + 15) >> 4) <= R.qhi &&
                  ro >= R.rlo && (unsigned long long)ro + ((len1 + 15) >> 4) <= R.rhi;
        if (!ok) { bad = 1; continue; }
        nominal += (unsigned long long)len1 * (unsigned long long)len2;
        atomicAdd(&s_hist[min(len2, LEN_HIST - 1)], 1u);
        qall = max(qall, len2);
        if (!raw) { qb += (unsigned)((len2 + 15) >> 4) * 16u; tb += (unsigned)((len1 + 15) >> 4) * 16u; }
        if (len2 <= short_max) {
            ++nshort;
            mn0 = min(mn0, len2); mx0 = max(mx0, len2);
            mn1 = min(mn1, h0);   mx1 = max(mx1, h0);
            mn2 = min(mn2, len1); mx2 = max(mx2, len1);
            if (!raw && packed16 && !k16::eligible(match, len2, h0)) ++nwide;
        }
    }
    const unsigned FULL = 0xffffffffu;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        nominal += __shfl_xor_sync(FULL, nominal, o); qb += __shfl_xor_sync(FULL, qb, o); tb += __shfl_xor_sync(FULL, tb, o);
    }
    mn0 = __reduce_min_sync(FULL, mn0); mn1 = __reduce_min_sync(FULL, mn1); mn2 = __reduce_min_sync(FULL, mn2);
    mx0 = __reduce_max_sync(FULL, mx0); mx1 = __reduce_max_sync(FULL, mx1); mx2 = __reduce_max_sync(FULL, mx2);
    bad = __reduce_max_sync(FULL, bad); nshort = __reduce_add_sync(FULL, nshort); qall = __reduce_max_sync(FULL, qall);
    nwide = __reduce_add_sync(FULL, nwide);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&info->nominal, nominal); atomicAdd(&info->qbases, qb); atomicAdd(&info->tbases, tb);
        atomicMin(&info->mn[0], mn0); atomicMin(&info->mn[1], mn1); atomicMin(&info->mn[2], mn2);
        atomicMax(&info->mx[0], mx0); atomicMax(&info->mx[1], mx1); atomicMax(&info->mx[2], mx2);
        if (bad) atomicAdd(&info->bad, 1);
        if (nshort) atomicAdd(&info->n_short, nshort);
        if (nwide) atomicAdd(&info->n_wide, nwide);
        atomicMax(&info->qmax_all, qall);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < LEN_HIST; k += blockDim.x)
        if (s_hist[k]) atomicAdd(&info->hist[k], s_hist[k]);
}

// 16 base codes (one per byte) at any alignment -> one 2-bit word.  *bad collects codes > 3.
// `room` = bytes of the sequence from src on: the word-wise path may touch up to 3 bytes past its
// 16 and is only taken when they still belong to the sequence (the buffer may be host memory
// that ends with it).
// `overread` = the bytes behind the sequence may be read (device copy with slack behind it): the last,
// partial word of a sequence then takes the word-wise path too, with the bytes past nb masked off --
// otherwise every sequence ends in a byte loop that half the warp waits for.
__device__ __forceinline__ uint32_t bsw_pack16(const uint8_t* src, int nb, int room, uint32_t& bad, bool overread)
{
    uint32_t out = 0;
    if (room >= 20 || overread) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(src);
        const uint32_t* aw = reinterpret_cast<const uint32_t*>(a & ~(uintptr_t)3);
        const unsigned sh = (unsigned)(a & 3) * 8u;
        uint32_t w[5];
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = __ldg(aw + k);
        w[4] = sh ? __ldg(aw + 4) : 0u;              // never reads past the 16 bytes when aligned
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t v = __funnelshift_r(w[k], w[k + 1], sh);
            const int valid = nb - 4 * k;                 // bytes of this word that belong to the sequence
            if (valid < 4) v = valid <= 0 ? 0u : v & ((1u << (8 * valid)) - 1u);
            bad |= v & 0xFCFCFCFCu;
            v &= 0x03030303u;
            v = (v | (v >> 6)) & 0x000F000Fu;
            v = (v | (v >> 12)) & 0xFFu;
            out |= v << (8 * k);
        }
    } else {
        for (int k = 0; k < nb; ++k) {
            const uint32_t c = __ldg(src + k);
            bad |= c & 0xFCu;
            out |= (c & 3u) << (2 * k);
        }
    }
    return out;
}

// One warp packs the pairs at 32 consecutive positions of the processing order (perm[]), so that
// the DP kernel later reads descriptors and sequences of neighbouring threads from neighbouring
// addresses.  The word counts are scanned across the warp, one atomicAdd per sequence kind
// reserves the output range, then the lanes sweep the concatenated word list (lane -> word, pair
// found by binary search), so loads stay coalesced for short and long sequences alike.  The output
// range is reserved once per block tile (two atomics on the chunk's cursors per block).
// meta[s] (processing order) gets word offsets; desc[i] (input order) keeps byte offsets.
// The sources are one byte per base (the staged and direct routes); the packed route's 2-bit words are read in
// place by the DP kernels and never pass through here.
__global__ void __launch_bounds__(PREP_BLOCK)
bsw_pack_pairs(const int4* __restrict__ desc, const uint32_t* __restrict__ perm, int n_sorted,
               const uint8_t* __restrict__ qraw, const uint8_t* __restrict__ rraw, int4* __restrict__ meta,
               uint32_t* __restrict__ qpk, uint32_t* __restrict__ tpk,
               uint32_t* __restrict__ nlist, ChunkInfo* __restrict__ info, int packed16_match, int overread)
{
    constexpr int NW = PREP_BLOCK / 32;
    __shared__ uint32_t s_pre[NW][2][33];
    __shared__ uint32_t s_bad[NW][32];
    __shared__ int4 s_desc[NW][32];
    __shared__ uint32_t s_tot[NW][2], s_base[NW][2];
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    for (int tile = blockIdx.x * PREP_BLOCK; tile < n_sorted; tile += gridDim.x * PREP_BLOCK) {
        const int s = tile + wib * 32 + lane;
        int4 d = make_int4(0, 0, 0, 0);
        int len2 = 0, len1 = 0, pi = 0;
        if (s < n_sorted) {
            pi = (int)perm[s];
            d = desc[pi];
            len2 = d.z & 0xffff; len1 = (d.z >> 16) & 0xffff;
        }
        s_desc[wib][lane] = d;
        const uint32_t nq = (uint32_t)(len2 + 15) >> 4;
        const uint32_t nt = (uint32_t)(len1 + 15) >> 4;
        uint32_t pq = nq, pt = nt;                  // inclusive warp scans
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t a = __shfl_up_sync(FULL, pq, o), b = __shfl_up_sync(FULL, pt, o);
            if (lane >= o) { pq += a; pt += b; }
        }
        const uint32_t totq = __shfl_sync(FULL, pq, 31), tott = __shfl_sync(FULL, pt, 31);
        if (lane == 0) { s_tot[wib][0] = totq; s_tot[wib][1] = tott; }
        __syncthreads();
        if (threadIdx.x < 2) {                      // thread 0: query words, thread 1: reference words
            uint32_t sum = 0;
#pragma unroll
            for (int k = 0; k < NW; ++k) { s_base[k][threadIdx.x] = sum; sum += s_tot[k][threadIdx.x]; }
            const uint32_t b0 = atomicAdd(threadIdx.x ? &info->tcursor : &info->qcursor, sum);
#pragma unroll
            for (int k = 0; k < NW; ++k) s_base[k][threadIdx.x] += b0;
        }
        __syncthreads();
        const uint32_t bq = s_base[wib][0], bt = s_base[wib][1];
        s_pre[wib][0][lane + 1] = pq; s_pre[wib][1][lane + 1] = pt;
        if (lane == 0) { s_pre[wib][0][0] = 0; s_pre[wib][1][0] = 0; }
        s_bad[wib][lane] = 0;
        __syncwarp();
#pragma unroll
        for (int kind = 0; kind < 2; ++kind) {
            const uint32_t tot = kind ? tott : totq;
            const uint32_t* pre = s_pre[wib][kind];
            for (uint32_t wv = lane; wv < tot; wv += 32) {
                int lo = 0;                          // largest p with pre[p] <= wv
#pragma unroll
                for (int step = 16; step > 0; step >>= 1)
                    if (pre[lo + step] <= wv) lo += step;
                const int4 dd = s_desc[wib][lo];
                const uint32_t wi = wv - pre[lo];
                const int len = kind ? (dd.z >> 16) & 0xffff : dd.z & 0xffff;
                const uint8_t* src = (kind ? rraw + dd.y : qraw + dd.x) + 16 * (int)wi;
                uint32_t bad = 0;
                const int room = len - 16 * (int)wi;
                const uint32_t word = bsw_pack16(src, min(16, room), room, bad, overread != 0);
                (kind ? tpk + bt : qpk + bq)[wv] = word;
                if (bad) atomicOr(&s_bad[wib][lo], 1u);
            }
        }
        __syncwarp();
        if (s < n_sorted) {
            // pairs for the 32-bit byte kernel: those that contain N and, when the packed 16-bit kernel
            // runs the rest (packed16_match = its match score), those outside its score domain
            const bool has_n = s_bad[wib][lane] != 0 ||
                               (packed16_match > 0 && !k16::eligible(packed16_match, len2, d.w & 0xffff));
            meta[s] = make_int4((int)(bq + pq - nq), (int)(bt + pt - nt), d.z, (d.w & 0xffff) | (has_n ? BSW_META_NFLAG : 0));
            if (has_n) { nlist[atomicAdd(&info->n_nlist, 1u)] = (uint32_t)pi; atomicMax(&info->qmax_n, len2); }
        }
        __syncthreads();                            // s_tot / s_base / s_desc are reused by the next tile
    }
}

// ---- bucketing: counting sort by the compressed key (len2 | len1 | h0) >> drop --------------
struct BucketKey {
    int mn2, mnh, mn1;        // minima of len2, h0, len1
    int b_h0, b_l1;           // bit widths of the h0 and len1 fields (after their shifts)
    int s_h0, s_l1;           // low bits dropped from h0 - mnh / len1 - mn1 so that the key fits the bin table
    int short_max;
};

__device__ __forceinline__ uint32_t bsw_bucket_of(const BucketKey& K, const int4 d)
{
    const uint32_t len2 = d.z & 0xffff, len1 = (d.z >> 16) & 0xffff, h0 = d.w & 0xffff;
    const uint32_t a = (h0 - K.mnh) >> K.s_h0, b = (len1 - K.mn1) >> K.s_l1;
    return ((len2 - K.mn2) << (K.b_h0 + K.b_l1)) | (b << K.b_h0) | a;
}

// rank[i] = arrival order of pair i inside its bin; bins[] accumulates the bin sizes; pairs whose
// query is too long for the short kernel are listed for the warp-per-pair kernel instead
__global__ void __launch_bounds__(PREP_BLOCK)
bsw_bucket_count(const int4* __restrict__ desc, int n, const __grid_constant__ BucketKey K,
                 uint32_t* __restrict__ bins, uint32_t* __restrict__ rank,
                 uint32_t* __restrict__ llist, ChunkInfo* __restrict__ info)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int4 d = desc[i];
        if ((d.z & 0xffff) > K.short_max) { llist[atomicAdd(&info->n_llist, 1u)] = (uint32_t)i; continue; }
        rank[i] = atomicAdd(&bins[bsw_bucket_of(K, d)], 1u);
    }
}

// Exclusive prefix sum of the bin table in two levels, one launch.  Every block scans one tile of
// 1024 bins in place (64 threads x 16 bins) and leaves the tile total; the block that finishes last
// (a ticket counter behind the totals, zeroed with the bin table) scans the <= 256 tile totals.
// The scatter adds the two levels.
constexpr int SCAN_TILE = 1024;
constexpr int SCAN_MAX_TILES = 256;

__global__ void __launch_bounds__(PREP_BLOCK)
bsw_bucket_scan(uint32_t* __restrict__ bins, int nbins, uint32_t* __restrict__ totals, unsigned int* __restrict__ ticket)
{
    constexpr int PER = SCAN_TILE / PREP_BLOCK;         // 16 bins per thread
    __shared__ uint32_t s_warp[PREP_BLOCK / 32];
    __shared__ bool s_last;
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int base = blockIdx.x * SCAN_TILE + threadIdx.x * PER;
    uint32_t v[PER];
    uint32_t mine = 0;
#pragma unroll
    for (int k = 0; k < PER; k += 4) {
        const uint4 q = base + k < nbins ? *reinterpret_cast<const uint4*>(bins + base + k) : make_uint4(0, 0, 0, 0);   // nbins is a power of two >= 1; the table is padded
        v[k] = q.x; v[k + 1] = q.y; v[k + 2] = q.z; v[k + 3] = q.w;
        mine += q.x + q.y + q.z + q.w;
    }
    uint32_t inc = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(FULL, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) s_warp[wib] = inc;
    __syncthreads();
    uint32_t wbase = 0;
    for (int k = 0; k < wib; ++k) wbase += s_warp[k];
    uint32_t run = wbase + inc - mine;
#pragma unroll
    for (int k = 0; k < PER; ++k) {
        const uint32_t t = v[k];
        v[k] = run;
        run += t;
    }
#pragma unroll
    for (int k = 0; k < PER; k += 4)
        if (base + k < nbins) *reinterpret_cast<uint4*>(bins + base + k) = make_uint4(v[k], v[k + 1], v[k + 2], v[k + 3]);
    if (threadIdx.x == PREP_BLOCK - 1) {
        totals[blockIdx.x] = run;
        __threadfence();
        s_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // second level: exclusive scan of the tile totals, 4 per thread
    const int ntiles = (int)gridDim.x;
    uint32_t t4[4];
    uint32_t sum4 = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int idx = threadIdx.x * 4 + k;
        t4[k] = idx < ntiles ? __ldcg(totals + idx) : 0u;
        sum4 += t4[k];
    }
    uint32_t inc2 = sum4;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(FULL, inc2, o);
        if (lane >= o) inc2 += y;
    }
    __syncthreads();
    if (lane == 31) s_warp[wib] = inc2;
    __syncthreads();
    uint32_t run2 = inc2 - sum4;
    for (int k = 0; k < wib; ++k) run2 += s_warp[k];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int idx = threadIdx.x * 4 + k;
        if (idx < ntiles) totals[idx] = run2;
        run2 += t4[k];
    }
}

// PACKED (packed route): the sequences stay where the host packed them -- the DP kernels read them in place -- so
// the scatter also writes the processing-order descriptor meta[pos] = {query word, reference word (relative to the
// chunk's first word), len2 | len1 << 16, h0}; RAW pairs get BSW_META_NFLAG and are listed for the byte kernel.
template <bool PACKED>
__global__ void __launch_bounds__(PREP_BLOCK)
bsw_bucket_scatter(const int4* __restrict__ desc, int n, const __grid_constant__ BucketKey K,
                   const uint32_t* __restrict__ bins, const uint32_t* __restrict__ totals,
                   const uint32_t* __restrict__ rank, uint32_t* __restrict__ perm,
                   int4* __restrict__ meta = nullptr, uint32_t* __restrict__ nlist = nullptr,
                   ChunkInfo* __restrict__ info = nullptr, unsigned int q_word_lo = 0, unsigned int r_word_lo = 0)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int4 d = desc[i];
        if ((d.z & 0xffff) > K.short_max) continue;
        const uint32_t b = bsw_bucket_of(K, d);
        const uint32_t pos = bins[b] + totals[b / SCAN_TILE] + rank[i];
        perm[pos] = (uint32_t)i;
        if (PACKED) {
            const bool raw = ((d.w >> 16) & BSW_PAIR_RAW) != 0;
            meta[pos] = make_int4((int)((uint32_t)d.x - q_word_lo), (int)((uint32_t)d.y - r_word_lo), d.z,
                                  (d.w & 0xffff) | (raw ? BSW_META_NFLAG : 0));
            if (raw) { nlist[atomicAdd(&info->n_nlist, 1u)] = (uint32_t)i; atomicMax(&info->qmax_n, d.z & 0xffff); }
        }
    }
}

// res[i] (8 x int16) -> the six int32 result fields of the caller's record i (score@44 tle@48
// gtle@52 qle@56 gscore@60 max_off@64, bandedSWA.h:91-100); pairs may be host-mapped memory.
__global__ void __launch_bounds__(PREP_BLOCK)
bsw_writeback(const int4* __restrict__ res, int n, SeqPair* __restrict__ pairs)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int4 v = res[i];
        int* out = reinterpret_cast<int*>(pairs + i) + 11;
        out[0] = (int)(short)(v.x & 0xffff);        // score
        out[1] = (int)(short)(v.y & 0xffff);        // tle
        out[2] = (int)(short)(v.y >> 16);           // gtle
        out[3] = (int)(short)(v.x >> 16);           // qle
        out[4] = (int)(short)(v.z & 0xffff);        // gscore
        out[5] = (int)(short)(v.z >> 16);           // max_off
    }
}

// packed route: res[i] -> OutScore[i] (bandedSWA.h:103-107: score tle gtle qle gscore max_off), 24 bytes per pair
__global__ void __launch_bounds__(PREP_BLOCK)
bsw_out_scores(const int4* __restrict__ res, int n, int2* __restrict__ out)
{
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int4 v = res[i];
        int2* o = out + 3 * (size_t)i;
        o[0] = make_int2((int)(short)(v.x & 0xffff), (int)(short)(v.y & 0xffff));     // score, tle
        o[1] = make_int2((int)(short)(v.y >> 16), (int)(short)(v.x >> 16));           // gtle, qle
        o[2] = make_int2((int)(short)(v.z & 0xffff), (int)(short)(v.z >> 16));        // gscore, max_off
    }
}

} // namespace bsw
