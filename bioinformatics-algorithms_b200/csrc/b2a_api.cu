// b2a_api.cu -- C ABI (include/b2align.h) over the sm_100a kernels.
//
// Host side of the batch boundary that replaces the loop hw2.cpp:328-338.  A batch is cut into
// SEGMENTS of consecutive pairs.  Per segment the host (1) queues the host->device copy of the
// segment's sequence bytes, (2) plans it while the copy is in flight: pairs of identical shape are
// zipped into pair-pairs (the two 16-bit halves of the s16x2 kernels) and grouped by rows-per-lane,
// (3) queues the fill + traceback kernels of every RUN of the batch (one mode each: -g, -l) on the
// next of several record lanes.  Nothing in that loop waits for the device: the pattern alphabet of
// a segment is discovered by device kernels and stays on the device (AlphaInfo, per-pair-pair
// `dirty` flags), the DP record of a lane is reused by a later launch, so the copy of segment k+1
// overlaps the kernels of segment k and the record footprint is a few segments, not the batch.
// Pair-pairs whose patterns hold a fifth symbol are served by the 8-symbol variant of the s16x2
// kernel; pairs the s16x2 record cannot hold (long patterns, wide scores, > 7 pattern symbols) are
// collected and served afterwards by the wide32 family, and those whose wide32 record would not fit
// in memory by checkpointed recomputation (wide_ckpt_run).
// No CPU alignment code lives here: if CUDA is unavailable every compute entry point fails.
#include <cuda_runtime.h>
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/b2align.h"
#include "b2a_format.h"
#include "short16_fill.cuh"
#include "traceback.cuh"
#include "wide32.cuh"
#include "affine32.cuh"
#include "microbench.cuh"

using namespace b2a;

static_assert(sizeof(PairResult) == sizeof(b2a_result) && sizeof(b2a_result) == 32, "result record layout");
static_assert(B2A_OP_M == OP_M && B2A_OP_D == OP_D && B2A_OP_I == OP_I, "op codes");

namespace {

template <class T>
struct DevBuf {                                   // grow-only device buffer, reused across batches
    T* p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc((void**)&p, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
template <class T>
struct HostBuf {                                  // grow-only pinned host buffer (sources of async copies)
    T* p = nullptr; size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFreeHost(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaHostAlloc((void**)&p, std::max<size_t>(n, 1) * sizeof(T), cudaHostAllocDefault);
        if (e == cudaSuccess) cap = n;
        return e;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

struct ClassRange { int R; uint32_t first, count, max_n; };   // first: pair-pair index inside its segment

struct Segment {
    uint64_t first = 0, count = 0;                // pairs [first, first + count)
    uint64_t pp_first = 0, n_pp = 0;              // slice of the batch-wide pair-pair arrays
    uint64_t chunks = 0, rowbest_words = 0;       // record size of the segment
    uint64_t n_wide = 0;                          // pairs of the segment planned for wide32
    std::vector<ClassRange> classes;
};

struct Lane {                                     // one DP record, reused by every n_lanes-th (segment, run) launch
    DevBuf<Chunk> codes;
    DevBuf<uint32_t> rowbest;
    cudaEvent_t tb_done = nullptr;                // last traceback that read this record
    cudaStream_t s_tb = nullptr;                  // the lane's traceback stream (high priority): tracebacks of different lanes run concurrently
    cudaStream_t s_tb_lo = nullptr;               // the same at the fill's priority: used when there are >= 3 lanes (see batch_prepare)
};

// host-side state of the wide32 family for the current batch
struct WideState {
    std::vector<WidePair> pairs;
    std::vector<WideTask> tasks;
    uint64_t chunks = 0, bound_words = 0, rowbest_words = 0;
    uint32_t epoch = 0;                           // boundary-entry tags carry it, so stale entries of earlier launches never validate
    int K = 32;
    bool alpha4 = false, store = true;
    DevBuf<WidePair> d_pairs;
    DevBuf<WideTask> d_tasks;
    DevBuf<Chunk> d_codes;
    DevBuf<uint64_t> d_bound;                     // tagged boundary entries (wide32.cuh)
    DevBuf<int32_t> d_final, d_final_col;         // per wide pair: H at the end cell; semi-global mode: also its column j*
    DevBuf<uint32_t> d_rowbest, d_progress;       // d_progress[0] is the ticket counter
    // pairs whose full record would exceed the budget: score pass with checkpoint rows, then band groups re-filled bottom-up (wide_ckpt_run)
    struct CkptSpec { uint32_t pair, m, n; uint64_t pat_off, txt_off; };
    std::vector<CkptSpec> ckpt_pairs;
    DevBuf<int32_t> d_ck;
    DevBuf<CkptWalk> d_walk;
    // epoch tag of the next launch; the boundary buffer is cleared when it was reallocated or the 12-bit epoch wraps
    cudaError_t next_epoch(uint64_t need_words, cudaStream_t st, uint32_t* tag) {
        const size_t cap_before = d_bound.cap;
        cudaError_t e = d_bound.reserve(need_words);
        if (e != cudaSuccess) return e;
        epoch = (epoch + 1u) & 0xFFFu;
        // a reallocation may hand back the same address with uncleared memory behind the old end
        if (d_bound.cap != cap_before || epoch == 0u) {
            epoch = 1u;
            e = cudaMemsetAsync(d_bound.p, 0, d_bound.cap * sizeof(uint64_t), st);
        }
        *tag = epoch << 20;
        return e;
    }
    void release() {
        d_pairs.release(); d_tasks.release(); d_codes.release(); d_bound.release(); d_final.release(); d_final_col.release();
        d_rowbest.release(); d_progress.release(); d_ck.release(); d_walk.release();
    }
};

// What differs between the runs of one batch (b2a_align_batch_multi: same pairs, same scoring, another mode): the outputs.
// Inputs, segments and the pair-pair plan are shared.
struct RunBuf {
    int32_t mode = B2A_MODE_GLOBAL;
    DevBuf<PairResult> d_results;
    DevBuf<uint32_t> d_ops;
    DevBuf<int4> d_endcell;                       // local mode: end cell per pair, written by the short16 fill epilogue
    void release() { d_results.release(); d_ops.release(); d_endcell.release(); }
};

constexpr int MAX_LANES = 8;
constexpr int MAX_RUNS = B2A_MAX_RUNS;
constexpr size_t DIRTY_CLASSES = 16;              // >= classes (distinct rows-per-lane values) of one segment
constexpr uint64_t SEG_MIN_PAIRS = 2048;          // a segment is never closed below this many pairs

} // namespace

struct b2a_ctx {
    int device = 0;
    int sm_count = 0;
    bool tb_low = false;                          // tracebacks at the fill's stream priority (chosen per batch with the lane count)
    int lanes_cfg = 0;                            // B2A_OPT_LANES / B2A_LANES: 0 = automatic (2, or 8 for small batches, see batch_prepare)
    int n_lanes = 2;                              // DP records the launches alternate over: the traceback of one launch (its lane's s_tb) overlaps
                                                  // the fill of segment k+1 (s_fill); end to end 61.8 -> 59.1 ms per 1 M pairs NW+SW
    bool trace = false;                           // B2A_TRACE=1: per-segment timeline of b2a_align_batch on stderr
    uint64_t seg_budget_bytes = 8ull << 30;       // record bytes per segment (B2A_SEG_MB overrides)
    // Segments of b2a_align_batch.  16 k pairs, then doubling up to 128 k (the kernels start after a short copy; swept in
    // scripts/seg_e2e_sweep.py: every schedule between 58.3 and 60.0 ms for 1 M pairs).
    uint64_t seg_max_pairs = 131072;              // B2A_SEG_PAIRS / B2A_OPT_SEG_PAIRS override
    uint64_t seg_first_pairs = 1ull << 14;        // B2A_SEG_FIRST / B2A_OPT_SEG_FIRST override
    bool seg_user = false;                        // the caller set the schedule: take it literally
    uint64_t seg_resident_pairs = 1ull << 20;     // pairs per segment of b2a_batch_upload / b2a_batch_run ...
    uint64_t seg_resident_bytes = 60ull << 30;    // ... and its record bytes (a 1 M-pair batch with 4-bit deltas would need 110 GB)
    // s_fill runs the fill kernels back to back; every lane has its own traceback stream, so the latency-bound
    // walks of earlier launches fill the issue slots the ALU-bound fill of the current one leaves idle
    cudaStream_t s_copy = nullptr, s_down = nullptr, s_fill = nullptr;
    Lane lanes[MAX_LANES];
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    std::vector<cudaEvent_t> ev_pool;             // per segment: ready, fill start, fill end, traceback end
    std::string err;

    // batch state
    bool have_batch = false, ran = false;
    bool affine_ops = false;                      // the last call was b2a_affine_align_batch: d_ops / d_nops hold its op lists
    b2a_params prm{};                             // scoring + flags of the batch; prm.mode = mode of run 0
    RunBuf run[MAX_RUNS];
    uint32_t n_runs = 1, sel_run = 0;             // sel_run: the run b2a_fetch_ops / b2a_copy_ops / b2a_batch_download read
    uint32_t* ops_sink[MAX_RUNS] = {};            // b2a_set_ops_sink: host buffers the op words of run r are copied to segment by segment
    uint32_t ops_sink_runs = 0;
    uint64_t ops_sink_cap = 0;
    uint64_t n_launched = 0;                      // (segment, run) launches so far: they alternate over the lanes
    uint64_t n_pairs = 0;
    int K = 0;
    uint64_t wide_ckpt_bytes = 48ull << 30;       // a wide32 pair whose traceback record would be larger is walked from checkpoints instead
    uint64_t wide_ckpt_group_bytes = 1ull << 30;  // ... re-filling groups of bands whose record fits this
    uint32_t wide_ckpt_col_shift = 13;            // ... cut into tiles at every 2^13-th column, which the score pass keeps too
    std::vector<Segment> segs;
    std::vector<uint32_t> wide_pairs;             // pairs served by the wide32 family
    uint64_t total_ops_words = 0, n_pp_total = 0;
    uint64_t cells = 0, fill_bytes = 0, launches = 0, h2d = 0, d2h = 0;
    float last_fill_ms = 0, last_tb_ms = 0, last_total_ms = 0;

    DevBuf<uint8_t> d_pat, d_txt;
    DevBuf<uint64_t> d_pat_off, d_txt_off, d_code_off, d_ops_off;
    DevBuf<PPDesc> d_pps;
    DevBuf<uint32_t> d_nops;                      // affine only
    DevBuf<AlphaInfo> d_alpha;                    // one per segment + one for the whole batch (wide32)
    DevBuf<uint32_t> d_hist;                      // 256 pattern-byte counts per segment
    DevBuf<uint8_t> d_dirty;                      // per pair-pair: a pattern byte outside the segment's 4 table symbols -> wide32 serves its pairs
    HostBuf<uint8_t> h_dirty;
    DevBuf<uint32_t> d_dirty_list, d_dirty_cnt;   // per class of a segment: its flagged pair-pairs, compacted (dirty_compact_kernel); DIRTY_CLASSES counters per segment
    // compact input (b2a_seq2): the codes and exception lists as they arrive, [0] patterns, [1] texts; expanded into d_pat / d_txt
    struct Seq2Dev { DevBuf<uint8_t> codes, ebyte; DevBuf<uint64_t> epos; void release() { codes.release(); ebyte.release(); epos.release(); } } seq2[2];
    HostBuf<PPDesc> h_pps;
    HostBuf<uint64_t> h_code_off, h_ops_off;
    HostBuf<AlphaInfo> h_alpha;
    size_t alpha_slots = 0;
    WideState wide;
};

namespace {

int fail(b2a_ctx* c, int code, const std::string& msg) { if (c) c->err = msg; return code; }
int cuda_fail(b2a_ctx* c, cudaError_t e, const char* where) {
    cudaGetLastError();                                   // a failed call (cudaMalloc: out of memory) leaves its code for the NEXT cudaGetLastError
    return fail(c, e == cudaErrorMemoryAllocation ? B2A_ERR_NOMEM : B2A_ERR_CUDA,
                std::string(where) + ": " + cudaGetErrorString(e));
}
#define CU(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call); } while (0)

// ---- compact input (b2a_seq2): expand 2-bit codes to the byte buffer the kernels read --------------------------------------------------
// One thread per 16-byte group of the OUTPUT (global group index, so the vector store is aligned whatever the segment's first byte is):
// one 32-bit load of 16 codes, four PRMTs against the alphabet word, one 16-byte store.  Groups that straddle the segment's ends store
// their bytes one by one: the neighbouring segment owns the rest (its bytes may already carry patched exceptions).  HBM-bound:
// 0.25 + 1 bytes of traffic per base.
__global__ void seq2_expand_kernel(const uint8_t* __restrict__ codes, uint8_t* __restrict__ out, uint64_t b0, uint64_t b1, uint32_t alphabet) {
    const uint64_t g = b0 / 16 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t p = g * 16;
    if (p >= b1) return;
    const uint32_t w = *reinterpret_cast<const uint32_t*>(codes + g * 4);
    uint32_t v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t x = (w >> (8 * k)) & 0xFFu;                         // four codes -> four PRMT selector nibbles
        const uint32_t sel = (x & 3u) | ((x & 0xCu) << 2) | ((x & 0x30u) << 4) | ((x & 0xC0u) << 6);
        v[k] = __byte_perm(alphabet, 0u, sel);
    }
    if (p >= b0 && p + 16 <= b1) { *reinterpret_cast<uint4*>(out + p) = make_uint4(v[0], v[1], v[2], v[3]); return; }
#pragma unroll
    for (int k = 0; k < 16; ++k)
        if (p + k >= b0 && p + k < b1) out[p + k] = (uint8_t)(v[k >> 2] >> (8 * (k & 3)));
}
// ... and put the listed exceptions back
__global__ void seq2_patch_kernel(uint8_t* __restrict__ out, const uint64_t* __restrict__ pos, const uint8_t* __restrict__ byte, uint64_t n) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n) out[pos[e]] = byte[e];
}

// Histogram of the pattern bytes of a segment: hist[256] += counts of the bytes in [p, p+n)
__global__ void alphabet_kernel(const uint8_t* __restrict__ p, uint64_t n, uint32_t* __restrict__ hist) {
    __shared__ uint32_t s[256];
    for (int k = threadIdx.x; k < 256; k += blockDim.x) s[k] = 0;
    __syncthreads();
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t b = p[i];
        // the lanes of a warp mostly hold the same few symbols: one atomic per distinct symbol and warp
        const uint32_t peers = __match_any_sync(__activemask(), b);
        if ((uint32_t)(__ffs(peers) - 1) == (threadIdx.x & 31u)) atomicAdd(&s[b], (uint32_t)__popc(peers));
    }
    __syncthreads();
    for (int k = threadIdx.x; k < 256; k += blockDim.x) if (s[k]) atomicAdd(&hist[k], s[k]);
}
// histogram -> presence mask + the (<= 4) MOST FREQUENT symbols, which the PRMT score tables are built for.  too_many = the segment
// holds other pattern bytes as well (an 'N' in a read): the pair-pairs that contain one are flagged by dirty_kernel and served by wide32.
__global__ void alphabet_finish_kernel(AlphaInfo* __restrict__ info, const uint32_t* __restrict__ hist) {
    if (threadIdx.x != 0) return;
    uint32_t cnt[4] = {0, 0, 0, 0};
    uint8_t sym[4] = {0, 0, 0, 0};
    int present = 0;
    for (int w = 0; w < 8; ++w) info->mask[w] = 0;
    for (int b = 0; b < 256; ++b) {
        const uint32_t h = hist[b];
        if (!h) continue;
        ++present;
        info->mask[b >> 5] |= 1u << (b & 31);
        for (int c = 0; c < 4; ++c)
            if (h > cnt[c]) {                                  // insert into the top-4 (ties: lower byte value first)
                for (int k = 3; k > c; --k) { cnt[k] = cnt[k - 1]; sym[k] = sym[k - 1]; }
                cnt[c] = h; sym[c] = (uint8_t)b;
                break;
            }
    }
    for (int c = 0; c < 4; ++c) info->sym[c] = sym[c];
    info->nsym = present < 4 ? present : 4;
    info->too_many = present > 4;
}
// dirty[pp] = 1 iff a pattern of pair-pair pp holds a byte outside the segment's four table symbols (runs only when there is one)
__global__ void dirty_kernel(const uint8_t* __restrict__ pat, const uint64_t* __restrict__ pat_off, const PPDesc* __restrict__ pps, uint32_t n_pp,
                             const AlphaInfo* __restrict__ info, uint8_t* __restrict__ dirty) {
    if (!info->too_many) return;                               // uniform: nothing to flag (the flags were cleared by the host)
    const uint32_t pp = blockIdx.x * blockDim.x + threadIdx.x;
    if (pp >= n_pp) return;
    const int nsym = info->nsym;
    const uint8_t s0 = info->sym[0], s1 = info->sym[1], s2 = info->sym[2], s3 = info->sym[3];
    const PPDesc d = pps[pp];
    bool bad = false;
    for (int half = 0; half < 2 && !bad; ++half) {
        if (half && d.b == d.a) break;
        const uint8_t* p = pat + pat_off[half ? d.b : d.a];
        const uint32_t m = pp_dim(d.m, half);
        for (uint32_t i = 0; i < m; ++i) {
            const uint8_t x = p[i];
            if (!((nsym > 0 && x == s0) || (nsym > 1 && x == s1) || (nsym > 2 && x == s2) || (nsym > 3 && x == s3))) { bad = true; break; }
        }
    }
    dirty[pp] = bad ? 1 : 0;
}
// The flagged pair-pairs of one class, compacted: the 8-symbol kernel then runs FULL CTAs over list[0 .. *count) instead of one busy warp
// per CTA scattered over the class (0.1 % 'N' in 150-mers flags 26 % of the pair-pairs).  The order of the list is whatever the atomics
// give; every pair-pair keeps its own record, so results do not depend on it.
__global__ void dirty_compact_kernel(const uint8_t* __restrict__ dirty, uint32_t n_pp, const AlphaInfo* __restrict__ info,
                                     uint32_t* __restrict__ list, uint32_t* __restrict__ count) {
    if (!info->too_many) return;
    const uint32_t pp = blockIdx.x * blockDim.x + threadIdx.x;
    const bool flagged = pp < n_pp && dirty[pp] == 1;
    const uint32_t peers = __ballot_sync(0xFFFFFFFFu, flagged);
    if (!peers) return;
    uint32_t base = 0;
    if ((threadIdx.x & 31u) == 0u) base = atomicAdd(count, (uint32_t)__popc(peers));
    base = __shfl_sync(0xFFFFFFFFu, base, 0);
    if (flagged) list[base + (uint32_t)__popc(peers & ((1u << (threadIdx.x & 31u)) - 1u))] = pp;
}
void alpha_from_mask(AlphaInfo& a) {
    a.nsym = 0; a.too_many = 0;
    for (int c = 0; c < 4; ++c) a.sym[c] = 0;
    for (int b = 0; b < 256; ++b)
        if (a.mask[b >> 5] & (1u << (b & 31))) { if (a.nsym == 4) { a.too_many = 1; break; } a.sym[a.nsym++] = (uint8_t)b; }
}

// two launches per class: the 4-symbol kernel for the pair-pairs the segment's table symbols cover, the 8-symbol kernel for the flagged
// rest (its grid leaves at once when the segment has no fifth pattern symbol)
template <int R, int K>
cudaError_t launch_fill_rk(int mode, const FillArgs& a, cudaStream_t st) {
    const unsigned grid = (a.n_pp + FILL_WARPS - 1) / FILL_WARPS;
    const bool local = mode == B2A_MODE_LOCAL;
    if (mode == B2A_MODE_SEMIGLOBAL) {
        short16_fill_kernel<R, K, false, false, true><<<grid, FILL_WARPS * 32, 0, st>>>(a);
        short16_fill_kernel<R, K, false, true, true><<<grid, FILL_WARPS * 32, 0, st>>>(a);
    } else if (local) { short16_fill_kernel<R, K, true, false><<<grid, FILL_WARPS * 32, 0, st>>>(a); short16_fill_kernel<R, K, true, true><<<grid, FILL_WARPS * 32, 0, st>>>(a); }
    else { short16_fill_kernel<R, K, false, false><<<grid, FILL_WARPS * 32, 0, st>>>(a); short16_fill_kernel<R, K, false, true><<<grid, FILL_WARPS * 32, 0, st>>>(a); }
    return cudaGetLastError();
}
template <int K>
cudaError_t launch_fill_k(int R, int mode, const FillArgs& a, cudaStream_t st) {
    switch (R) {
        case 1: return launch_fill_rk<1, K>(mode, a, st);
        case 2: return launch_fill_rk<2, K>(mode, a, st);
        case 3: return launch_fill_rk<3, K>(mode, a, st);
        case 4: return launch_fill_rk<4, K>(mode, a, st);
        case 5: return launch_fill_rk<5, K>(mode, a, st);
        case 6: return launch_fill_rk<6, K>(mode, a, st);
        case 7: return launch_fill_rk<7, K>(mode, a, st);
        case 8: return launch_fill_rk<8, K>(mode, a, st);
        case 10: return launch_fill_rk<10, K>(mode, a, st);
        case 12: return launch_fill_rk<12, K>(mode, a, st);
        case 16: return launch_fill_rk<16, K>(mode, a, st);
    }
    return cudaErrorInvalidValue;
}
cudaError_t launch_fill(int K, int R, int mode, const FillArgs& a, cudaStream_t st) {
    switch (K) {
        case 2: return launch_fill_k<2>(R, mode, a, st);
        case 4: return launch_fill_k<4>(R, mode, a, st);
        case 8: return launch_fill_k<8>(R, mode, a, st);
    }
    return cudaErrorInvalidValue;
}
// The per-thread walk lives on L1 hits (measured: any shared-memory carve-out costs 2-4x): ask for all of it.  Function attributes
// are per DEVICE, so every context sets them after its cudaSetDevice (b2a_create), not once per process.
void set_kernel_attributes() {
    cudaFuncSetAttribute(short16_traceback_kernel<2, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(short16_traceback_kernel<2, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(short16_traceback_kernel<4, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(short16_traceback_kernel<4, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(short16_traceback_kernel<8, false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(short16_traceback_kernel<8, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(short16_traceback_kernel<2, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(short16_traceback_kernel<4, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(short16_traceback_kernel<8, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaGetLastError();
}
cudaError_t launch_tb(int K, int mode, const TbArgs& a, cudaStream_t st) {
    const unsigned threads = TB_THREADS, grid = (2u * a.n_pp + threads - 1) / threads;
    if (mode == B2A_MODE_SEMIGLOBAL) {
        switch (K) {
            case 2: short16_traceback_kernel<2, false, true><<<grid, threads, 0, st>>>(a); break;
            case 4: short16_traceback_kernel<4, false, true><<<grid, threads, 0, st>>>(a); break;
            case 8: short16_traceback_kernel<8, false, true><<<grid, threads, 0, st>>>(a); break;
            default: return cudaErrorInvalidValue;
        }
        return cudaGetLastError();
    }
    switch (K * 2 + (mode == B2A_MODE_LOCAL ? 1 : 0)) {
        case 4:  short16_traceback_kernel<2, false><<<grid, threads, 0, st>>>(a); break;
        case 5:  short16_traceback_kernel<2, true><<<grid, threads, 0, st>>>(a); break;
        case 8:  short16_traceback_kernel<4, false><<<grid, threads, 0, st>>>(a); break;
        case 9:  short16_traceback_kernel<4, true><<<grid, threads, 0, st>>>(a); break;
        case 16: short16_traceback_kernel<8, false><<<grid, threads, 0, st>>>(a); break;
        case 17: short16_traceback_kernel<8, true><<<grid, threads, 0, st>>>(a); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

inline int chunk_steps(int K) { return 3 * (16 / K); }

// ---------------------------------------------------------------------------------------------
// wide32 family: host planning and launches
// ---------------------------------------------------------------------------------------------
template <int K, bool LOCAL, bool STORE>
cudaError_t launch_wide_fill_a(bool alpha4, const WideArgs& a, unsigned grid, cudaStream_t st) {
    if (alpha4) wide32_fill_kernel<K, LOCAL, STORE, true><<<grid, WIDE_WARPS * 32, 0, st>>>(a);
    else wide32_fill_kernel<K, LOCAL, STORE, false><<<grid, WIDE_WARPS * 32, 0, st>>>(a);
    return cudaGetLastError();
}
template <int K>
cudaError_t launch_wide_fill_k(bool local, bool store, bool alpha4, const WideArgs& a, unsigned grid, cudaStream_t st) {
    if (store) return local ? launch_wide_fill_a<K, true, true>(alpha4, a, grid, st) : launch_wide_fill_a<K, false, true>(alpha4, a, grid, st);
    if (K != 2) return cudaErrorInvalidValue;                 // score-only kernels exist for K = 2 only
    return local ? launch_wide_fill_a<2, true, false>(alpha4, a, grid, st) : launch_wide_fill_a<2, false, false>(alpha4, a, grid, st);
}
// pass 1 of a checkpointed pair: score-only + kept columns
cudaError_t launch_wide_fill_keepcol(bool local, bool alpha4, const WideArgs& a, unsigned grid, cudaStream_t st) {
    if (local) { if (alpha4) wide32_fill_kernel<2, true, false, true, true><<<grid, WIDE_WARPS * 32, 0, st>>>(a);
                 else wide32_fill_kernel<2, true, false, false, true><<<grid, WIDE_WARPS * 32, 0, st>>>(a); }
    else       { if (alpha4) wide32_fill_kernel<2, false, false, true, true><<<grid, WIDE_WARPS * 32, 0, st>>>(a);
                 else wide32_fill_kernel<2, false, false, false, true><<<grid, WIDE_WARPS * 32, 0, st>>>(a); }
    return cudaGetLastError();
}
// semi-global: whole pairs only (no KEEPCOL pass, see wide_plan)
template <int K>
cudaError_t launch_wide_fill_semi_k(bool store, bool alpha4, const WideArgs& a, unsigned grid, cudaStream_t st) {
    if (!store && K != 2) return cudaErrorInvalidValue;        // score-only kernels exist for K = 2 only
    if (store) { if (alpha4) wide32_fill_kernel<K, false, true, true, false, true><<<grid, WIDE_WARPS * 32, 0, st>>>(a);
                 else wide32_fill_kernel<K, false, true, false, false, true><<<grid, WIDE_WARPS * 32, 0, st>>>(a); }
    else       { if (alpha4) wide32_fill_kernel<2, false, false, true, false, true><<<grid, WIDE_WARPS * 32, 0, st>>>(a);
                 else wide32_fill_kernel<2, false, false, false, false, true><<<grid, WIDE_WARPS * 32, 0, st>>>(a); }
    return cudaGetLastError();
}
cudaError_t launch_wide_fill_semi(int K, bool store, bool alpha4, const WideArgs& a, unsigned grid, cudaStream_t st) {
    switch (K) {
        case 2:  return launch_wide_fill_semi_k<2>(store, alpha4, a, grid, st);
        case 4:  return launch_wide_fill_semi_k<4>(store, alpha4, a, grid, st);
        case 8:  return launch_wide_fill_semi_k<8>(store, alpha4, a, grid, st);
        case 16: return launch_wide_fill_semi_k<16>(store, alpha4, a, grid, st);
        case 32: return launch_wide_fill_semi_k<32>(store, alpha4, a, grid, st);
    }
    return cudaErrorInvalidValue;
}
cudaError_t launch_wide_fill(int K, bool local, bool store, bool alpha4, const WideArgs& a, unsigned grid, cudaStream_t st) {
    switch (K) {
        case 2:  return launch_wide_fill_k<2>(local, store, alpha4, a, grid, st);
        case 4:  return launch_wide_fill_k<4>(local, store, alpha4, a, grid, st);
        case 8:  return launch_wide_fill_k<8>(local, store, alpha4, a, grid, st);
        case 16: return launch_wide_fill_k<16>(local, store, alpha4, a, grid, st);
        case 32: return launch_wide_fill_k<32>(local, store, alpha4, a, grid, st);
    }
    return cudaErrorInvalidValue;
}
cudaError_t launch_wide_tb(int K, int mode, const WideTbArgs& a, cudaStream_t st) {
    const unsigned threads = WIDE_TB_WARPS * 32, grid = (a.n_wide + WIDE_TB_WARPS - 1) / WIDE_TB_WARPS;
    if (mode == B2A_MODE_SEMIGLOBAL) {
        switch (K) {
            case 2:  wide32_traceback_kernel<2, false, true><<<grid, threads, 0, st>>>(a); break;
            case 4:  wide32_traceback_kernel<4, false, true><<<grid, threads, 0, st>>>(a); break;
            case 8:  wide32_traceback_kernel<8, false, true><<<grid, threads, 0, st>>>(a); break;
            case 16: wide32_traceback_kernel<16, false, true><<<grid, threads, 0, st>>>(a); break;
            case 32: wide32_traceback_kernel<32, false, true><<<grid, threads, 0, st>>>(a); break;
            default: return cudaErrorInvalidValue;
        }
        return cudaGetLastError();
    }
    switch (K * 2 + (mode == B2A_MODE_LOCAL ? 1 : 0)) {
        case 4:  wide32_traceback_kernel<2, false><<<grid, threads, 0, st>>>(a); break;
        case 5:  wide32_traceback_kernel<2, true><<<grid, threads, 0, st>>>(a); break;
        case 8:  wide32_traceback_kernel<4, false><<<grid, threads, 0, st>>>(a); break;
        case 9:  wide32_traceback_kernel<4, true><<<grid, threads, 0, st>>>(a); break;
        case 16: wide32_traceback_kernel<8, false><<<grid, threads, 0, st>>>(a); break;
        case 17: wide32_traceback_kernel<8, true><<<grid, threads, 0, st>>>(a); break;
        case 32: wide32_traceback_kernel<16, false><<<grid, threads, 0, st>>>(a); break;
        case 33: wide32_traceback_kernel<16, true><<<grid, threads, 0, st>>>(a); break;
        case 64: wide32_traceback_kernel<32, false><<<grid, threads, 0, st>>>(a); break;
        case 65: wide32_traceback_kernel<32, true><<<grid, threads, 0, st>>>(a); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

int wide_plan(b2a_ctx* ctx, const uint64_t* pat_off, const uint64_t* txt_off, bool store, bool alpha4, cudaStream_t st)
{
    WideState& W = ctx->wide;
    const b2a_params& prm = ctx->prm;
    W.pairs.clear(); W.tasks.clear(); W.ckpt_pairs.clear();
    W.chunks = W.bound_words = W.rowbest_words = 0;
    W.K = delta_bits_wide(prm.match, prm.mismatch, prm.gap);
    W.store = store;
    W.alpha4 = alpha4 && prm.match <= 127 && prm.match >= -128 && prm.mismatch <= 127 && prm.mismatch >= -128;
    const int CS = 2 * (32 / W.K);
    uint32_t max_bands = 0;
    for (uint32_t k : ctx->wide_pairs) {
        WidePair p{};
        p.pat_off = pat_off[k]; p.txt_off = txt_off[k];
        p.m = (uint32_t)(pat_off[k + 1] - pat_off[k]); p.n = (uint32_t)(txt_off[k + 1] - txt_off[k]);
        p.pair = k;
        p.nbands = (p.m && p.n) ? (p.m + 32u * WIDE_R - 1u) / (32u * WIDE_R) : 0u;
        p.top_off = WIDE_NO_TOP; p.left_off = WIDE_NO_TOP;
        if (p.nbands >= (1u << 20)) return fail(ctx, B2A_ERR_RANGE, "wide32: pattern too long (band index must fit 20 bits)");
        if (store && (uint64_t)p.nbands * WIDE_R * num_chunks(p.n, CS, wide_skew(W.K)) * 32u * sizeof(Chunk) > ctx->wide_ckpt_bytes) {
            // the checkpointed walk (wide_ckpt_run) has global and local borders only
            for (uint32_t r = 0; r < ctx->n_runs; ++r)
                if (ctx->run[r].mode == B2A_MODE_SEMIGLOBAL)
                    return fail(ctx, B2A_ERR_RANGE, "semi-global mode: a pair whose traceback record exceeds B2A_OPT_CKPT_BYTES (the checkpointed "
                                                    "path) is not supported; raise the option or align the pair in global or local mode");
            W.ckpt_pairs.push_back(WideState::CkptSpec{k, p.m, p.n, p.pat_off, p.txt_off});   // too large to keep: served one by one from checkpoints
            continue;
        }
        p.code_off = W.chunks;
        if (store) W.chunks += (uint64_t)p.nbands * WIDE_R * num_chunks(p.n, CS, wide_skew(W.K)) * 32u;
        p.bound_stride = ((p.n + 64u) + 31u) & ~31u;
        p.bound_off = W.bound_words; if (p.nbands > 1u) W.bound_words += 2ull * p.bound_stride;   // single-band pairs exchange nothing
        p.rowbest_off = W.rowbest_words; W.rowbest_words += (uint64_t)p.nbands * 32u * WIDE_R;
        max_bands = std::max(max_bands, p.nbands);
        W.pairs.push_back(p);
    }
    // ticket order: band-major, so the band a warp depends on always holds an earlier ticket
    std::vector<uint32_t> order(W.pairs.size());
    for (uint32_t i = 0; i < order.size(); ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return W.pairs[a].nbands > W.pairs[b].nbands; });
    for (uint32_t b = 0; b < max_bands; ++b)
        for (uint32_t i : order) { if (W.pairs[i].nbands <= b) break; W.tasks.push_back(WideTask{i, b}); }
    CU(W.d_pairs.reserve(W.pairs.size())); CU(W.d_tasks.reserve(W.tasks.size()));
    CU(W.d_codes.reserve(W.chunks)); CU(W.d_final.reserve(W.pairs.size())); CU(W.d_final_col.reserve(W.pairs.size()));
    CU(W.d_rowbest.reserve(W.rowbest_words)); CU(W.d_progress.reserve(1));
    // the vectors outlive the copies: every caller synchronises `st` before the next batch touches them
    if (!W.pairs.empty()) CU(cudaMemcpyAsync(W.d_pairs.p, W.pairs.data(), W.pairs.size() * sizeof(WidePair), cudaMemcpyHostToDevice, st));
    if (!W.tasks.empty()) CU(cudaMemcpyAsync(W.d_tasks.p, W.tasks.data(), W.tasks.size() * sizeof(WideTask), cudaMemcpyHostToDevice, st));
    ctx->h2d += W.pairs.size() * sizeof(WidePair) + W.tasks.size() * sizeof(WideTask);
    ctx->fill_bytes += W.chunks * sizeof(Chunk);
    return B2A_OK;
}

int wide_fill(b2a_ctx* ctx, int r, cudaStream_t st, uint64_t* launches)
{
    WideState& W = ctx->wide;
    if (W.tasks.empty()) return B2A_OK;
    const b2a_params& prm = ctx->prm;
    CU(cudaMemsetAsync(W.d_progress.p, 0, 4, st));
    WideArgs a{};
    CU(W.next_epoch(W.bound_words, st, &a.epoch_tag));
    a.pat = ctx->d_pat.p; a.txt = ctx->d_txt.p; a.pairs = W.d_pairs.p; a.tasks = W.d_tasks.p;
    a.n_tasks = (uint32_t)W.tasks.size(); a.ticket = W.d_progress.p;
    a.codes = W.d_codes.p; a.bound = W.d_bound.p; a.rowbest = W.d_rowbest.p;
    a.final_score = W.d_final.p; a.final_col = W.d_final_col.p;
    a.ck = nullptr;
    a.match = prm.match; a.mismatch = prm.mismatch; a.gap = prm.gap;
    a.radix = W.K < 32 ? (1u << W.K) : 0u;
    a.alpha = ctx->d_alpha.p + (ctx->alpha_slots - 1);
    const unsigned need = (unsigned)((W.tasks.size() + WIDE_WARPS - 1) / WIDE_WARPS);
    const unsigned grid = std::min<unsigned>(need, (unsigned)ctx->sm_count * 8u);
    if (ctx->run[r].mode == B2A_MODE_SEMIGLOBAL) CU(launch_wide_fill_semi(W.store ? W.K : 2, W.store, W.alpha4, a, grid, st));
    else CU(launch_wide_fill(W.store ? W.K : 2, ctx->run[r].mode == B2A_MODE_LOCAL, W.store, W.alpha4, a, grid, st));   // score-only: no record, one instance
    ++*launches;
    return B2A_OK;
}

int wide_traceback(b2a_ctx* ctx, int r, cudaStream_t st, uint64_t* launches, bool score_only)
{
    WideState& W = ctx->wide;
    if (W.pairs.empty()) return B2A_OK;
    const b2a_params& prm = ctx->prm;
    WideTbArgs a{};
    a.pat = ctx->d_pat.p; a.txt = ctx->d_txt.p; a.pairs = W.d_pairs.p; a.n_wide = (uint32_t)W.pairs.size();
    a.codes = W.d_codes.p; a.rowbest = W.d_rowbest.p; a.final_score = W.d_final.p; a.final_col = W.d_final_col.p;
    a.results = ctx->run[r].d_results.p;
    a.ops = (prm.flags & B2A_WANT_OPS) && !score_only ? ctx->run[r].d_ops.p : nullptr;
    a.ops_off = ctx->d_ops_off.p;
    a.match = prm.match; a.mismatch = prm.mismatch; a.gap = prm.gap; a.score_only = score_only ? 1 : 0;
    a.opt = (prm.flags & B2A_TIE_HW4) ? 4 : 0;
    CU(launch_wide_tb(W.K, ctx->run[r].mode, a, st));
    ++*launches;
    return B2A_OK;
}

template <int K>
cudaError_t launch_ckpt_walk_k(bool local, const CkptWalkArgs& a, cudaStream_t st) {
    if (local) wide32_ckpt_walk_kernel<K, true><<<1, 32, 0, st>>>(a);
    else wide32_ckpt_walk_kernel<K, false><<<1, 32, 0, st>>>(a);
    return cudaGetLastError();
}
cudaError_t launch_ckpt_walk(int K, bool local, const CkptWalkArgs& a, cudaStream_t st) {
    switch (K) {
        case 2:  return launch_ckpt_walk_k<2>(local, a, st);
        case 4:  return launch_ckpt_walk_k<4>(local, a, st);
        case 8:  return launch_ckpt_walk_k<8>(local, a, st);
        case 16: return launch_ckpt_walk_k<16>(local, a, st);
        case 32: return launch_ckpt_walk_k<32>(local, a, st);
    }
    return cudaErrorInvalidValue;
}

// Pairs whose traceback record does not fit (ctx->wide_ckpt_bytes; 0.5 byte per cell, so a 1 Mb x 1 Mb pair would need 500 GB -- the
// reference's own full matrices, hw2.cpp:119-120, are what NOT to imitate).  Checkpointed recomputation, one pair at a time:
//   pass 1  score-only fill of the whole pair (the tiled kernel) that keeps the bottom row of every G-th band (4 bytes per column and
//           kept row) and, local mode, the per-row maxima -> score, and the row of the first row-major maximum (hw2.cpp:225-229);
//   pass 2  from the end cell upwards: the group of <= G bands that holds the path's current row is filled again WITH its record, from
//           the checkpoint row above it and only up to the path's current column, and the warp walker continues through it with the
//           reference's own comparisons (hw2.cpp:145-153 / :214-222) until it leaves the group at the top.
// Memory: kept rows (m / 128 G x n x 4 B) + one group record (128 G x n x 0.5 B).  Work: one score pass + at most one more fill.
int wide_ckpt_run(b2a_ctx* ctx, int r, cudaStream_t st, uint64_t* launches)
{
    WideState& W = ctx->wide;
    if (W.ckpt_pairs.empty()) return B2A_OK;
    const b2a_params& prm = ctx->prm;
    RunBuf& rb = ctx->run[r];
    const bool local = rb.mode == B2A_MODE_LOCAL, want_ops = (prm.flags & B2A_WANT_OPS) != 0;
    const int K = W.K, CS = 2 * (32 / K), skew = wide_skew(K);
    const uint32_t band_rows = 32u * WIDE_R;
    CU(W.d_pairs.reserve(1)); CU(W.d_final.reserve(1)); CU(W.d_progress.reserve(1)); CU(W.d_walk.reserve(1));
    for (const WideState::CkptSpec& sp : W.ckpt_pairs) {
        const uint32_t k = sp.pair, m = sp.m, n = sp.n;
        const uint32_t nbands = (m + band_rows - 1u) / band_rows;
        const uint64_t band_bytes = (uint64_t)WIDE_R * num_chunks(n, CS, skew) * 32u * sizeof(Chunk);
        const uint32_t G = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(nbands, ctx->wide_ckpt_group_bytes / std::max<uint64_t>(band_bytes, 1)));
        const uint32_t ck_stride = (n + 1u + 31u) & ~31u, n_ck = (nbands - 1u) / G;     // kept: the bottom rows of bands G-1, 2G-1, ... that have a band below
        const uint32_t bound_stride = ((n + 64u) + 31u) & ~31u;
        // kept columns: every 8192-th, so that pass 2 re-fills tiles of G bands x 8192 columns instead of strips as wide as the path's column
        const uint32_t col_shift = n > (2u << ctx->wide_ckpt_col_shift) ? ctx->wide_ckpt_col_shift : 0u, n_cc = col_shift ? n >> col_shift : 0u;
        const uint32_t col_stride = (m + 31u) & ~31u;
        const uint64_t colck_off = (uint64_t)n_ck * ck_stride;
        CU(W.d_ck.reserve(std::max<uint64_t>(1, colck_off + (uint64_t)n_cc * col_stride)));
        CU(W.d_rowbest.reserve(std::max<uint64_t>((uint64_t)nbands * band_rows, 1)));
        CU(W.d_tasks.reserve(nbands));
        CU(W.d_codes.reserve((uint64_t)G * band_bytes / sizeof(Chunk)));
        std::vector<WideTask> tasks(nbands);
        for (uint32_t b = 0; b < nbands; ++b) tasks[b] = WideTask{0u, b};
        CU(cudaMemcpyAsync(W.d_tasks.p, tasks.data(), nbands * sizeof(WideTask), cudaMemcpyHostToDevice, st));
        ctx->h2d += nbands * sizeof(WideTask);

        auto fill = [&](const WidePair& p, bool store) -> int {
            CU(cudaMemcpyAsync(W.d_pairs.p, &p, sizeof(p), cudaMemcpyHostToDevice, st));
            CU(cudaMemsetAsync(W.d_progress.p, 0, 4, st));
            WideArgs a{};
            CU(W.next_epoch(2ull * bound_stride, st, &a.epoch_tag));
            a.pat = ctx->d_pat.p; a.txt = ctx->d_txt.p; a.pairs = W.d_pairs.p; a.tasks = W.d_tasks.p;
            a.n_tasks = p.nbands; a.ticket = W.d_progress.p;
            a.codes = W.d_codes.p; a.bound = W.d_bound.p; a.rowbest = W.d_rowbest.p; a.final_score = W.d_final.p; a.ck = W.d_ck.p;
            a.match = prm.match; a.mismatch = prm.mismatch; a.gap = prm.gap;
            a.radix = K < 32 ? (1u << K) : 0u;
            a.alpha = ctx->d_alpha.p + (ctx->alpha_slots - 1);
            const unsigned need = (unsigned)((p.nbands + WIDE_WARPS - 1) / WIDE_WARPS);
            const unsigned grid = std::min<unsigned>(need, (unsigned)ctx->sm_count * 8u);
            if (!store && p.col_shift) CU(launch_wide_fill_keepcol(local, W.alpha4, a, grid, st));
            else CU(launch_wide_fill(store ? K : 2, local, store, W.alpha4, a, grid, st));
            ++*launches;
            CU(cudaStreamSynchronize(st));                        // &p and the next sub-problem's plan depend on this launch
            return B2A_OK;
        };

        // ---- pass 1: scores + kept rows ----
        WidePair whole{};
        whole.pat_off = sp.pat_off; whole.txt_off = sp.txt_off; whole.m = m; whole.n = n; whole.pair = k; whole.nbands = nbands;
        whole.bound_stride = bound_stride; whole.top_off = WIDE_NO_TOP; whole.left_off = WIDE_NO_TOP;
        whole.ck_every = n_ck ? G : 0u; whole.ck_stride = ck_stride;
        whole.col_shift = col_shift; whole.colck_off = colck_off; whole.col_stride = col_stride;
        { int rc = fill(whole, false); if (rc != B2A_OK) return rc; }
        CkptWalk wst{};
        wst.i = m; wst.j = n;
        if (local) {
            CU(cudaMemcpyAsync(W.d_walk.p, &wst, sizeof(wst), cudaMemcpyHostToDevice, st));
            wide32_first_best_row_kernel<<<1, 32, 0, st>>>(W.d_rowbest.p, m, W.d_walk.p);
            CU(cudaGetLastError()); ++*launches;
            CU(cudaMemcpyAsync(&wst, W.d_walk.p, sizeof(wst), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            wst.j = n;                                            // the column of the maximum is found in the first re-filled group
        } else {
            int32_t sc = 0;
            CU(cudaMemcpyAsync(&sc, W.d_final.p, 4, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            wst.score = sc; wst.end_i = m; wst.end_j = n;
        }
        // ---- pass 2: band groups, bottom-up ----
        bool first = true;
        if (local && wst.score == 0) {                            // hw2.cpp:202-203: no positive cell, empty alignment
            PairResult res{0, 0, 0, 0, 0, 0, 0, 2};
            CU(cudaMemcpyAsync(rb.d_results.p + k, &res, sizeof(res), cudaMemcpyHostToDevice, st));
            CU(cudaStreamSynchronize(st));
            continue;
        }
        while (!wst.done) {
            const uint32_t g = (wst.i - 1u) / (G * band_rows), r0 = g * G * band_rows;
            // local mode, first group: the end column is not known yet -> full width; afterwards the tile right of the last kept column
            const uint32_t cb = (col_shift && !(local && first)) ? (wst.j - 1u) >> col_shift : 0u, c0 = cb << col_shift;
            WidePair sub{};
            sub.pat_off = sp.pat_off + r0; sub.txt_off = sp.txt_off + c0; sub.m = wst.i - r0; sub.n = wst.j - c0; sub.pair = k;
            sub.nbands = (sub.m + band_rows - 1u) / band_rows;
            sub.bound_stride = bound_stride; sub.row_base = r0; sub.col_base = c0;
            sub.top_off = g ? (uint64_t)(g - 1u) * ck_stride + c0 : WIDE_NO_TOP;
            sub.left_off = cb ? colck_off + (uint64_t)(cb - 1u) * col_stride + r0 : WIDE_NO_TOP;
            { int rc = fill(sub, true); if (rc != B2A_OK) return rc; }
            CU(cudaMemcpyAsync(W.d_walk.p, &wst, sizeof(wst), cudaMemcpyHostToDevice, st));
            CkptWalkArgs wa{};
            wa.pat = ctx->d_pat.p; wa.txt = ctx->d_txt.p; wa.pair = W.d_pairs.p; wa.codes = W.d_codes.p; wa.rowbest = W.d_rowbest.p; wa.ck = W.d_ck.p;
            wa.st = W.d_walk.p; wa.result = rb.d_results.p + k;
            wa.ops = want_ops ? rb.d_ops.p + ctx->h_ops_off.p[k] : nullptr;
            wa.m_total = m; wa.n_total = n;
            wa.match = prm.match; wa.mismatch = prm.mismatch; wa.gap = prm.gap;
            wa.opt = (prm.flags & B2A_TIE_HW4) ? 4 : 0;
            wa.first = (local && first) ? 1 : 0;
            CU(launch_ckpt_walk(K, local, wa, st));
            ++*launches;
            CU(cudaMemcpyAsync(&wst, W.d_walk.p, sizeof(wst), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            first = false;
            if (!wst.done && (wst.i == 0 || wst.j == 0)) return fail(ctx, B2A_ERR_STATE, "internal: checkpointed walk left the matrix without finishing");
            if (!wst.done && wst.i > r0 && wst.j > c0) return fail(ctx, B2A_ERR_STATE, "internal: checkpointed walk stopped inside a tile");
        }
        ctx->fill_bytes += ((uint64_t)n_ck * ck_stride + (uint64_t)n_cc * col_stride) * 4;
    }
    return B2A_OK;
}

// ---------------------------------------------------------------------------------------------
// short16 family: segments
// ---------------------------------------------------------------------------------------------
// 4 events per (segment, run), created on demand: inputs ready (run 0's slot only), fill start, fill end, traceback end
cudaEvent_t* seg_events(b2a_ctx* ctx, size_t si, int r = 0) {
    const size_t slot = si * MAX_RUNS + (size_t)r;
    while (ctx->ev_pool.size() < 4 * (slot + 1)) {
        cudaEvent_t e = nullptr;
        if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
        ctx->ev_pool.push_back(e);
    }
    return ctx->ev_pool.data() + 4 * slot;
}

// fill + traceback kernels of one segment for run r, on the next lane
int launch_segment(b2a_ctx* ctx, size_t si, int r, uint64_t* launches)
{
    Segment& sg = ctx->segs[si];
    if (sg.classes.empty()) return B2A_OK;
    const b2a_params& prm = ctx->prm;
    RunBuf& rb = ctx->run[r];
    const int mode = rb.mode;
    const bool local = mode == B2A_MODE_LOCAL, want_ops = (prm.flags & B2A_WANT_OPS) != 0;
    Lane& ln = ctx->lanes[ctx->n_launched++ % (uint64_t)ctx->n_lanes];
    cudaStream_t st = ctx->s_fill;
    cudaEvent_t* ev = seg_events(ctx, si, r);
    cudaEvent_t* ev_in = seg_events(ctx, si, 0);
    if (!ev || !ev_in) return fail(ctx, B2A_ERR_CUDA, "cudaEventCreate failed");
    if (sg.chunks > ln.codes.cap || (local && sg.rowbest_words > ln.rowbest.cap)) {     // (rowbest is a local-mode buffer: a lane that only ever
                                                                                         // serves global runs never grows it)
        CU(cudaStreamSynchronize(ctx->s_fill)); CU(cudaStreamSynchronize(ln.s_tb)); CU(cudaStreamSynchronize(ln.s_tb_lo));   // the lane's record is about to be reallocated
        CU(ln.codes.reserve(sg.chunks));
        if (local) CU(ln.rowbest.reserve(sg.rowbest_words));
    }
    CU(cudaStreamWaitEvent(st, ev_in[0], 0));                // inputs + plan of this segment are on the device
    CU(cudaStreamWaitEvent(st, ln.tb_done, 0));              // the previous user of this lane's record has been walked
    CU(cudaEventRecord(ev[1], st));
    const AlphaInfo* alpha = ctx->d_alpha.p + si;
    for (size_t ci = 0; ci < sg.classes.size(); ++ci) {
        const ClassRange& c = sg.classes[ci];
        Short16Plan pl{0, 0, 0};
        short16_plan(mode, (uint32_t)c.R * 32u, c.max_n, prm.match, prm.mismatch, prm.gap, pl);   // bias for the class' largest shape
        FillArgs a{};
        a.pat = ctx->d_pat.p; a.txt = ctx->d_txt.p; a.pat_off = ctx->d_pat_off.p; a.txt_off = ctx->d_txt_off.p;
        a.pps = ctx->d_pps.p + sg.pp_first + c.first; a.code_off = ctx->d_code_off.p + sg.pp_first + c.first; a.codes = ln.codes.p;
        a.rowbest = local ? ln.rowbest.p + (size_t)c.first * c.R * 32 : nullptr;
        a.endcell = rb.d_endcell.p;
        a.n_pp = c.count;
        a.match = prm.match; a.mismatch = prm.mismatch; a.gap = prm.gap; a.bias = pl.bias;
        a.radix = 1u << ctx->K;
        a.alpha = alpha;
        a.dirty = ctx->d_dirty.p + sg.pp_first + c.first;
        a.dirty_list = ctx->d_dirty_list.p + sg.pp_first + c.first;
        a.dirty_cnt = ctx->d_dirty_cnt.p + si * DIRTY_CLASSES + ci;
        CU(launch_fill(ctx->K, c.R, mode, a, st));
        *launches += 2;
    }
    CU(cudaEventRecord(ev[2], st));
    st = ctx->tb_low ? ln.s_tb_lo : ln.s_tb;
    CU(cudaStreamWaitEvent(st, ev[2], 0));
    for (const ClassRange& c : sg.classes) {
        Short16Plan pl{0, 0, 0};
        short16_plan(mode, (uint32_t)c.R * 32u, c.max_n, prm.match, prm.mismatch, prm.gap, pl);
        TbArgs a{};
        a.pat = ctx->d_pat.p; a.txt = ctx->d_txt.p; a.pat_off = ctx->d_pat_off.p; a.txt_off = ctx->d_txt_off.p;
        a.pps = ctx->d_pps.p + sg.pp_first + c.first; a.code_off = ctx->d_code_off.p + sg.pp_first + c.first; a.codes = ln.codes.p;
        a.rowbest = local ? ln.rowbest.p + (size_t)c.first * c.R * 32 : nullptr;
        a.endcell = rb.d_endcell.p;
        a.results = rb.d_results.p; a.ops = want_ops ? rb.d_ops.p : nullptr; a.ops_off = ctx->d_ops_off.p;
        a.n_pp = c.count; a.R = c.R;
        a.match = prm.match; a.mismatch = prm.mismatch; a.gap = prm.gap; a.bias = pl.bias;
        a.opt = 0;
        a.tie_hw4 = (prm.flags & B2A_TIE_HW4) ? 1 : 0;
        a.alpha = alpha;
        a.dirty = ctx->d_dirty.p + sg.pp_first + c.first;
        CU(launch_tb(ctx->K, mode, a, st));
        ++*launches;
    }
    CU(cudaEventRecord(ev[3], st));
    CU(cudaEventRecord(ln.tb_done, st));
    return B2A_OK;
}

// s_fill waits for every traceback queued so far (the wide32 phase and the end-of-run event follow on s_fill)
int join_tracebacks(b2a_ctx* ctx) {
    for (int l = 0; l < MAX_LANES; ++l) CU(cudaStreamWaitEvent(ctx->s_fill, ctx->lanes[l].tb_done, 0));
    return B2A_OK;
}

// ---------------------------------------------------------------------------------------------
// affine32: hw3's distance stage (score only).  `specs` index into the device copies of pat / txt.
// ---------------------------------------------------------------------------------------------
struct AffSpec { uint64_t pat_off, txt_off; uint32_t m, n; };

int affine_run(b2a_ctx* ctx, int match, int mismatch, int gopen, int gext, const uint8_t* pat, uint64_t pat_bytes,
               const uint8_t* txt, uint64_t txt_bytes, bool same_buffer, const std::vector<AffSpec>& specs, int32_t* scores,
               bool trace, uint32_t* n_ops_out)
{
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->s_copy)); CU(cudaStreamSynchronize(ctx->s_down));
    CU(cudaStreamSynchronize(ctx->s_fill));
    for (auto& ln : ctx->lanes) { CU(cudaStreamSynchronize(ln.s_tb)); CU(cudaStreamSynchronize(ln.s_tb_lo)); }
    ctx->have_batch = false; ctx->ran = false; ctx->affine_ops = false;   // the batch buffers are reused below
    ctx->cells = ctx->fill_bytes = ctx->launches = ctx->h2d = ctx->d2h = 0;
    const int64_t smag = std::max<int64_t>({std::llabs((long long)match), std::llabs((long long)mismatch),
                                            std::llabs((long long)gopen) + std::llabs((long long)gext)});
    const size_t n = specs.size();
    uint64_t opsw = 0;
    if (trace) CU(ctx->h_ops_off.reserve(n + 1));
    for (size_t k = 0; k < n; ++k) {
        const AffSpec& sp = specs[k];
        // the sentinel arithmetic of hw3.cpp:16 must not wrap: NEG - (m+n)*max|score| has to stay above INT_MIN
        if (((uint64_t)sp.m + sp.n + 2) * (uint64_t)smag >= (1ull << 30))
            return fail(ctx, B2A_ERR_RANGE, "b2a_affine: (m+n)*max|score| exceeds 2^30 (hw3's INT_MIN/2 sentinel would wrap)");
        if ((sp.m + 32u * WIDE_R - 1u) / (32u * WIDE_R) >= (1u << 20))
            return fail(ctx, B2A_ERR_RANGE, "b2a_affine: sequence too long (band index must fit 20 bits)");
        ctx->cells += (uint64_t)sp.m * sp.n;
        if (trace) { ctx->h_ops_off.p[k] = opsw; opsw += ((uint64_t)sp.m + sp.n + 15) / 16 + 1; }
    }
    WideState& W = ctx->wide;
    cudaStream_t st = ctx->s_fill;
    CU(ctx->d_pat.reserve(pat_bytes + 16));
    if (!same_buffer) CU(ctx->d_txt.reserve(txt_bytes + 16));
    CU(ctx->d_alpha.reserve(2)); CU(ctx->h_alpha.reserve(2)); CU(ctx->d_hist.reserve(256));
    CU(W.d_progress.reserve(1));
    if (trace) {
        ctx->h_ops_off.p[n] = opsw;
        CU(ctx->run[0].d_ops.reserve(opsw)); CU(ctx->d_ops_off.reserve(n + 1)); CU(ctx->d_nops.reserve(n));
        CU(cudaMemcpyAsync(ctx->d_ops_off.p, ctx->h_ops_off.p, (n + 1) * 8, cudaMemcpyHostToDevice, st));
        if (n) CU(cudaMemsetAsync(ctx->d_nops.p, 0, n * 4, st));
    }
    if (pat_bytes) CU(cudaMemcpyAsync(ctx->d_pat.p, pat, pat_bytes, cudaMemcpyHostToDevice, st));
    if (!same_buffer && txt_bytes) CU(cudaMemcpyAsync(ctx->d_txt.p, txt, txt_bytes, cudaMemcpyHostToDevice, st));
    ctx->h2d += pat_bytes + (same_buffer ? 0 : txt_bytes);
    CU(cudaMemsetAsync(ctx->d_alpha.p, 0, sizeof(AlphaInfo), st));
    CU(cudaMemsetAsync(ctx->d_hist.p, 0, 256 * sizeof(uint32_t), st));
    uint64_t launches = 0;
    if (pat_bytes) {
        const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)ctx->sm_count * 4u, (pat_bytes + 4095) / 4096);
        alphabet_kernel<<<grid, 256, 0, st>>>(ctx->d_pat.p, pat_bytes, ctx->d_hist.p);
        CU(cudaGetLastError()); ++launches;
    }
    alphabet_finish_kernel<<<1, 32, 0, st>>>(ctx->d_alpha.p, ctx->d_hist.p);
    CU(cudaGetLastError()); ++launches;
    CU(cudaMemcpyAsync(ctx->h_alpha.p, ctx->d_alpha.p, sizeof(AlphaInfo), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const bool alpha4 = !ctx->h_alpha.p[0].too_many && match <= 127 && match >= -128 && mismatch <= 127 && mismatch >= -128;

    // pairs are served in groups whose trace codes (0.5 byte per cell) fit the budget; score-only runs are one group
    const uint64_t code_budget_chunks = (48ull << 30) / sizeof(Chunk);
    float ms_total = 0;
    size_t first = 0;
    while (first < n) {
        W.pairs.clear(); W.tasks.clear();
        W.bound_words = 0; W.chunks = 0;
        uint32_t max_bands = 0;
        std::vector<uint32_t> slot;                         // spec index of every planned pair of the group
        size_t k = first;
        for (; k < n; ++k) {
            const AffSpec& sp = specs[k];
            if (sp.m == 0 || sp.n == 0) continue;           // borders only: answered on the host below
            WidePair p{};
            p.top_off = WIDE_NO_TOP; p.left_off = WIDE_NO_TOP;
            p.pat_off = sp.pat_off; p.txt_off = sp.txt_off; p.m = sp.m; p.n = sp.n; p.pair = (uint32_t)k;
            const uint32_t band_rows = 32u * (uint32_t)(trace ? WIDE_R : AFFINE_R_SCORE);
            p.nbands = (sp.m + band_rows - 1u) / band_rows;
            const uint64_t need = trace ? (uint64_t)p.nbands * WIDE_R * ((sp.n + 63u) / 32u) * 32u : 0;
            if (trace && !W.pairs.empty() && W.chunks + need > code_budget_chunks) break;
            p.code_off = W.chunks; W.chunks += need;
            p.bound_stride = ((sp.n + 64u) + 31u) & ~31u;
            p.bound_off = W.bound_words; if (p.nbands > 1u) W.bound_words += 6ull * p.bound_stride;   // 2 buffers x {Vg, F, M3}
            max_bands = std::max(max_bands, p.nbands);
            slot.push_back((uint32_t)k);
            W.pairs.push_back(p);
        }
        const size_t group_end = k;
        std::vector<uint32_t> order(W.pairs.size());
        for (uint32_t i = 0; i < order.size(); ++i) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return W.pairs[a].nbands > W.pairs[b].nbands; });
        for (uint32_t b = 0; b < max_bands; ++b)             // band-major tickets: a band's producer always holds an earlier ticket
            for (uint32_t i : order) { if (W.pairs[i].nbands <= b) break; W.tasks.push_back(WideTask{i, b}); }
        std::vector<int32_t> fin(W.pairs.size());
        if (!W.tasks.empty()) {
            CU(W.d_pairs.reserve(W.pairs.size())); CU(W.d_tasks.reserve(W.tasks.size())); CU(W.d_final.reserve(W.pairs.size()));
            if (trace) CU(W.d_codes.reserve(W.chunks));
            CU(cudaMemcpyAsync(W.d_pairs.p, W.pairs.data(), W.pairs.size() * sizeof(WidePair), cudaMemcpyHostToDevice, st));
            CU(cudaMemcpyAsync(W.d_tasks.p, W.tasks.data(), W.tasks.size() * sizeof(WideTask), cudaMemcpyHostToDevice, st));
            ctx->h2d += W.pairs.size() * sizeof(WidePair) + W.tasks.size() * sizeof(WideTask);
            CU(cudaMemsetAsync(W.d_progress.p, 0, 4, st));
            AffineArgs a{};
            CU(W.next_epoch(W.bound_words, st, &a.epoch_tag));
            a.pat = ctx->d_pat.p; a.txt = same_buffer ? ctx->d_pat.p : ctx->d_txt.p; a.pairs = W.d_pairs.p; a.tasks = W.d_tasks.p;
            a.n_tasks = (uint32_t)W.tasks.size(); a.ticket = W.d_progress.p;
            a.bound = W.d_bound.p; a.final_score = W.d_final.p;
            a.match = match; a.mismatch = mismatch; a.gopen = gopen; a.gext = gext; a.alpha = ctx->d_alpha.p;
            a.codes = trace ? reinterpret_cast<uint4*>(W.d_codes.p) : nullptr;
            const unsigned need = (unsigned)((W.tasks.size() + WIDE_WARPS - 1) / WIDE_WARPS);
            const unsigned grid = std::min<unsigned>(need, (unsigned)ctx->sm_count * 8u);
            CU(cudaEventRecord(ctx->ev_begin, st));
            if (trace) { if (alpha4) affine32_score_kernel<true, true, WIDE_R><<<grid, WIDE_WARPS * 32, 0, st>>>(a);
                         else affine32_score_kernel<false, true, WIDE_R><<<grid, WIDE_WARPS * 32, 0, st>>>(a); }
            else       { if (alpha4) affine32_score_kernel<true, false, AFFINE_R_SCORE><<<grid, WIDE_WARPS * 32, 0, st>>>(a);
                         else affine32_score_kernel<false, false, AFFINE_R_SCORE><<<grid, WIDE_WARPS * 32, 0, st>>>(a); }
            CU(cudaGetLastError()); ++launches;
            if (trace) {
                AffineTbArgs ta{W.d_pairs.p, (uint32_t)W.pairs.size(), reinterpret_cast<const uint4*>(W.d_codes.p), ctx->d_nops.p, ctx->run[0].d_ops.p, ctx->d_ops_off.p};
                affine32_traceback_kernel<<<(unsigned)((W.pairs.size() + WIDE_TB_WARPS - 1) / WIDE_TB_WARPS), WIDE_TB_WARPS * 32, 0, st>>>(ta);
                CU(cudaGetLastError()); ++launches;
                ctx->fill_bytes += W.chunks * sizeof(Chunk);
            }
            CU(cudaEventRecord(ctx->ev_end, st));
            CU(cudaMemcpyAsync(fin.data(), W.d_final.p, fin.size() * 4, cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            float ms = 0;
            CU(cudaEventElapsedTime(&ms, ctx->ev_begin, ctx->ev_end));
            ms_total += ms;
            ctx->d2h += fin.size() * 4;
        }
        for (size_t q = 0; q < slot.size(); ++q) scores[slot[q]] = fin[q];
        first = group_end;
    }
    for (size_t k = 0; k < n; ++k) {
        const AffSpec& sp = specs[k];
        if (sp.m && sp.n) continue;
        if (sp.m == 0 && sp.n == 0) scores[k] = 0;                                       // V[0][0]               hw3.cpp:40
        else if (sp.m == 0) scores[k] = gopen + gext * (int32_t)(sp.n - 1);              // E[0][n]               hw3.cpp:50
        else scores[k] = gopen + gext * (int32_t)(sp.m - 1);                             // F[m][0]               hw3.cpp:44
    }
    if (trace) {
        std::vector<uint32_t> nops(n);
        if (n) CU(cudaMemcpy(nops.data(), ctx->d_nops.p, n * 4, cudaMemcpyDeviceToHost));
        for (size_t k = 0; k < n; ++k) {
            const AffSpec& sp = specs[k];
            if (sp.m == 0 || sp.n == 0) {
                // one gap run along a border (hw3.cpp:42-53): all 'D' (column 0) or all 'I' (row 0); written from the host
                const uint32_t len = sp.m + sp.n, op = sp.n == 0 ? OP_D : OP_I;
                std::vector<uint32_t> w(((uint64_t)len + 15) / 16 + 1, op * 0x55555555u);
                if (len) CU(cudaMemcpy(ctx->run[0].d_ops.p + ctx->h_ops_off.p[k], w.data(), (((uint64_t)len + 15) / 16) * 4, cudaMemcpyHostToDevice));
                nops[k] = len;
            }
            if (n_ops_out) n_ops_out[k] = nops[k];
        }
        if (n) CU(cudaMemcpy(ctx->d_nops.p, nops.data(), n * 4, cudaMemcpyHostToDevice));
        ctx->affine_ops = true; ctx->n_pairs = n; ctx->total_ops_words = opsw;
    }
    ctx->last_fill_ms = ms_total; ctx->last_tb_ms = 0; ctx->last_total_ms = ms_total;
    ctx->launches = launches;
    return B2A_OK;
}

bool is_pinned(const void* p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

// Cuts the batch into segments, queues the copies, plans, and (pipelined == true) launches every
// segment as soon as it is planned and returns the result records.  With pipelined == false the
// batch ends up resident and planned; b2a_batch_run launches it.
int batch_prepare(b2a_ctx* ctx, const b2a_params* prms, uint32_t n_runs, const uint8_t* pat, const uint64_t* pat_off,
                  const uint8_t* txt, const uint64_t* txt_off, uint64_t n_pairs, bool pipelined, b2a_result* const* results,
                  const b2a_seq2* pat2 = nullptr, const b2a_seq2* txt2 = nullptr)
{
    if (!ctx) return B2A_ERR_ARG;
    const bool compact = pat2 != nullptr;                          // b2a_seq2 inputs: pat / txt are null, the device expands the codes
    if (!prms || !pat_off || !txt_off || n_runs < 1 || n_runs > (uint32_t)MAX_RUNS)
        return fail(ctx, B2A_ERR_ARG, "b2a_batch_upload: null argument or bad run count");
    const b2a_params* prm = &prms[0];
    bool any_local = false;
    for (uint32_t r = 0; r < n_runs; ++r) {
        const b2a_params& q = prms[r];
        if (q.mode != B2A_MODE_GLOBAL && q.mode != B2A_MODE_LOCAL && q.mode != B2A_MODE_SEMIGLOBAL) return fail(ctx, B2A_ERR_ARG, "b2a_batch_upload: bad mode");
        if ((q.flags & B2A_TIE_HW4) && q.mode != B2A_MODE_GLOBAL) return fail(ctx, B2A_ERR_ARG, "B2A_TIE_HW4 applies to the global mode only");
        if (q.match != prm->match || q.mismatch != prm->mismatch || q.gap != prm->gap || ((q.flags ^ prm->flags) & ~B2A_TIE_HW4))
            return fail(ctx, B2A_ERR_ARG, "b2a_align_batch_multi: the runs of one batch share scoring and flags (they differ in mode)");
        if (pipelined && n_pairs && (!results || !results[r])) return fail(ctx, B2A_ERR_ARG, "b2a_align_batch: null results");
        any_local |= q.mode == B2A_MODE_LOCAL;
    }
    if (n_pairs > 0x7FFFFFF0ull) return fail(ctx, B2A_ERR_ARG, "b2a_batch_upload: too many pairs");
    CU(cudaSetDevice(ctx->device));
    // a previous batch may still own the pinned plan arrays / device buffers
    CU(cudaStreamSynchronize(ctx->s_copy)); CU(cudaStreamSynchronize(ctx->s_down));
    CU(cudaStreamSynchronize(ctx->s_fill));
    for (auto& ln : ctx->lanes) { CU(cudaStreamSynchronize(ln.s_tb)); CU(cudaStreamSynchronize(ln.s_tb_lo)); }
    ctx->have_batch = false; ctx->ran = false; ctx->affine_ops = false;
    ctx->prm = *prm; ctx->n_pairs = n_pairs;
    ctx->n_runs = n_runs; ctx->sel_run = 0; ctx->n_launched = 0;
    // A traceback kernel has a latency floor of ~1.3 ms however few pairs it walks (every thread takes its ~700 dependent steps), and a fill
    // may only overwrite a lane's record after the traceback that reads it.  So the launches alternate over several record lanes, each with
    // its own traceback stream: 4 lanes (7 GB each) for large batches, 8 for batches below two maximal segments (e.g. one rank's 125 k
    // pairs of a 1 M batch strong-scaled over 8 GPUs), whose tracebacks would otherwise gate the next fill.  With >= 3 lanes the
    // tracebacks run at the fill's priority and fill the gaps the fill grids leave; with 2 lanes they must overtake the next fill (high
    // priority) or that fill waits.  Measured end to end, both modes (scripts/small_batch_exp.py, scripts/seg_e2e_sweep.py):
    //   125 k pairs: 2 lanes 9.80 ms, 8 lanes 9.19 ms, 8 lanes + fill priority 8.40 ms;   1 M pairs: 57.98 / 57.25 (4 lanes) / 57.06 ms.
    // Equal segments of exactly two fill waves were tried for small batches and lose: resident traceback CTAs take a CTA slot per SM from
    // the fill, which turns two waves into three.
    const bool small_batch = pipelined && !ctx->seg_user && n_pairs < 2 * ctx->seg_max_pairs;
    ctx->n_lanes = ctx->lanes_cfg ? ctx->lanes_cfg : (small_batch ? MAX_LANES : (pipelined ? 4 : 2));
    ctx->tb_low = ctx->n_lanes >= 3;
    for (uint32_t r = 0; r < n_runs; ++r) ctx->run[r].mode = prms[r].mode;
    ctx->segs.clear(); ctx->wide_pairs.clear();
    ctx->cells = ctx->fill_bytes = ctx->launches = ctx->h2d = ctx->d2h = 0;
    ctx->n_pp_total = 0;
    const uint64_t pat_bytes = n_pairs ? pat_off[n_pairs] : 0, txt_bytes = n_pairs ? txt_off[n_pairs] : 0;
    if (!compact && ((pat_bytes && !pat) || (txt_bytes && !txt))) return fail(ctx, B2A_ERR_ARG, "b2a_batch_upload: null sequence buffer");
    const b2a_seq2* sq[2] = {pat2, txt2};
    const uint64_t sq_bytes[2] = {pat_bytes, txt_bytes};
    uint64_t sq_copied[2] = {0, 0}, sq_exc[2] = {0, 0};            // code bytes / exceptions already queued (segments ascend)
    uint32_t sq_alpha[2] = {0, 0};
    for (int w = 0; compact && w < 2; ++w) {
        if (!sq[w]) return fail(ctx, B2A_ERR_ARG, "b2a_align_batch_multi_seq2: null b2a_seq2");
        if (sq[w]->n_bytes < sq_bytes[w] || (sq_bytes[w] && !sq[w]->codes) || (sq[w]->n_exc && (!sq[w]->exc_pos || !sq[w]->exc_byte)))
            return fail(ctx, B2A_ERR_ARG, "b2a_align_batch_multi_seq2: the b2a_seq2 is shorter than its offsets say, or lacks an array");
        std::memcpy(&sq_alpha[w], sq[w]->alphabet, 4);
        // The offsets need not start at 0: a caller that shards ONE packed buffer over several contexts hands each of them the same
        // b2a_seq2 and its own slice of the offsets; only the slice's codes and exceptions are copied and expanded.
        const uint64_t base = n_pairs ? (w ? txt_off[0] : pat_off[0]) : 0;
        sq_copied[w] = base / 4;
        sq_exc[w] = (uint64_t)(std::lower_bound(sq[w]->exc_pos, sq[w]->exc_pos + sq[w]->n_exc, base) - sq[w]->exc_pos);
    }
    // Appendix A.8: (m+n)*max|score| must stay inside int32 (beyond that the reference itself is undefined)
    const int64_t smag = std::max<int64_t>({std::llabs((long long)prm->match), std::llabs((long long)prm->mismatch),
                                            std::llabs((long long)prm->gap)});
    const bool want_ops = (prm->flags & B2A_WANT_OPS) != 0;
    const bool score_only = (prm->flags & B2A_SCORE_ONLY) != 0;
    // one plan serves every run: a pair is a short16 pair iff the s16x2 record holds it in every run's mode (NW is the stricter one)
    auto plan_all = [&](uint32_t m, uint32_t n, Short16Plan& pl) {
        for (uint32_t r = 0; r < n_runs; ++r)
            if (!short16_plan(prms[r].mode, m, n, prm->match, prm->mismatch, prm->gap, pl)) return false;
        return true;
    };
    ctx->K = delta_bits(prm->match, prm->mismatch, prm->gap);
    const int CS = ctx->K ? chunk_steps(ctx->K) : 24;

    // ---- batch-wide buffers (grow-only) ----
    const uint64_t ops_bound = (pat_bytes + txt_bytes) / 16 + 2 * n_pairs + 2;     // >= sum((m+n+15)/16 + 1)
    ctx->alpha_slots = (size_t)(n_pairs / SEG_MIN_PAIRS + 3);        // >= segments + 1
    CU(ctx->d_pat.reserve(pat_bytes + 16)); CU(ctx->d_txt.reserve(txt_bytes + 16));
    CU(ctx->d_pat_off.reserve(n_pairs + 1)); CU(ctx->d_txt_off.reserve(n_pairs + 1));
    for (int w = 0; compact && w < 2; ++w) {
        CU(ctx->seq2[w].codes.reserve(sq_bytes[w] / 4 + 32));
        if (sq[w]->n_exc) { CU(ctx->seq2[w].epos.reserve(sq[w]->n_exc)); CU(ctx->seq2[w].ebyte.reserve(sq[w]->n_exc)); }
    }
    CU(ctx->d_pps.reserve(n_pairs)); CU(ctx->d_code_off.reserve(n_pairs));
    CU(ctx->h_pps.reserve(n_pairs)); CU(ctx->h_code_off.reserve(n_pairs)); CU(ctx->h_ops_off.reserve(n_pairs + 1));
    for (uint32_t r = 0; r < n_runs; ++r) {
        RunBuf& rb = ctx->run[r];
        CU(rb.d_results.reserve(n_pairs));
        if (rb.mode != B2A_MODE_GLOBAL) CU(rb.d_endcell.reserve(n_pairs));    // the short16 fill epilogues' end cells (local, semi-global)
        if (want_ops) CU(rb.d_ops.reserve(ops_bound));
    }
    CU(ctx->d_alpha.reserve(ctx->alpha_slots)); CU(ctx->h_alpha.reserve(ctx->alpha_slots));
    CU(ctx->d_hist.reserve(ctx->alpha_slots * 256)); CU(ctx->d_dirty.reserve(n_pairs)); CU(ctx->h_dirty.reserve(n_pairs));
    CU(ctx->d_dirty_list.reserve(n_pairs)); CU(ctx->d_dirty_cnt.reserve(ctx->alpha_slots * DIRTY_CLASSES));
    CU(cudaMemsetAsync(ctx->d_dirty_cnt.p, 0, ctx->alpha_slots * DIRTY_CLASSES * sizeof(uint32_t), ctx->s_copy));
    if (want_ops) CU(ctx->d_ops_off.reserve(n_pairs + 1));
    CU(cudaMemsetAsync(ctx->d_alpha.p, 0, ctx->alpha_slots * sizeof(AlphaInfo), ctx->s_copy));
    CU(cudaMemsetAsync(ctx->d_hist.p, 0, ctx->alpha_slots * 256 * sizeof(uint32_t), ctx->s_copy));
    if (n_pairs) CU(cudaMemsetAsync(ctx->d_dirty.p, 0, n_pairs, ctx->s_copy));
    bool async_down = pipelined && results;
    for (uint32_t r = 0; r < n_runs && async_down; ++r) async_down = is_pinned(results[r]);
    const bool sink = pipelined && want_ops && ctx->ops_sink_runs >= n_runs;      // op lists go to the host per segment, under the kernels
    uint64_t launches = 0;
    using clk = std::chrono::steady_clock;
    const clk::time_point t_begin = clk::now();
    auto ms_since = [&](clk::time_point t) { return std::chrono::duration<double, std::milli>(clk::now() - t).count(); };
    std::vector<double> tr_host;                                         // per segment: host ms at pass-1 end, plan end, launch end
    if (ctx->trace) CU(cudaEventRecord(ctx->ev_begin, ctx->s_copy));

    std::vector<PPDesc> pps[SHORT16_MAX_R + 1];
    std::unordered_map<uint64_t, uint32_t> pending;
    uint64_t opsw = 0, cells = 0;
    uint64_t first = 0;
    while (first < n_pairs) {
        // ---- pass 1: validate, find the end of the segment, per-pair op offsets ----
        uint64_t k = first, seg_bytes = 0;
        const size_t si_next = ctx->segs.size();
        const uint64_t lim_pairs = !pipelined ? ctx->seg_resident_pairs
                           : std::min<uint64_t>(ctx->seg_max_pairs, si_next < 20 ? ctx->seg_first_pairs << si_next : ctx->seg_max_pairs);
        const uint64_t lim_bytes = pipelined ? ctx->seg_budget_bytes : ctx->seg_resident_bytes;
        uint64_t plan_key = ~0ull; bool plan_ok = false; Short16Plan pl{0, 0, 0}; uint64_t pair_bytes = 0;
        for (; k < n_pairs; ++k) {
            if (pat_off[k + 1] < pat_off[k] || txt_off[k + 1] < txt_off[k])
                return fail(ctx, B2A_ERR_ARG, "b2a_batch_upload: offsets must be non-decreasing");
            const uint64_t m64 = pat_off[k + 1] - pat_off[k], n64 = txt_off[k + 1] - txt_off[k];
            if ((m64 + n64 + 2) * (uint64_t)smag >= 0x7FFFFFFFull || m64 + n64 >= 0x7FFFFFF0ull)
                return fail(ctx, B2A_ERR_RANGE, "b2a_batch_upload: (m+n)*max|score| exceeds int32 (SURVEY.md A.8)");
            ctx->h_ops_off.p[k] = opsw;
            opsw += (m64 + n64 + 15) / 16 + 1;
            cells += m64 * n64;
            const uint64_t key = (m64 << 32) | n64;
            if (key != plan_key) {
                plan_key = key;
                plan_ok = !score_only && plan_all((uint32_t)m64, (uint32_t)n64, pl);
                pair_bytes = plan_ok ? (uint64_t)pl.R * num_chunks((uint32_t)n64, CS) * 32u * sizeof(Chunk) / 2 : 0;
            }
            seg_bytes += pair_bytes;
            const uint64_t cnt = k + 1 - first;
            if (cnt >= SEG_MIN_PAIRS && !(cnt & 1) && (seg_bytes >= lim_bytes || cnt >= lim_pairs)) { ++k; break; }
        }
        if (ctx->trace) tr_host.push_back(ms_since(t_begin));
        const size_t si = ctx->segs.size();
        ctx->segs.emplace_back();
        Segment& sg = ctx->segs.back();
        sg.first = first; sg.count = k - first;
        sg.pp_first = ctx->n_pp_total;
        if (si + 2 > ctx->alpha_slots) return fail(ctx, B2A_ERR_STATE, "internal: segment count exceeds its bound");

        // ---- queue the copies of this segment's inputs ----
        cudaStream_t sc = ctx->s_copy;
        const uint64_t pb0 = pat_off[first], pb1 = pat_off[k], tb0 = txt_off[first], tb1 = txt_off[k];
        const uint64_t sb0[2] = {pb0, tb0}, sb1[2] = {pb1, tb1};
        uint64_t se0[2] = {0, 0}, se1[2] = {0, 0};                       // the segment's slice of each exception list
        if (!compact) {
            if (pb1 > pb0) CU(cudaMemcpyAsync(ctx->d_pat.p + pb0, pat + pb0, pb1 - pb0, cudaMemcpyHostToDevice, sc));
            if (tb1 > tb0) CU(cudaMemcpyAsync(ctx->d_txt.p + tb0, txt + tb0, tb1 - tb0, cudaMemcpyHostToDevice, sc));
            ctx->h2d += (pb1 - pb0) + (tb1 - tb0);
        } else {
            for (int w = 0; w < 2; ++w) {
                // code bytes [copied, ceil(b1 / 4)): a byte shared with the previous segment went up with that one
                const uint64_t c1 = (sb1[w] + 3) / 4;
                if (c1 > sq_copied[w]) {
                    CU(cudaMemcpyAsync(ctx->seq2[w].codes.p + sq_copied[w], sq[w]->codes + sq_copied[w], c1 - sq_copied[w], cudaMemcpyHostToDevice, sc));
                    ctx->h2d += c1 - sq_copied[w];
                    sq_copied[w] = c1;
                }
                uint64_t e = sq_exc[w];
                se0[w] = e;
                while (e < sq[w]->n_exc && sq[w]->exc_pos[e] < sb1[w]) {
                    if (sq[w]->exc_pos[e] < sb0[w] || (e > se0[w] && sq[w]->exc_pos[e] <= sq[w]->exc_pos[e - 1]))
                        return fail(ctx, B2A_ERR_ARG, "b2a_align_batch_multi_seq2: exception positions must ascend");
                    ++e;
                }
                se1[w] = sq_exc[w] = e;
                if (e > se0[w]) {
                    CU(cudaMemcpyAsync(ctx->seq2[w].epos.p + se0[w], sq[w]->exc_pos + se0[w], (e - se0[w]) * 8, cudaMemcpyHostToDevice, sc));
                    CU(cudaMemcpyAsync(ctx->seq2[w].ebyte.p + se0[w], sq[w]->exc_byte + se0[w], e - se0[w], cudaMemcpyHostToDevice, sc));
                    ctx->h2d += (e - se0[w]) * 9;
                }
            }
        }
        CU(cudaMemcpyAsync(ctx->d_pat_off.p + first, pat_off + first, (sg.count + 1) * 8, cudaMemcpyHostToDevice, sc));
        CU(cudaMemcpyAsync(ctx->d_txt_off.p + first, txt_off + first, (sg.count + 1) * 8, cudaMemcpyHostToDevice, sc));
        ctx->h2d += 2 * (sg.count + 1) * 8;

        // ---- pass 2 (overlaps the copies): zip pairs of identical shape into pair-pairs, group by R ----
        for (auto& v : pps) v.clear();
        pending.clear();
        bool have_last = false; uint64_t last_key = 0; uint32_t last_idx = 0;
        plan_key = ~0ull; plan_ok = false;
        for (uint64_t q = first; q < k; ++q) {
            const uint64_t m64 = pat_off[q + 1] - pat_off[q], n64 = txt_off[q + 1] - txt_off[q];
            const uint32_t m = (uint32_t)m64, n = (uint32_t)n64;
            const uint64_t key = (m64 << 32) | n64;
            if (key != plan_key) { plan_key = key; plan_ok = !score_only && plan_all(m, n, pl); }
            if (!plan_ok) { ctx->wide_pairs.push_back((uint32_t)q); ++sg.n_wide; continue; }
            if (have_last && key == last_key) { pps[pl.R].push_back(PPDesc{last_idx, (uint32_t)q, pp_pack(m, m), pp_pack(n, n)}); have_last = false; continue; }
            if (have_last) {                                             // the previous pair found no neighbour: park it
                auto it = pending.find(last_key);
                const uint32_t lm = (uint32_t)(last_key >> 32), ln = (uint32_t)last_key;
                if (it != pending.end()) { pps[short16_R(lm)].push_back(PPDesc{it->second, last_idx, pp_pack(lm, lm), pp_pack(ln, ln)}); pending.erase(it); }
                else pending[last_key] = last_idx;
                have_last = false;
            }
            auto it = pending.find(key);
            if (it != pending.end()) { pps[pl.R].push_back(PPDesc{it->second, (uint32_t)q, pp_pack(m, m), pp_pack(n, n)}); pending.erase(it); }
            else { have_last = true; last_key = key; last_idx = (uint32_t)q; }
        }
        if (have_last) {
            auto it = pending.find(last_key);
            const uint32_t lm = (uint32_t)(last_key >> 32), ln = (uint32_t)last_key;
            if (it != pending.end()) { pps[short16_R(lm)].push_back(PPDesc{it->second, last_idx, pp_pack(lm, lm), pp_pack(ln, ln)}); pending.erase(it); }
            else pending[last_key] = last_idx;
        }
        // Leftovers (one per distinct shape): zip pairs of DIFFERENT shapes, neighbours in (rows per lane, n, m) order so that little
        // is padded.  Safe for NW always (the score is read at the true end cell) and for semi-global mode (its epilogue scans only
        // the pair's own row m, columns 0..n, and its walk only the pair's own cells); for SW the junk columns of the shorter text must
        // stay strictly below the real maximum, which needs gap < 0 and mismatch < 0.  What still has no partner runs as a singleton
        // (both halves carry the same pair).
        {
            struct Left { int R; uint32_t n, m, idx; };
            std::vector<Left> left;
            left.reserve(pending.size());
            for (auto& kv : pending) { const uint32_t lm = (uint32_t)(kv.first >> 32), ln = (uint32_t)kv.first; left.push_back(Left{short16_R(lm), ln, lm, kv.second}); }
            std::sort(left.begin(), left.end(), [](const Left& x, const Left& y) {
                return x.R != y.R ? x.R < y.R : (x.n != y.n ? x.n < y.n : (x.m != y.m ? x.m < y.m : x.idx < y.idx)); });
            static const bool no_mix = std::getenv("B2A_NO_MIX") != nullptr;           // A/B switch for scripts/ragged_exp.py
            const bool mix_ok = !no_mix && (!any_local || (prm->gap < 0 && prm->mismatch < 0));
            for (size_t q = 0; q < left.size(); ++q) {
                const Left& x = left[q];
                if (mix_ok && q + 1 < left.size() && left[q + 1].R == x.R) {
                    const Left& y = left[q + 1];
                    Short16Plan both{0, 0, 0};
                    if (plan_all(std::max(x.m, y.m), std::max(x.n, y.n), both) && both.R == x.R) {
                        const bool xfirst = x.idx < y.idx;               // low half = lower pair index (deterministic records)
                        const Left& lo = xfirst ? x : y; const Left& hi = xfirst ? y : x;
                        pps[x.R].push_back(PPDesc{lo.idx, hi.idx, pp_pack(lo.m, hi.m), pp_pack(lo.n, hi.n)});
                        ++q;
                        continue;
                    }
                }
                pps[x.R].push_back(PPDesc{x.idx, x.idx, pp_pack(x.m, x.m), pp_pack(x.n, x.n)});
            }
        }
        PPDesc* hp = ctx->h_pps.p + sg.pp_first;
        uint64_t* hc = ctx->h_code_off.p + sg.pp_first;
        uint64_t npp = 0, chunks = 0, rb = 0;
        for (int R = 1; R <= SHORT16_MAX_R; ++R) {
            if (pps[R].empty()) continue;
            ClassRange cr{R, (uint32_t)npp, (uint32_t)pps[R].size(), 0};
            for (const PPDesc& d : pps[R]) {
                hp[npp] = d; hc[npp] = chunks; ++npp;
                chunks += (uint64_t)R * num_chunks(pp_max(d.n), CS) * 32u;
                cr.max_n = std::max(cr.max_n, pp_max(d.n));
            }
            rb = std::max<uint64_t>(rb, (uint64_t)(cr.first + cr.count) * R * 32u);
            sg.classes.push_back(cr);
        }
        sg.n_pp = npp; sg.chunks = chunks; sg.rowbest_words = any_local ? rb : 0;
        ctx->n_pp_total += npp;
        ctx->fill_bytes += chunks * sizeof(Chunk);
        if (npp) {
            CU(cudaMemcpyAsync(ctx->d_pps.p + sg.pp_first, hp, npp * sizeof(PPDesc), cudaMemcpyHostToDevice, sc));
            CU(cudaMemcpyAsync(ctx->d_code_off.p + sg.pp_first, hc, npp * 8, cudaMemcpyHostToDevice, sc));
            ctx->h2d += npp * (sizeof(PPDesc) + 8);
        }
        if (want_ops) {
            ctx->h_ops_off.p[k] = opsw;                                  // rewritten by the next segment with the same value
            CU(cudaMemcpyAsync(ctx->d_ops_off.p + first, ctx->h_ops_off.p + first, (sg.count + 1) * 8, cudaMemcpyHostToDevice, sc));
            ctx->h2d += (sg.count + 1) * 8;
        }
        // pattern alphabet of the segment, on the device, in copy-stream order right behind the bytes
        cudaEvent_t* ev = seg_events(ctx, si);
        if (!ev) return fail(ctx, B2A_ERR_CUDA, "cudaEventCreate failed");
        CU(cudaEventRecord(ev[0], sc));
        // Pattern alphabet of the segment, found on the device.  NOT on the copy stream: a kernel there
        // queues behind the running traceback and stalls every later copy (measured: +25 % end to end).
        CU(cudaStreamWaitEvent(ctx->s_fill, ev[0], 0));
        for (int w = 0; compact && w < 2; ++w) {                         // codes -> bytes in HBM, ahead of everything that reads the segment
            if (sb1[w] == sb0[w]) continue;
            uint8_t* out = w ? ctx->d_txt.p : ctx->d_pat.p;
            const uint64_t groups = (sb1[w] + 15) / 16 - sb0[w] / 16;
            seq2_expand_kernel<<<(unsigned)((groups + 255) / 256), 256, 0, ctx->s_fill>>>(ctx->seq2[w].codes.p, out, sb0[w], sb1[w], sq_alpha[w]);
            CU(cudaGetLastError());
            ++launches;
            if (se1[w] > se0[w]) {
                const uint64_t ne = se1[w] - se0[w];
                seq2_patch_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, ctx->s_fill>>>(out, ctx->seq2[w].epos.p + se0[w], ctx->seq2[w].ebyte.p + se0[w], ne);
                CU(cudaGetLastError());
                ++launches;
            }
        }
        if (pb1 > pb0) {
            const unsigned grid = (unsigned)std::min<uint64_t>((uint64_t)ctx->sm_count * 4u, (pb1 - pb0 + 4095) / 4096);
            alphabet_kernel<<<grid, 256, 0, ctx->s_fill>>>(ctx->d_pat.p + pb0, pb1 - pb0, ctx->d_hist.p + si * 256);
            CU(cudaGetLastError());
            ++launches;
        }
        alphabet_finish_kernel<<<1, 32, 0, ctx->s_fill>>>(ctx->d_alpha.p + si, ctx->d_hist.p + si * 256);
        CU(cudaGetLastError());
        ++launches;
        if (npp) {                                                       // exits at once unless the segment holds a fifth pattern symbol
            dirty_kernel<<<(unsigned)((npp + 255) / 256), 256, 0, ctx->s_fill>>>(ctx->d_pat.p, ctx->d_pat_off.p, ctx->d_pps.p + sg.pp_first, (uint32_t)npp,
                                                                                  ctx->d_alpha.p + si, ctx->d_dirty.p + sg.pp_first);
            CU(cudaGetLastError());
            ++launches;
            if (sg.classes.size() > DIRTY_CLASSES) return fail(ctx, B2A_ERR_STATE, "internal: more short16 classes than counters");
            for (size_t ci = 0; ci < sg.classes.size(); ++ci) {          // exits at once as well
                const ClassRange& c = sg.classes[ci];
                dirty_compact_kernel<<<(c.count + 255) / 256, 256, 0, ctx->s_fill>>>(ctx->d_dirty.p + sg.pp_first + c.first, c.count, ctx->d_alpha.p + si,
                                                                                       ctx->d_dirty_list.p + sg.pp_first + c.first, ctx->d_dirty_cnt.p + si * DIRTY_CLASSES + ci);
                CU(cudaGetLastError());
                ++launches;
            }
        }
        if (ctx->trace) tr_host.push_back(ms_since(t_begin));

        if (pipelined) {
            for (uint32_t r = 0; r < n_runs; ++r) {              // every run's kernels follow the ONE upload of the segment
                int rc = launch_segment(ctx, si, (int)r, &launches);
                if (rc != B2A_OK) return rc;
                if ((async_down || sink) && !sg.classes.empty()) {
                    cudaEvent_t* evr = seg_events(ctx, si, (int)r);
                    CU(cudaStreamWaitEvent(ctx->s_down, evr[3], 0));
                }
                if (async_down && !sg.classes.empty()) {
                    CU(cudaMemcpyAsync(results[r] + first, ctx->run[r].d_results.p + first, sg.count * sizeof(b2a_result), cudaMemcpyDeviceToHost, ctx->s_down));
                    ctx->d2h += sg.count * sizeof(b2a_result);
                }
                if (sink && !sg.classes.empty()) {
                    const uint64_t w0 = ctx->h_ops_off.p[first];                  // the segment's words: [w0, opsw)
                    if (opsw > ctx->ops_sink_cap) return fail(ctx, B2A_ERR_ARG, "b2a_set_ops_sink: the op lists of this batch do not fit the sink");
                    CU(cudaMemcpyAsync(ctx->ops_sink[r] + w0, ctx->run[r].d_ops.p + w0, (opsw - w0) * 4, cudaMemcpyDeviceToHost, ctx->s_down));
                    ctx->d2h += (opsw - w0) * 4;
                }
            }
        }
        if (ctx->trace) tr_host.push_back(ms_since(t_begin));
        first = k;
    }
    ctx->h_ops_off.p[n_pairs] = opsw;
    ctx->total_ops_words = opsw;
    ctx->cells = cells;

    // ---- everything is queued: wait for the segments, collect the alphabets, decide what wide32 has to serve ----
    cudaStream_t s0 = ctx->s_fill;
    { int rc = join_tracebacks(ctx); if (rc != B2A_OK) return rc; }
    CU(cudaMemcpyAsync(ctx->h_alpha.p, ctx->d_alpha.p, ctx->alpha_slots * sizeof(AlphaInfo), cudaMemcpyDeviceToHost, s0));
    CU(cudaStreamSynchronize(s0));
    AlphaInfo batch_alpha{};
    bool any_dirty = false;
    for (size_t si = 0; si < ctx->segs.size(); ++si) {
        const AlphaInfo& a = ctx->h_alpha.p[si];
        for (int w = 0; w < 8; ++w) batch_alpha.mask[w] |= a.mask[w];
        any_dirty |= a.too_many && ctx->segs[si].n_pp;
    }
    if (any_dirty) {
        // some segment holds a fifth pattern symbol: pair-pairs with MORE THAN 7 distinct pattern symbols were skipped by the s16x2 kernels
        // (the 8-symbol kernel raised their flag to 2); wide32 serves their pairs
        CU(cudaMemcpyAsync(ctx->h_dirty.p, ctx->d_dirty.p, ctx->n_pp_total, cudaMemcpyDeviceToHost, s0));
        CU(cudaStreamSynchronize(s0));
        ctx->d2h += ctx->n_pp_total;
        const size_t before = ctx->wide_pairs.size();
        for (uint64_t q = 0; q < ctx->n_pp_total; ++q)
            if (ctx->h_dirty.p[q] == 2) {                      // 1 = served by the 8-symbol s16x2 kernel
                const PPDesc& d = ctx->h_pps.p[q];
                ctx->wide_pairs.push_back(d.a); if (d.b != d.a) ctx->wide_pairs.push_back(d.b);
            }
        if (ctx->wide_pairs.size() != before) std::sort(ctx->wide_pairs.begin(), ctx->wide_pairs.end());
    }
    alpha_from_mask(batch_alpha);
    ctx->h_alpha.p[ctx->alpha_slots - 1] = batch_alpha;
    if (!ctx->wide_pairs.empty()) {
        CU(cudaMemcpyAsync(ctx->d_alpha.p + (ctx->alpha_slots - 1), ctx->h_alpha.p + (ctx->alpha_slots - 1), sizeof(AlphaInfo), cudaMemcpyHostToDevice, s0));
        int rc = wide_plan(ctx, pat_off, txt_off, !score_only, !batch_alpha.too_many, s0);
        if (rc != B2A_OK) return rc;
    } else { ctx->wide.pairs.clear(); ctx->wide.tasks.clear(); }

    if (!pipelined) {
        // resident mode: size the lanes' records now so that b2a_batch_run never allocates
        uint64_t nl = 0;                                          // b2a_batch_run hands the lanes out in launch order
        for (const Segment& sg : ctx->segs) {
            if (sg.classes.empty()) continue;
            Lane& ln = ctx->lanes[nl++ % (uint64_t)ctx->n_lanes];
            CU(ln.codes.reserve(sg.chunks));
            if (any_local) CU(ln.rowbest.reserve(sg.rowbest_words));
        }
        CU(cudaStreamSynchronize(s0));
        ctx->launches = launches;
        ctx->have_batch = true;
        return B2A_OK;
    }

    // ---- pipelined mode: the wide32 phase (if any) runs behind the segments, then the records come back ----
    for (uint32_t r = 0; r < n_runs && !ctx->wide_pairs.empty(); ++r) {     // one record, the runs take turns in stream order
        int rc = wide_fill(ctx, (int)r, s0, &launches);
        if (rc != B2A_OK) return rc;
        rc = wide_traceback(ctx, (int)r, s0, &launches, score_only);
        if (rc != B2A_OK) return rc;
        rc = wide_ckpt_run(ctx, (int)r, s0, &launches);
        if (rc != B2A_OK) return rc;
    }
    CU(cudaStreamSynchronize(s0));
    if (n_pairs && (!async_down || !ctx->wide_pairs.empty())) {
        for (uint32_t r = 0; r < n_runs; ++r)
            CU(cudaMemcpyAsync(results[r], ctx->run[r].d_results.p, n_pairs * sizeof(b2a_result), cudaMemcpyDeviceToHost, ctx->s_down));
        ctx->d2h = n_runs * n_pairs * sizeof(b2a_result);
    }
    if (sink && !ctx->wide_pairs.empty()) {                      // wide32 wrote its pairs' op lists after the segments were copied
        if (opsw > ctx->ops_sink_cap) return fail(ctx, B2A_ERR_ARG, "b2a_set_ops_sink: the op lists of this batch do not fit the sink");
        for (uint32_t r = 0; r < n_runs; ++r)
            CU(cudaMemcpyAsync(ctx->ops_sink[r], ctx->run[r].d_ops.p, opsw * 4, cudaMemcpyDeviceToHost, ctx->s_down));
        ctx->d2h += n_runs * opsw * 4;
    }
    CU(cudaStreamSynchronize(ctx->s_down));
    if (ctx->trace) {
        std::fprintf(stderr, "[b2a trace] %llu pairs, %zu segments, host total %.2f ms\n", (unsigned long long)n_pairs, ctx->segs.size(), ms_since(t_begin));
        for (size_t si = 0; si < ctx->segs.size(); ++si) {
            const Segment& sg = ctx->segs[si];
            cudaEvent_t* ev = seg_events(ctx, si, 0);
            float g[4] = {0, 0, 0, 0};
            for (int e = 0; e < 4; ++e) if (e == 0 || !sg.classes.empty()) cudaEventElapsedTime(&g[e], ctx->ev_begin, ev[e]);
            std::fprintf(stderr, "[b2a trace] seg %2zu pairs %7llu | host: scanned %6.2f planned %6.2f launched %6.2f | device: inputs %6.2f fill %6.2f..%6.2f tb ..%6.2f\n",
                         si, (unsigned long long)sg.count, tr_host[3 * si], tr_host[3 * si + 1], tr_host[3 * si + 2], g[0], g[1], g[2], g[3]);
        }
        cudaGetLastError();
    }
    ctx->launches = launches;
    ctx->have_batch = true; ctx->ran = true;
    return B2A_OK;
}

} // namespace

extern "C" {

int b2a_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

b2a_ctx* b2a_create(int device) {
    int n = b2a_device_count();
    if (device < 0 || device >= n) return nullptr;
    b2a_ctx* ctx = new (std::nothrow) b2a_ctx();
    if (!ctx) return nullptr;
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess ||
        prop.major < 10) {                                   // kernels are sm_100a only: no fallback
        delete ctx; cudaGetLastError(); return nullptr;
    }
    ctx->sm_count = prop.multiProcessorCount;
    set_kernel_attributes();
    if (const char* e = std::getenv("B2A_TRACE")) ctx->trace = std::atoi(e) != 0;
    if (const char* e = std::getenv("B2A_LANES")) ctx->lanes_cfg = std::max(0, std::min(MAX_LANES, std::atoi(e)));
    if (const char* e = std::getenv("B2A_SEG_MB")) ctx->seg_budget_bytes = std::max<uint64_t>(1, std::strtoull(e, nullptr, 10)) << 20;
    if (const char* e = std::getenv("B2A_SEG_PAIRS")) { ctx->seg_max_pairs = ctx->seg_resident_pairs = std::max<uint64_t>(SEG_MIN_PAIRS, std::strtoull(e, nullptr, 10)); ctx->seg_user = true; }
    if (const char* e = std::getenv("B2A_SEG_FIRST")) { ctx->seg_first_pairs = std::max<uint64_t>(SEG_MIN_PAIRS, std::strtoull(e, nullptr, 10)); ctx->seg_user = true; }
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);   // numerically lower = higher priority
    bool ok = cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&ctx->s_down, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithPriority(&ctx->s_fill, cudaStreamNonBlocking, prio_lo) == cudaSuccess &&
              cudaEventCreate(&ctx->ev_begin) == cudaSuccess && cudaEventCreate(&ctx->ev_end) == cudaSuccess;
    for (int l = 0; l < MAX_LANES && ok; ++l)
        ok = cudaEventCreateWithFlags(&ctx->lanes[l].tb_done, cudaEventDisableTiming) == cudaSuccess &&
             cudaStreamCreateWithPriority(&ctx->lanes[l].s_tb, cudaStreamNonBlocking, prio_hi) == cudaSuccess &&
             cudaStreamCreateWithPriority(&ctx->lanes[l].s_tb_lo, cudaStreamNonBlocking, prio_lo) == cudaSuccess;

    if (!ok) { b2a_destroy(ctx); cudaGetLastError(); return nullptr; }
    return ctx;
}

void b2a_destroy(b2a_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->s_copy) cudaStreamSynchronize(ctx->s_copy);
    if (ctx->s_down) cudaStreamSynchronize(ctx->s_down);
    if (ctx->s_fill) cudaStreamSynchronize(ctx->s_fill);
    for (auto& ln : ctx->lanes) { if (ln.s_tb) cudaStreamSynchronize(ln.s_tb); if (ln.s_tb_lo) cudaStreamSynchronize(ln.s_tb_lo); }
    for (auto& ln : ctx->lanes) {
        ln.codes.release(); ln.rowbest.release();
        if (ln.tb_done) cudaEventDestroy(ln.tb_done);
    }
    if (ctx->s_fill) cudaStreamDestroy(ctx->s_fill);
    for (auto& ln : ctx->lanes) { if (ln.s_tb) cudaStreamDestroy(ln.s_tb); if (ln.s_tb_lo) cudaStreamDestroy(ln.s_tb_lo); }
    ctx->d_pat.release(); ctx->d_txt.release(); ctx->d_pat_off.release(); ctx->d_txt_off.release();
    ctx->d_code_off.release(); ctx->d_ops_off.release(); ctx->d_pps.release();
    ctx->seq2[0].release(); ctx->seq2[1].release();
    ctx->d_alpha.release(); ctx->d_nops.release(); ctx->d_hist.release(); ctx->d_dirty.release(); ctx->d_dirty_list.release(); ctx->d_dirty_cnt.release(); ctx->h_dirty.release();
    for (auto& rb : ctx->run) rb.release();
    ctx->h_pps.release(); ctx->h_code_off.release(); ctx->h_ops_off.release(); ctx->h_alpha.release();
    ctx->wide.release();
    for (auto& e : ctx->ev_pool) if (e) cudaEventDestroy(e);
    if (ctx->ev_begin) cudaEventDestroy(ctx->ev_begin);
    if (ctx->ev_end) cudaEventDestroy(ctx->ev_end);
    if (ctx->s_copy) cudaStreamDestroy(ctx->s_copy);
    if (ctx->s_down) cudaStreamDestroy(ctx->s_down);
    delete ctx;
}

const char* b2a_last_error(const b2a_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context (CUDA device unavailable?)"; }

void* b2a_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void b2a_host_free(void* p) { if (p) cudaFreeHost(p); }

int b2a_batch_upload(b2a_ctx* ctx, const b2a_params* prm, const uint8_t* pat, const uint64_t* pat_off,
                     const uint8_t* txt, const uint64_t* txt_off, uint64_t n_pairs)
{
    return batch_prepare(ctx, prm, 1, pat, pat_off, txt, txt_off, n_pairs, false, nullptr);
}

int b2a_batch_run(b2a_ctx* ctx, float* fill_ms, float* traceback_ms)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!ctx->have_batch) return fail(ctx, B2A_ERR_STATE, "b2a_batch_run: no batch uploaded");
    CU(cudaSetDevice(ctx->device));
    const b2a_params& prm = ctx->prm;
    const bool score_only = (prm.flags & B2A_SCORE_ONLY) != 0;
    uint64_t launches = 0;
    cudaStream_t s0 = ctx->s_fill;
    ctx->n_launched = 0;
    CU(cudaEventRecord(ctx->ev_begin, s0));
    for (size_t si = 0; si < ctx->segs.size(); ++si) {
        int rc = launch_segment(ctx, si, 0, &launches);
        if (rc != B2A_OK) return rc;
    }
    { int rc = join_tracebacks(ctx); if (rc != B2A_OK) return rc; }
    cudaEvent_t* wev = seg_events(ctx, ctx->segs.size());          // spare slot: wide32 phase
    if (!wev) return fail(ctx, B2A_ERR_CUDA, "cudaEventCreate failed");
    CU(cudaEventRecord(wev[1], s0));
    if (!ctx->wide_pairs.empty()) { int rc = wide_fill(ctx, 0, s0, &launches); if (rc != B2A_OK) return rc; }
    CU(cudaEventRecord(wev[2], s0));
    if (!ctx->wide_pairs.empty()) { int rc = wide_traceback(ctx, 0, s0, &launches, score_only); if (rc != B2A_OK) return rc; }
    if (!ctx->wide_pairs.empty()) { int rc = wide_ckpt_run(ctx, 0, s0, &launches); if (rc != B2A_OK) return rc; }
    CU(cudaEventRecord(wev[3], s0));
    CU(cudaEventRecord(ctx->ev_end, s0));
    CU(cudaStreamSynchronize(s0));
    float f = 0, t = 0, tot = 0, x = 0;
    for (size_t si = 0; si <= ctx->segs.size(); ++si) {
        if (si < ctx->segs.size() && ctx->segs[si].classes.empty()) continue;
        cudaEvent_t* ev = seg_events(ctx, si, 0);
        CU(cudaEventElapsedTime(&x, ev[1], ev[2])); f += x;
        CU(cudaEventElapsedTime(&x, ev[2], ev[3])); t += x;
    }
    CU(cudaEventElapsedTime(&tot, ctx->ev_begin, ctx->ev_end));
    if (fill_ms) *fill_ms = f;
    if (traceback_ms) *traceback_ms = t;
    ctx->last_fill_ms = f; ctx->last_tb_ms = t; ctx->last_total_ms = tot;
    ctx->launches += launches;
    ctx->ran = true;
    return B2A_OK;
}

int b2a_batch_times(const b2a_ctx* ctx, float* fill_ms, float* traceback_ms, float* total_ms)
{
    if (!ctx) return B2A_ERR_ARG;
    if (fill_ms) *fill_ms = ctx->last_fill_ms;
    if (traceback_ms) *traceback_ms = ctx->last_tb_ms;
    if (total_ms) *total_ms = ctx->last_total_ms;
    return B2A_OK;
}

int b2a_batch_download(b2a_ctx* ctx, b2a_result* results)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!ctx->ran) return fail(ctx, B2A_ERR_STATE, "b2a_batch_download: batch not run");
    if (!results && ctx->n_pairs) return fail(ctx, B2A_ERR_ARG, "b2a_batch_download: null results");
    CU(cudaSetDevice(ctx->device));
    if (ctx->n_pairs) {
        CU(cudaMemcpyAsync(results, ctx->run[ctx->sel_run].d_results.p, ctx->n_pairs * sizeof(b2a_result), cudaMemcpyDeviceToHost, ctx->s_down));
        CU(cudaStreamSynchronize(ctx->s_down));
        ctx->d2h += ctx->n_pairs * sizeof(b2a_result);
    }
    return B2A_OK;
}

int b2a_align_batch(b2a_ctx* ctx, const b2a_params* prm, const uint8_t* pat, const uint64_t* pat_off,
                    const uint8_t* txt, const uint64_t* txt_off, uint64_t n_pairs, b2a_result* results)
{
    return batch_prepare(ctx, prm, 1, pat, pat_off, txt, txt_off, n_pairs, true, &results);
}

int b2a_align_batch_multi(b2a_ctx* ctx, const b2a_params* prm, uint32_t n_runs, const uint8_t* pat, const uint64_t* pat_off,
                          const uint8_t* txt, const uint64_t* txt_off, uint64_t n_pairs, b2a_result* const* results)
{
    return batch_prepare(ctx, prm, n_runs, pat, pat_off, txt, txt_off, n_pairs, true, results);
}

int b2a_align_batch_multi_seq2(b2a_ctx* ctx, const b2a_params* prm, uint32_t n_runs, const b2a_seq2* pat, const uint64_t* pat_off,
                               const b2a_seq2* txt, const uint64_t* txt_off, uint64_t n_pairs, b2a_result* const* results)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!pat || !txt) return fail(ctx, B2A_ERR_ARG, "b2a_align_batch_multi_seq2: null b2a_seq2");
    return batch_prepare(ctx, prm, n_runs, nullptr, pat_off, nullptr, txt_off, n_pairs, true, results, pat, txt);
}

int b2a_set_ops_sink(b2a_ctx* ctx, uint32_t* const* ops_words, uint32_t n_runs, uint64_t cap_words)
{
    if (!ctx || n_runs > (uint32_t)MAX_RUNS) return B2A_ERR_ARG;
    ctx->ops_sink_runs = 0; ctx->ops_sink_cap = 0;
    if (!ops_words || n_runs == 0) return B2A_OK;
    for (uint32_t r = 0; r < n_runs; ++r) { if (!ops_words[r]) return fail(ctx, B2A_ERR_ARG, "b2a_set_ops_sink: null buffer"); ctx->ops_sink[r] = ops_words[r]; }
    ctx->ops_sink_runs = n_runs; ctx->ops_sink_cap = cap_words;
    return B2A_OK;
}

int b2a_select_run(b2a_ctx* ctx, uint32_t run)
{
    if (!ctx) return B2A_ERR_ARG;
    if (run >= ctx->n_runs) return fail(ctx, B2A_ERR_ARG, "b2a_select_run: the last batch had fewer runs");
    ctx->sel_run = run;
    return B2A_OK;
}

int b2a_host_register(void* p, size_t bytes)
{
    if (!p || !bytes) return B2A_ERR_ARG;
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) { cudaGetLastError(); return B2A_ERR_CUDA; }
    return B2A_OK;
}
int b2a_host_unregister(void* p)
{
    if (!p) return B2A_ERR_ARG;
    if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return B2A_ERR_CUDA; }
    return B2A_OK;
}

int b2a_affine_score_batch(b2a_ctx* ctx, int32_t match, int32_t mismatch, int32_t gap_open, int32_t gap_extend,
                           const uint8_t* pat, const uint64_t* pat_off, const uint8_t* txt, const uint64_t* txt_off,
                           uint64_t n_pairs, int32_t* scores)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!pat_off || !txt_off || (!scores && n_pairs)) return fail(ctx, B2A_ERR_ARG, "b2a_affine_score_batch: null argument");
    if (n_pairs > 0x7FFFFFF0ull) return fail(ctx, B2A_ERR_ARG, "b2a_affine_score_batch: too many pairs");
    const uint64_t pat_bytes = n_pairs ? pat_off[n_pairs] : 0, txt_bytes = n_pairs ? txt_off[n_pairs] : 0;
    if ((pat_bytes && !pat) || (txt_bytes && !txt)) return fail(ctx, B2A_ERR_ARG, "b2a_affine_score_batch: null sequence buffer");
    std::vector<AffSpec> specs(n_pairs);
    for (uint64_t k = 0; k < n_pairs; ++k) {
        if (pat_off[k + 1] < pat_off[k] || txt_off[k + 1] < txt_off[k])
            return fail(ctx, B2A_ERR_ARG, "b2a_affine_score_batch: offsets must be non-decreasing");
        const uint64_t m = pat_off[k + 1] - pat_off[k], n = txt_off[k + 1] - txt_off[k];
        if (m + n >= 0x7FFFFFF0ull) return fail(ctx, B2A_ERR_RANGE, "b2a_affine_score_batch: sequence too long");
        specs[k] = AffSpec{pat_off[k], txt_off[k], (uint32_t)m, (uint32_t)n};
    }
    return affine_run(ctx, match, mismatch, gap_open, gap_extend, pat, pat_bytes, txt, txt_bytes, false, specs, scores, false, nullptr);
}

int b2a_affine_align_batch(b2a_ctx* ctx, int32_t match, int32_t mismatch, int32_t gap_open, int32_t gap_extend,
                           const uint8_t* pat, const uint64_t* pat_off, const uint8_t* txt, const uint64_t* txt_off,
                           uint64_t n_pairs, int32_t* scores, uint32_t* n_ops)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!pat_off || !txt_off || (!scores && n_pairs)) return fail(ctx, B2A_ERR_ARG, "b2a_affine_align_batch: null argument");
    if (n_pairs > 0x7FFFFFF0ull) return fail(ctx, B2A_ERR_ARG, "b2a_affine_align_batch: too many pairs");
    const uint64_t pat_bytes = n_pairs ? pat_off[n_pairs] : 0, txt_bytes = n_pairs ? txt_off[n_pairs] : 0;
    if ((pat_bytes && !pat) || (txt_bytes && !txt)) return fail(ctx, B2A_ERR_ARG, "b2a_affine_align_batch: null sequence buffer");
    std::vector<AffSpec> specs(n_pairs);
    for (uint64_t k = 0; k < n_pairs; ++k) {
        if (pat_off[k + 1] < pat_off[k] || txt_off[k + 1] < txt_off[k])
            return fail(ctx, B2A_ERR_ARG, "b2a_affine_align_batch: offsets must be non-decreasing");
        const uint64_t m = pat_off[k + 1] - pat_off[k], n = txt_off[k + 1] - txt_off[k];
        if (m + n >= 0x7FFFFFF0ull) return fail(ctx, B2A_ERR_RANGE, "b2a_affine_align_batch: sequence too long");
        specs[k] = AffSpec{pat_off[k], txt_off[k], (uint32_t)m, (uint32_t)n};
    }
    return affine_run(ctx, match, mismatch, gap_open, gap_extend, pat, pat_bytes, txt, txt_bytes, false, specs, scores, true, n_ops);
}

int64_t b2a_affine_fetch_ops(b2a_ctx* ctx, uint64_t pair, char* ops, uint64_t ops_cap)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!ctx->affine_ops) return fail(ctx, B2A_ERR_STATE, "b2a_affine_fetch_ops: call b2a_affine_align_batch first");
    if (pair >= ctx->n_pairs) return fail(ctx, B2A_ERR_ARG, "b2a_affine_fetch_ops: pair index out of range");
    CU(cudaSetDevice(ctx->device));
    uint32_t n_ops = 0;
    CU(cudaMemcpy(&n_ops, ctx->d_nops.p + pair, 4, cudaMemcpyDeviceToHost));
    if (n_ops > ops_cap) return fail(ctx, B2A_ERR_ARG, "b2a_affine_fetch_ops: buffer too small");
    const uint64_t nw = ((uint64_t)n_ops + 15) / 16;
    std::vector<uint32_t> w(nw);
    if (nw) CU(cudaMemcpy(w.data(), ctx->run[0].d_ops.p + ctx->h_ops_off.p[pair], nw * 4, cudaMemcpyDeviceToHost));
    ctx->d2h += 4 + nw * 4;
    static const char L[4] = {'M', 'D', 'I', '?'};
    for (uint32_t t = 0; t < n_ops; ++t) ops[t] = L[(w[t >> 4] >> (2 * (t & 15))) & 3u];
    return (int64_t)n_ops;
}

int b2a_affine_star_scores(b2a_ctx* ctx, int32_t match, int32_t mismatch, int32_t gap_open, int32_t gap_extend,
                           const uint8_t* seqs, const uint64_t* seq_off, uint32_t n_seqs,
                           uint32_t pair_first, uint32_t pair_count, int32_t* pair_scores, int32_t* sum_scores, int64_t* center)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!seq_off || (n_seqs && !seqs && seq_off[n_seqs])) return fail(ctx, B2A_ERR_ARG, "b2a_affine_star_scores: null argument");
    const uint64_t total = (uint64_t)n_seqs * (n_seqs ? n_seqs - 1 : 0) / 2;
    if (pair_first > total) return fail(ctx, B2A_ERR_ARG, "b2a_affine_star_scores: pair range out of bounds");
    const uint64_t count = std::min<uint64_t>(pair_count, total - pair_first);
    std::vector<AffSpec> specs;
    std::vector<std::pair<uint32_t, uint32_t>> ij;
    uint64_t idx = 0;
    for (uint32_t i = 0; i < n_seqs; ++i)                                    // hw3.cpp:233-234: i < j, row-major
        for (uint32_t j = i + 1; j < n_seqs; ++j, ++idx) {
            if (idx < pair_first || idx >= pair_first + count) continue;
            if (seq_off[i + 1] < seq_off[i] || seq_off[j + 1] < seq_off[j]) return fail(ctx, B2A_ERR_ARG, "b2a_affine_star_scores: offsets must be non-decreasing");
            const uint64_t m = seq_off[i + 1] - seq_off[i], n = seq_off[j + 1] - seq_off[j];
            if (m + n >= 0x7FFFFFF0ull) return fail(ctx, B2A_ERR_RANGE, "b2a_affine_star_scores: sequence too long");
            specs.push_back(AffSpec{seq_off[i], seq_off[j], (uint32_t)m, (uint32_t)n});
            ij.emplace_back(i, j);
        }
    std::vector<int32_t> sc(specs.size());
    int rc = affine_run(ctx, match, mismatch, gap_open, gap_extend, seqs, n_seqs ? seq_off[n_seqs] : 0, nullptr, 0, true, specs, sc.data(), false, nullptr);
    if (rc != B2A_OK) return rc;
    if (pair_scores) std::copy(sc.begin(), sc.end(), pair_scores);
    std::vector<int32_t> sums(n_seqs, 0);                                    // hw3.cpp:238-239 (partial sums of this pair range)
    for (size_t k = 0; k < ij.size(); ++k) { sums[ij[k].first] += sc[k]; sums[ij[k].second] += sc[k]; }
    if (sum_scores) std::copy(sums.begin(), sums.end(), sum_scores);
    if (center) {                                                            // hw3.cpp:243-251: first strict maximum -- of COMPLETE sums only
        *center = -1;
        if (n_seqs && pair_first == 0 && count == total) {
            int64_t c = 0;
            for (uint32_t i = 1; i < n_seqs; ++i) if (sums[i] > sums[c]) c = i;
            *center = c;
        }
    }
    return B2A_OK;
}

int b2a_set_option(b2a_ctx* ctx, int option, int64_t value)
{
    if (!ctx) return B2A_ERR_ARG;
    switch (option) {
        case B2A_OPT_LANES:      if (value < 0 || value > MAX_LANES) break; ctx->lanes_cfg = (int)value; return B2A_OK;
        case B2A_OPT_SEG_PAIRS:  if (value < 1) break; ctx->seg_max_pairs = ctx->seg_resident_pairs = std::max<uint64_t>(SEG_MIN_PAIRS, (uint64_t)value); ctx->seg_user = true; return B2A_OK;
        case B2A_OPT_SEG_FIRST:  if (value < 1) break; ctx->seg_first_pairs = std::max<uint64_t>(SEG_MIN_PAIRS, (uint64_t)value); ctx->seg_user = true; return B2A_OK;
        case B2A_OPT_SEG_BYTES:  if (value < 1) break; ctx->seg_budget_bytes = (uint64_t)value; return B2A_OK;
        case B2A_OPT_CKPT_BYTES: if (value < 0) break; ctx->wide_ckpt_bytes = (uint64_t)value; return B2A_OK;
        case B2A_OPT_CKPT_GROUP: if (value < 1) break; ctx->wide_ckpt_group_bytes = (uint64_t)value; return B2A_OK;
        case B2A_OPT_CKPT_COLS:  if (value < 2 || value > 30) break; ctx->wide_ckpt_col_shift = (uint32_t)value; return B2A_OK;
    }
    return fail(ctx, B2A_ERR_ARG, "b2a_set_option: unknown option or bad value");
}

int b2a_batch_stats(const b2a_ctx* ctx, uint64_t* kernel_launches, uint64_t* cells, uint64_t* fill_bytes,
                    uint64_t* h2d_bytes, uint64_t* d2h_bytes)
{
    if (!ctx) return B2A_ERR_ARG;
    if (kernel_launches) *kernel_launches = ctx->launches;
    if (cells) *cells = ctx->cells;
    if (fill_bytes) *fill_bytes = ctx->fill_bytes;
    if (h2d_bytes) *h2d_bytes = ctx->h2d;
    if (d2h_bytes) *d2h_bytes = ctx->d2h;
    return B2A_OK;
}

int64_t b2a_fetch_ops(b2a_ctx* ctx, uint64_t pair, char* ops, uint64_t ops_cap)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!ctx->ran || !(ctx->prm.flags & B2A_WANT_OPS)) return fail(ctx, B2A_ERR_STATE, "b2a_fetch_ops: run a batch with B2A_WANT_OPS first");
    if (pair >= ctx->n_pairs) return fail(ctx, B2A_ERR_ARG, "b2a_fetch_ops: pair index out of range");
    CU(cudaSetDevice(ctx->device));
    PairResult r;
    const RunBuf& rb = ctx->run[ctx->sel_run];
    CU(cudaMemcpy(&r, rb.d_results.p + pair, sizeof(r), cudaMemcpyDeviceToHost));
    if (r.n_ops > ops_cap) return fail(ctx, B2A_ERR_ARG, "b2a_fetch_ops: buffer too small");
    const uint64_t nw = ((uint64_t)r.n_ops + 15) / 16;
    std::vector<uint32_t> w(nw);
    if (nw) CU(cudaMemcpy(w.data(), rb.d_ops.p + ctx->h_ops_off.p[pair], nw * 4, cudaMemcpyDeviceToHost));
    ctx->d2h += sizeof(r) + nw * 4;
    static const char L[4] = {'M', 'D', 'I', '?'};
    for (uint32_t t = 0; t < r.n_ops; ++t) ops[t] = L[(w[t >> 4] >> (2 * (t & 15))) & 3u];
    return (int64_t)r.n_ops;
}

int64_t b2a_copy_ops(b2a_ctx* ctx, uint32_t* ops_words, uint64_t cap_words, uint64_t* ops_off)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!ctx->ran || !(ctx->prm.flags & B2A_WANT_OPS)) return fail(ctx, B2A_ERR_STATE, "b2a_copy_ops: run a batch with B2A_WANT_OPS first");
    if (ops_off) std::memcpy(ops_off, ctx->h_ops_off.p, (ctx->n_pairs + 1) * 8);
    if (!ops_words) return (int64_t)ctx->total_ops_words;
    if (cap_words < ctx->total_ops_words) return fail(ctx, B2A_ERR_ARG, "b2a_copy_ops: buffer too small");
    CU(cudaSetDevice(ctx->device));
    if (ctx->total_ops_words) {
        CU(cudaMemcpyAsync(ops_words, ctx->run[ctx->sel_run].d_ops.p, ctx->total_ops_words * 4, cudaMemcpyDeviceToHost, ctx->s_down));
        CU(cudaStreamSynchronize(ctx->s_down));
        ctx->d2h += ctx->total_ops_words * 4;
    }
    return (int64_t)ctx->total_ops_words;
}

int64_t b2a_debug_copy_record(b2a_ctx* ctx, void* chunks, uint64_t chunk_cap, void* rowbest, uint64_t rowbest_cap)
{
    if (!ctx) return B2A_ERR_ARG;
    if (!ctx->ran || ctx->segs.empty() || ctx->segs[0].classes.empty())
        return fail(ctx, B2A_ERR_STATE, "b2a_debug_copy_record: no short16 record");
    // the first segment's record still sits in lane 0 only if no later (segment, run) launch reused that lane
    if (ctx->n_launched > (uint64_t)ctx->n_lanes)
        return fail(ctx, B2A_ERR_STATE, "b2a_debug_copy_record: the first segment's record has been overwritten (batch has more launches than lanes)");
    CU(cudaSetDevice(ctx->device));
    const Segment& sg = ctx->segs[0];
    const Lane& ln = ctx->lanes[0];
    const uint64_t bytes = sg.chunks * sizeof(Chunk);
    if (chunks) CU(cudaMemcpy(chunks, ln.codes.p, std::min<uint64_t>(bytes, chunk_cap), cudaMemcpyDeviceToHost));
    if (rowbest && ctx->run[0].mode == B2A_MODE_LOCAL)
        CU(cudaMemcpy(rowbest, ln.rowbest.p, std::min<uint64_t>(sg.rowbest_words * 4, rowbest_cap), cudaMemcpyDeviceToHost));
    return (int64_t)bytes;
}

int b2a_microbench_int16x2(b2a_ctx* ctx, int kind, double* gops, float* sm_mhz)
{
    if (!ctx || !gops) return B2A_ERR_ARG;
    CU(cudaSetDevice(ctx->device));
    double g = 0; float mhz = 0;
    cudaError_t e = run_microbench(kind, ctx->sm_count, ctx->s_fill, &g, &mhz);
    if (e != cudaSuccess) return cuda_fail(ctx, e, "microbench");
    *gops = g;
    if (sm_mhz) *sm_mhz = mhz;
    return B2A_OK;
}

} // extern "C"
