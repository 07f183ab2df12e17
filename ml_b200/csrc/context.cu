// Contexts (GPU sets), the resident point matrix, the synthetic generator and the deterministic
// partial-statistics reduction + exchange shared by the EM and K-means paths.
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <random>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "internal.h"

namespace mlb {

static thread_local std::string g_last_error = "";

void set_error(const char* fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
}

const NcclApi* nccl()
{
    static NcclApi api{};
    static bool ok = false;
    static std::string why;
    static std::once_flag once;
    std::call_once(once, [] {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // the copy the process already has (PyTorch's)
        if (!h) {
            const char* env = std::getenv("MLB200_NCCL_LIB");
            if (env && *env) h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
        }
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) { why = std::string("cannot load libnccl.so.2: ") + dlerror(); return; }
        bool all = true;
        auto bind = [&](auto& fn, const char* name) {
            fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(h, name));
            if (!fn) { all = false; why = std::string("libnccl.so.2 lacks ") + name; }
        };
        bind(api.GetUniqueId, "ncclGetUniqueId");
        bind(api.CommInitAll, "ncclCommInitAll");
        bind(api.CommInitRank, "ncclCommInitRank");
        bind(api.CommDestroy, "ncclCommDestroy");
        bind(api.AllGather, "ncclAllGather");
        bind(api.GroupStart, "ncclGroupStart");
        bind(api.GroupEnd, "ncclGroupEnd");
        bind(api.GetErrorString, "ncclGetErrorString");
        bind(api.GetVersion, "ncclGetVersion");
        ok = all;
    });
    if (!ok) { set_error("NCCL unavailable: %s", why.c_str()); return nullptr; }
    return &api;
}

constexpr size_t kBounceBytes = 4u << 20;
constexpr size_t kThreadedCopyBytes = 16u << 20;   // below this one thread does the whole copy

static int ensure_bounce(Gpu& gpu)
{
    for (int i = 0; i < 2 * kCopyThreadsMax; ++i) {
        if (!gpu.bounce[i]) {
            MLB_CUDA(cudaMallocHost(&gpu.bounce[i], kBounceBytes));
            MLB_CUDA(cudaEventCreateWithFlags(&gpu.bounce_ev[i], cudaEventDisableTiming));
        }
    }
    return MLB_OK;
}

static bool is_pinned_host(const void* ptr)
{
    cudaPointerAttributes attr{};
    if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess) {
        cudaGetLastError();   // older drivers report unregistered host memory as an error
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}

// Processes of a one-process-per-GPU job share the host's cores: every rank takes its share of the copy threads.
static int g_ranks_on_host = 1;

static int copy_threads(size_t bytes)
{
    if (bytes < kThreadedCopyBytes) return 1;
    const unsigned cores = std::max(1u, std::thread::hardware_concurrency());
    int t = static_cast<int>(std::min<unsigned>(kCopyThreadsMax, std::max(2u, g_ranks_on_host > 1 ? cores / static_cast<unsigned>(g_ranks_on_host) : cores / 2u)));
    if (const char* env = std::getenv("MLB200_COPY_THREADS")) t = std::max(1, std::min(kCopyThreadsMax, std::atoi(env)));
    return t;
}

// Runs body(t) on `threads` host threads (the caller is thread 0) and returns the first failure.
template <class F>
static int run_copy_threads(int threads, F&& body)
{
    std::vector<int> rc(static_cast<size_t>(threads), MLB_OK);
    std::vector<std::string> why(static_cast<size_t>(threads));
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; ++t)
        pool.emplace_back([&, t] {
            rc[t] = body(t);
            if (rc[t] != MLB_OK) why[t] = mlb_last_error();   // the error text is thread-local
        });
    rc[0] = body(0);
    for (std::thread& th : pool) th.join();
    for (int t = 0; t < threads; ++t)
        if (rc[t] != MLB_OK) {
            if (t > 0) set_error("%s", why[t].c_str());
            return rc[t];
        }
    return MLB_OK;
}

int staged_h2d(Gpu& gpu, void* dst_device, const void* src, size_t rows, size_t row_bytes, size_t src_stride)
{
    const size_t total = rows * row_bytes;
    if (total == 0) return MLB_OK;
    const bool contiguous = src_stride == row_bytes || rows == 1;
    if (total < (1u << 20) || is_pinned_host(src)) {
        if (contiguous) MLB_CUDA(cudaMemcpyAsync(dst_device, src, total, cudaMemcpyHostToDevice, gpu.stream));
        else MLB_CUDA(cudaMemcpy2DAsync(dst_device, row_bytes, src, src_stride, row_bytes, rows, cudaMemcpyHostToDevice, gpu.stream));
        return MLB_OK;
    }
    MLB_TRY(ensure_bounce(gpu));
    const size_t pieces = (total + kBounceBytes - 1) / kBounceBytes;
    const int threads = static_cast<int>(std::min<size_t>(copy_threads(total), pieces));
    const char* in = static_cast<const char*>(src);
    char* out = static_cast<char*>(dst_device);
    return run_copy_threads(threads, [&](int t) -> int {
        MLB_CUDA(cudaSetDevice(gpu.device));
        int turn = 0;
        for (size_t piece = static_cast<size_t>(t); piece < pieces; piece += static_cast<size_t>(threads), ++turn) {
            const int slot = 2 * t + (turn & 1);
            const size_t off = piece * kBounceBytes, len = std::min(kBounceBytes, total - off);
            MLB_CUDA(cudaEventSynchronize(gpu.bounce_ev[slot]));   // the last DMA out of this buffer (this call or an earlier one)
            char* stage = static_cast<char*>(gpu.bounce[slot]);
            if (contiguous) {
                std::memcpy(stage, in + off, len);
            } else {
                // logical bytes [off, off + len) of the dense image, gathered from the strided rows
                size_t row = off / row_bytes, col = off - row * row_bytes, done = 0;
                while (done < len) {
                    const size_t take = std::min(row_bytes - col, len - done);
                    std::memcpy(stage + done, in + row * src_stride + col, take);
                    done += take;
                    ++row;
                    col = 0;
                }
            }
            MLB_CUDA(cudaMemcpyAsync(out + off, stage, len, cudaMemcpyHostToDevice, gpu.stream));
            MLB_CUDA(cudaEventRecord(gpu.bounce_ev[slot], gpu.stream));
        }
        return MLB_OK;
    });
}

int staged_d2h_2d(Gpu& gpu, void* dst, size_t dst_stride, const void* src_device, size_t src_stride, size_t rows, size_t row_bytes)
{
    const size_t total = rows * row_bytes;
    if (total == 0) return MLB_OK;
    if (is_pinned_host(dst)) {
        if (rows == 1) MLB_CUDA(cudaMemcpyAsync(dst, src_device, row_bytes, cudaMemcpyDeviceToHost, gpu.stream));
        else MLB_CUDA(cudaMemcpy2DAsync(dst, dst_stride, src_device, src_stride, row_bytes, rows, cudaMemcpyDeviceToHost, gpu.stream));
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        return MLB_OK;
    }
    MLB_TRY(ensure_bounce(gpu));
    // pieces of at most kBounceBytes that never straddle a row
    const size_t per_row = (row_bytes + kBounceBytes - 1) / kBounceBytes;
    const size_t pieces = rows * per_row;
    const int threads = static_cast<int>(std::min<size_t>(copy_threads(total), pieces));
    char* out = static_cast<char*>(dst);
    const char* in = static_cast<const char*>(src_device);
    return run_copy_threads(threads, [&](int t) -> int {
        MLB_CUDA(cudaSetDevice(gpu.device));
        // two buffers per thread: the DMA of this thread's next piece runs while it copies the previous one out (the
        // destination is usually fresh memory, so this copy is where its pages are first touched: that, spread over the
        // threads, is what bounds a large download)
        char* prev_dst = nullptr;
        size_t prev_len = 0;
        int turn = 0;
        for (size_t piece = static_cast<size_t>(t); piece < pieces; piece += static_cast<size_t>(threads), ++turn) {
            const int slot = 2 * t + (turn & 1);
            const size_t row = piece / per_row, off = (piece - row * per_row) * kBounceBytes, len = std::min(kBounceBytes, row_bytes - off);
            MLB_CUDA(cudaMemcpyAsync(gpu.bounce[slot], in + row * src_stride + off, len, cudaMemcpyDeviceToHost, gpu.stream));
            MLB_CUDA(cudaEventRecord(gpu.bounce_ev[slot], gpu.stream));
            if (turn > 0) {
                MLB_CUDA(cudaEventSynchronize(gpu.bounce_ev[slot ^ 1]));
                std::memcpy(prev_dst, gpu.bounce[slot ^ 1], prev_len);
            }
            prev_dst = out + row * dst_stride + off;
            prev_len = len;
        }
        if (turn > 0) {
            const int last = 2 * t + ((turn - 1) & 1);
            MLB_CUDA(cudaEventSynchronize(gpu.bounce_ev[last]));
            std::memcpy(prev_dst, gpu.bounce[last], prev_len);
        }
        return MLB_OK;
    });
}

int staged_d2h(Gpu& gpu, void* dst, const void* src_device, size_t bytes)
{
    return staged_d2h_2d(gpu, dst, bytes, src_device, bytes, 1, bytes);
}

int KernelTimer::begin(cudaStream_t stream)
{
    if (!enabled || used / 2 >= kMaxLaunches) return MLB_OK;
    if (events.size() < used + 2) {
        events.resize(used + 2, nullptr);
        MLB_CUDA(cudaEventCreate(&events[used]));
        MLB_CUDA(cudaEventCreate(&events[used + 1]));
    }
    MLB_CUDA(cudaEventRecord(events[used], stream));
    return MLB_OK;
}

int KernelTimer::end(cudaStream_t stream)
{
    if (!enabled || used / 2 >= kMaxLaunches) return MLB_OK;
    MLB_CUDA(cudaEventRecord(events[used + 1], stream));
    used += 2;
    return MLB_OK;
}

int KernelTimer::total(double* total_ms, int64_t* launches)
{
    double sum = 0;
    for (size_t i = 0; i + 1 < used; i += 2) {
        MLB_CUDA(cudaEventSynchronize(events[i + 1]));
        float ms = 0;
        MLB_CUDA(cudaEventElapsedTime(&ms, events[i], events[i + 1]));
        sum += ms;
    }
    if (total_ms) *total_ms = sum;
    if (launches) *launches = static_cast<int64_t>(used / 2);
    return MLB_OK;
}

void KernelTimer::destroy()
{
    for (cudaEvent_t e : events)
        if (e) cudaEventDestroy(e);
    events.clear();
    used = 0;
}

Layout Layout::make(int64_t n_total)
{
    Layout lay;
    lay.n_total = n_total;
    // About 6 chunks per SM on each of 8 GPUs, in multiples of the 128-point tile, at most 2048
    // points: small enough to balance 148 SMs x up to 4 resident CTAs under the dynamic scheduler (a
    // 4096-point cap left 4.1 chunks per CTA at 10M points per GPU: a 10 % tail), large enough that the
    // per-chunk flush of partial statistics is noise.  Depends on n_total ONLY (never on the GPU count).
    int64_t c = n_total / (8 * kSmCount * 6);
    c = (c + 127) / 128 * 128;
    c = std::max<int64_t>(128, std::min<int64_t>(2048, c));
    // MLB200_CHUNK: developer override (a multiple of 128), used to reproduce on one GPU the chunking a larger job
    // has (the chunk size follows the TOTAL point count).  Every rank of a job must see the same value.
    if (const char* env = std::getenv("MLB200_CHUNK")) {
        const long v = std::atol(env);
        if (v >= 128 && v <= 4096 && v % 128 == 0) c = v;
    }
    lay.chunk = static_cast<int>(c);
    lay.n_chunks = (n_total + c - 1) / c;
    for (int v = 0; v <= kVirtualShards; ++v) lay.vshard_chunk[v] = lay.n_chunks * v / kVirtualShards;
    return lay;
}

// ---------------------------------------------------------------- reduction of chunk partials

struct VshardRanges {
    int64_t lo[kVirtualShards];  // local chunk index ranges, one per local virtual shard
    int64_t hi[kVirtualShards];
};

// out[v][e] = sum over the chunks of local virtual shard v of partials[c][e], in a fixed order that
// depends only on the shard's chunk list: 8 chunk lanes x 4 interleaved sequential accumulators,
// combined as (a0+a1)+(a2+a3) per lane and then by a fixed tree over the lanes.  Block (32, 8).
__global__ void reduce_partials_kernel(const double* __restrict__ partials, VshardRanges r, int s, double* __restrict__ out)
{
    __shared__ double lanes[8][33];
    const int e = blockIdx.x * 32 + threadIdx.x;
    const int v = blockIdx.y, ty = threadIdx.y;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    if (e < s) {
        const int64_t hi = r.hi[v];
        for (int64_t c = r.lo[v] + 4 * ty; c < hi; c += 32) {
            a0 += partials[c * s + e];
            if (c + 1 < hi) a1 += partials[(c + 1) * s + e];
            if (c + 2 < hi) a2 += partials[(c + 2) * s + e];
            if (c + 3 < hi) a3 += partials[(c + 3) * s + e];
        }
    }
    lanes[ty][threadIdx.x] = (a0 + a1) + (a2 + a3);
    __syncthreads();
    if (ty == 0 && e < s) {
        const int x = threadIdx.x;
        out[static_cast<int64_t>(v) * s + e] =
            ((lanes[0][x] + lanes[1][x]) + (lanes[2][x] + lanes[3][x])) + ((lanes[4][x] + lanes[5][x]) + (lanes[6][x] + lanes[7][x]));
    }
}

// Level 1 of the reduction: every run of kReduceGroup consecutive chunks of a virtual shard is summed by one block
// (same lane scheme as above, so each of the 8 lanes adds exactly 4 chunks), which spreads the read of the
// partials over thousands of blocks instead of 8 per column tile.  blockIdx.y = group index over all local shards.
constexpr int kReduceGroup = 32;

__global__ void reduce_groups_kernel(const double* __restrict__ partials, VshardRanges r, int nv, int s, double* __restrict__ out)
{
    __shared__ double lanes[8][33];
    int group = blockIdx.y, v = 0;
    for (; v < nv; ++v) {
        const int ng = static_cast<int>((r.hi[v] - r.lo[v] + kReduceGroup - 1) / kReduceGroup);
        if (group < ng) break;
        group -= ng;
    }
    if (v == nv) return;
    const int64_t lo = r.lo[v] + static_cast<int64_t>(group) * kReduceGroup;
    const int64_t hi = min(lo + kReduceGroup, r.hi[v]);
    const int e = blockIdx.x * 32 + threadIdx.x, ty = threadIdx.y;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    if (e < s) {
        const int64_t c = lo + 4 * ty;
        if (c < hi) a0 = partials[c * s + e];
        if (c + 1 < hi) a1 = partials[(c + 1) * s + e];
        if (c + 2 < hi) a2 = partials[(c + 2) * s + e];
        if (c + 3 < hi) a3 = partials[(c + 3) * s + e];
    }
    lanes[ty][threadIdx.x] = (a0 + a1) + (a2 + a3);
    __syncthreads();
    if (ty == 0 && e < s) {
        const int x = threadIdx.x;
        out[static_cast<int64_t>(blockIdx.y) * s + e] =
            ((lanes[0][x] + lanes[1][x]) + (lanes[2][x] + lanes[3][x])) + ((lanes[4][x] + lanes[5][x]) + (lanes[6][x] + lanes[7][x]));
    }
}

void ReduceScratch::release(mlb_ctx* ctx)
{
    for (size_t g = 0; g < ptr.size(); ++g)
        if (ptr[g]) {
            cudaSetDevice(ctx->gpus[g].device);
            cudaFreeAsync(ptr[g], ctx->gpus[g].stream);
        }
    ptr.clear();
    len.clear();
}

int reduce_and_exchange_units(mlb_data* data, const std::vector<double*>& partials, const std::vector<double*>& vsum, int s, ReduceScratch& scratch,
                              const int64_t* bounds)
{
    mlb_ctx* ctx = data->ctx;
    const int vpg = ctx->vshards_per_gpu();
    scratch.ptr.resize(ctx->gpus.size(), nullptr);
    scratch.len.resize(ctx->gpus.size(), 0);
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        const int64_t local_begin = bounds[gpu.rank * vpg];   // partials[g] starts at the first unit of this GPU's first shard
        VshardRanges r, rg;
        int64_t total_groups = 0;
        for (int j = 0; j < vpg; ++j) {
            const int v = gpu.rank * vpg + j;
            r.lo[j] = bounds[v] - local_begin;
            r.hi[j] = bounds[v + 1] - local_begin;
            rg.lo[j] = total_groups;
            total_groups += (r.hi[j] - r.lo[j] + kReduceGroup - 1) / kReduceGroup;
            rg.hi[j] = total_groups;
        }
        double* out = vsum[g] + static_cast<int64_t>(gpu.rank) * vpg * s;
        if (bounds[kVirtualShards] <= 2 * kReduceGroup * kVirtualShards) {
            // few chunks: one level.  (The choice depends on N only, never on the GPU count: the two orders differ.)
            reduce_partials_kernel<<<dim3((s + 31) / 32, vpg), dim3(32, 8), 0, gpu.stream>>>(partials[g], r, s, out);
            MLB_CUDA(cudaGetLastError());
            return MLB_OK;
        }
        const size_t need = static_cast<size_t>(total_groups) * s;
        if (scratch.len[g] < need) {
            if (scratch.ptr[g]) {
                MLB_CUDA(cudaFreeAsync(scratch.ptr[g], gpu.stream));   // stream-ordered: earlier readers are done first
                scratch.ptr[g] = nullptr;
                scratch.len[g] = 0;
            }
            MLB_CUDA(cudaMallocFromPoolAsync(&scratch.ptr[g], sizeof(double) * need, gpu.pool, gpu.stream));
            scratch.len[g] = need;
        }
        reduce_groups_kernel<<<dim3((s + 31) / 32, static_cast<unsigned>(total_groups)), dim3(32, 8), 0, gpu.stream>>>(partials[g], r, vpg, s, scratch.ptr[g]);
        MLB_CUDA(cudaGetLastError());
        reduce_partials_kernel<<<dim3((s + 31) / 32, vpg), dim3(32, 8), 0, gpu.stream>>>(scratch.ptr[g], rg, s, out);
        MLB_CUDA(cudaGetLastError());
        return MLB_OK;
    }));
    if (ctx->world > 1) {
        // ONE collective per iteration: every GPU contributes its 8/G shard vectors, in place.
        MLB_NCCL_API(api);
        MLB_NCCL(api, api->GroupStart());
        for (size_t g = 0; g < ctx->gpus.size(); ++g) {
            Gpu& gpu = ctx->gpus[g];
            const size_t count = static_cast<size_t>(vpg) * s;
            MLB_NCCL(api, api->AllGather(vsum[g] + static_cast<int64_t>(gpu.rank) * count, vsum[g], count, ncclDouble, gpu.comm, gpu.stream));
        }
        MLB_NCCL(api, api->GroupEnd());
    }
    return MLB_OK;
}

int reduce_and_exchange(mlb_data* data, const std::vector<double*>& partials, const std::vector<double*>& vsum, int s, ReduceScratch& scratch)
{
    return reduce_and_exchange_units(data, partials, vsum, s, scratch, data->lay.vshard_chunk);
}

// ---------------------------------------------------------------- column sums (data mean)

// One block per chunk; thread t owns coordinate t % d of every (blockDim/d)-th point, then a fixed
// shared-memory tree.  Deterministic.
__global__ void column_sum_kernel(const double* __restrict__ x, int64_t n_local, int d, int chunk, double* __restrict__ partials)
{
    extern __shared__ double sm[];
    const int64_t p0 = static_cast<int64_t>(blockIdx.x) * chunk;
    const int64_t p1 = min(p0 + chunk, n_local);
    const int lanes = blockDim.x / d;  // points handled concurrently
    const int t = threadIdx.x;
    const int c = t % d, lane = t / d;
    double acc = 0;
    if (lane < lanes) {
        for (int64_t p = p0 + lane; p < p1; p += lanes) acc += x[p * d + c];
    }
    sm[t] = (lane < lanes) ? acc : 0.0;
    __syncthreads();
    if (t < d) {
        double s = 0;
        for (int l = 0; l < lanes; ++l) s += sm[l * d + t];
        partials[static_cast<int64_t>(blockIdx.x) * d + t] = s;
    }
}

static int compute_shift(mlb_data* data)
{
    mlb_ctx* ctx = data->ctx;
    const int d = data->d;
    std::vector<double*> partials(ctx->gpus.size(), nullptr), vsum(ctx->gpus.size(), nullptr);
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        DataShard& sh = data->shards[g];
        MLB_CUDA(cudaMallocFromPoolAsync(&partials[g], sizeof(double) * std::max<int64_t>(1, sh.n_chunks()) * d, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&vsum[g], sizeof(double) * kVirtualShards * d, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(vsum[g], 0, sizeof(double) * kVirtualShards * d, gpu.stream));
        if (sh.n_chunks() > 0) {
            const int threads = std::max(d, 256 / d * d);
            column_sum_kernel<<<static_cast<unsigned>(sh.n_chunks()), threads, sizeof(double) * threads, gpu.stream>>>(
                sh.x, sh.n(), d, data->lay.chunk, partials[g]);
            MLB_CUDA(cudaGetLastError());
        }
        return MLB_OK;
    }));
    ReduceScratch scratch;
    const int rc_reduce = reduce_and_exchange(data, partials, vsum, d, scratch);
    scratch.release(ctx);
    MLB_TRY(rc_reduce);
    std::vector<double> host(static_cast<size_t>(kVirtualShards) * d);
    MLB_CUDA(cudaSetDevice(ctx->gpus[0].device));
    MLB_CUDA(cudaMemcpyAsync(host.data(), vsum[0], sizeof(double) * host.size(), cudaMemcpyDeviceToHost, ctx->gpus[0].stream));
    MLB_TRY(mlb_ctx_synchronize(ctx));
    data->shift.resize(d);
    for (int c = 0; c < d; ++c) data->shift[c] = tree8(host.data() + c, d) / static_cast<double>(data->lay.n_total);
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        DataShard& sh = data->shards[g];
        MLB_CUDA(cudaMallocFromPoolAsync(&sh.shift, sizeof(double) * d, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemcpyAsync(sh.shift, data->shift.data(), sizeof(double) * d, cudaMemcpyHostToDevice, gpu.stream));
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        MLB_CUDA(cudaFreeAsync(partials[g], gpu.stream));
        MLB_CUDA(cudaFreeAsync(vsum[g], gpu.stream));
        return MLB_OK;
    }));
    return MLB_OK;
}

// ---------------------------------------------------------------- feature standardisation (cppyml/cppyml/utils.py:8-28)

// Per block of rows: column sums of x (mean == nullptr) or of (x - mean)^2.  Thread t owns coordinate t % d of every
// (blockDim / d)-th point of the block's rows, then a fixed shared-memory order: deterministic.
__global__ void standardise_partial_kernel(const double* __restrict__ x, int64_t n, int d, int64_t rows_per_block, const double* __restrict__ mean,
                                           double* __restrict__ partials)
{
    extern __shared__ double sm[];
    const int64_t p0 = static_cast<int64_t>(blockIdx.x) * rows_per_block;
    const int64_t p1 = min(p0 + rows_per_block, n);
    const int lanes = blockDim.x / d, t = threadIdx.x, c = t % d, lane = t / d;
    double acc = 0;
    if (lane < lanes) {
        const double m = mean ? mean[c] : 0.0;
        for (int64_t p = p0 + lane; p < p1; p += lanes) {
            const double v = x[p * d + c] - m;
            acc += mean ? v * v : v;
        }
    }
    sm[t] = lane < lanes ? acc : 0.0;
    __syncthreads();
    if (t < d) {
        double s = 0;
        for (int l = 0; l < lanes; ++l) s += sm[l * d + t];
        partials[static_cast<int64_t>(blockIdx.x) * d + t] = s;
    }
}

// out[c] = f(sum over the blocks of partials[b][c]) in a fixed pairwise order; f = / n (mean) or sqrt(. / n) (biased std).
__global__ void standardise_finish_kernel(const double* __restrict__ partials, int nblocks, int d, int64_t n, int want_std, double* __restrict__ out)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d) return;
    // pairwise (tree) sum over the blocks: the accuracy of numpy's pairwise summation, in a fixed order
    double level[32];
    int filled = 0;   // bit i set: level[i] holds the sum of 2^i blocks
    for (int b = 0; b < nblocks; ++b) {
        double v = partials[static_cast<int64_t>(b) * d + c];
        int i = 0;
        while (filled & (1 << i)) {
            v += level[i];
            filled &= ~(1 << i);
            ++i;
        }
        level[i] = v;
        filled |= 1 << i;
    }
    double total = 0.0;
    bool first = true;
    for (int i = 0; i < 32; ++i)
        if (filled & (1 << i)) {
            total = first ? level[i] : total + level[i];
            first = false;
        }
    out[c] = want_std ? sqrt(total / static_cast<double>(n)) : total / static_cast<double>(n);
}

__global__ void standardise_apply_kernel(double* __restrict__ x, int64_t total, int d, const double* __restrict__ mean, const double* __restrict__ sd, int divide)
{
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = static_cast<int>(i % d);
    const double v = x[i] - mean[c];
    x[i] = divide ? v / sd[c] : v;
}

// ---------------------------------------------------------------- synthetic GMM generator

struct Philox {
    // Philox4x32-10 (Salmon et al., SC'11): counter-based, so point i is a pure function of (seed, i).
    static __host__ __device__ inline void round(uint32_t (&c)[4], uint32_t k0, uint32_t k1)
    {
        const uint64_t p0 = static_cast<uint64_t>(0xD2511F53u) * c[0];
        const uint64_t p1 = static_cast<uint64_t>(0xCD9E8D57u) * c[2];
        const uint32_t n0 = static_cast<uint32_t>(p1 >> 32) ^ c[1] ^ k0;
        const uint32_t n1 = static_cast<uint32_t>(p1);
        const uint32_t n2 = static_cast<uint32_t>(p0 >> 32) ^ c[3] ^ k1;
        const uint32_t n3 = static_cast<uint32_t>(p0);
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    }
    static __host__ __device__ inline void generate(uint64_t seed, uint64_t index, uint32_t stream, uint32_t (&out)[4])
    {
        uint32_t c[4] = {static_cast<uint32_t>(index), static_cast<uint32_t>(index >> 32), stream, 0u};
        uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            round(c, k0, k1);
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
    }
    // uniform in (0, 1) from 53 random bits
    static __host__ __device__ inline double u01(uint32_t hi, uint32_t lo)
    {
        const uint64_t bits = (static_cast<uint64_t>(hi) << 21) ^ (lo >> 11);
        return (static_cast<double>(bits & ((1ull << 53) - 1)) + 0.5) * (1.0 / 9007199254740992.0);
    }
};

constexpr int kMaxGenDim = 128;

__global__ void generate_gmm_kernel(double* __restrict__ x, int64_t begin, int64_t n_local, int d, int k, uint64_t seed,
                                    const double* __restrict__ means /*[k][d]*/, const double* __restrict__ chol /*[k][d][d] row-major lower*/,
                                    const double* __restrict__ cum_weights /*[k]*/)
{
    const int64_t p = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (p >= n_local) return;
    const uint64_t gi = static_cast<uint64_t>(begin + p);
    uint32_t r[4];
    Philox::generate(seed, gi, 0u, r);
    const double u = Philox::u01(r[0], r[1]);
    int comp = 0;
    while (comp < k - 1 && u >= cum_weights[comp]) ++comp;
    double z[kMaxGenDim];
    for (int j = 0; j < d; j += 2) {
        Philox::generate(seed, gi, 1u + static_cast<uint32_t>(j / 2), r);
        const double u1 = Philox::u01(r[0], r[1]), u2 = Philox::u01(r[2], r[3]);
        const double rad = sqrt(-2.0 * log(u1));
        double s, c;
        sincospi(2.0 * u2, &s, &c);
        z[j] = rad * c;
        if (j + 1 < d) z[j + 1] = rad * s;
    }
    const double* m = means + static_cast<int64_t>(comp) * d;
    const double* l = chol + static_cast<int64_t>(comp) * d * d;
    double* out = x + p * d;
    for (int a = 0; a < d; ++a) {
        double v = m[a];
        for (int b = 0; b <= a; ++b) v += l[a * d + b] * z[b];
        out[a] = v;
    }
}

}  // namespace mlb

using namespace mlb;

// ======================================================================= C-ABI: library, context

extern "C" {

int mlb_version(void) { return 100; }

const char* mlb_last_error(void) { return g_last_error.c_str(); }

int mlb_device_count(int* count)
{
    MLB_REQUIRE(count, "mlb_device_count: null argument");
    MLB_CUDA(cudaGetDeviceCount(count));
    return MLB_OK;
}

static bool valid_world(int w) { return w == 1 || w == 2 || w == 4 || w == 8; }

static int init_gpu(Gpu& gpu)
{
    MLB_CUDA(cudaSetDevice(gpu.device));
    MLB_CUDA(cudaStreamCreateWithFlags(&gpu.stream, cudaStreamNonBlocking));
    // All device buffers are stream-ordered allocations from a pool the context owns (never the device's default
    // pool, which other CUDA code in the process, e.g. PyTorch, may be using with its own settings).  The pool keeps
    // freed memory cached: a second fit reuses the first one's buffers instead of paying cudaMalloc / cudaFree
    // (milliseconds each at these sizes).  The pool is destroyed with the context.
    cudaMemPoolProps props{};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = gpu.device;
    MLB_CUDA(cudaMemPoolCreate(&gpu.pool, &props));
    uint64_t keep = UINT64_MAX;
    MLB_CUDA(cudaMemPoolSetAttribute(gpu.pool, cudaMemPoolAttrReleaseThreshold, &keep));
    MLB_CUDA(cudaEventCreate(&gpu.ev0));
    MLB_CUDA(cudaEventCreate(&gpu.ev1));
    return MLB_OK;
}

int mlb_ctx_create(const int* devices, int n_devices, mlb_ctx** out)
{
    MLB_REQUIRE(out, "mlb_ctx_create: null output");
    MLB_REQUIRE(valid_world(n_devices), "mlb_ctx_create: n_devices must be 1, 2, 4 or 8 (got %d)", n_devices);
    int available = 0;
    MLB_CUDA(cudaGetDeviceCount(&available));
    if (available < 1) {
        set_error("mlb_ctx_create: no CUDA device (this library has no CPU fallback)");
        return MLB_ECUDA;
    }
    auto* ctx = new mlb_ctx;
    ctx->world = n_devices;
    ctx->rank_mode = false;
    ctx->gpus.resize(n_devices);
    std::vector<int> devs(n_devices);
    for (int g = 0; g < n_devices; ++g) {
        devs[g] = devices ? devices[g] : g;
        if (devs[g] < 0 || devs[g] >= available) {
            set_error("mlb_ctx_create: device %d not available (%d visible)", devs[g], available);
            delete ctx;
            return MLB_EINVAL;
        }
        ctx->gpus[g].device = devs[g];
        ctx->gpus[g].rank = g;
        int rc = init_gpu(ctx->gpus[g]);
        if (rc != MLB_OK) { delete ctx; return rc; }
    }
    if (n_devices > 1) {
        const NcclApi* api = nccl();
        if (!api) { delete ctx; return MLB_ENCCL; }
        std::vector<ncclComm_t> comms(n_devices);
        ncclResult_t r = api->CommInitAll(comms.data(), n_devices, devs.data());
        if (r != ncclSuccess) {
            set_error("ncclCommInitAll failed: %s", api->GetErrorString(r));
            delete ctx;
            return MLB_ENCCL;
        }
        for (int g = 0; g < n_devices; ++g) ctx->gpus[g].comm = comms[g];
    }
    *out = ctx;
    return MLB_OK;
}

int mlb_nccl_unique_id(void* out128)
{
    MLB_REQUIRE(out128, "mlb_nccl_unique_id: null output");
    static_assert(sizeof(ncclUniqueId) == MLB_NCCL_UNIQUE_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId id;
    MLB_NCCL_API(api);
    MLB_NCCL(api, api->GetUniqueId(&id));
    std::memcpy(out128, &id, sizeof(id));
    return MLB_OK;
}

int mlb_ctx_create_rank(int device, int rank, int world, const void* nccl_unique_id128, mlb_ctx** out)
{
    MLB_REQUIRE(out, "mlb_ctx_create_rank: null output");
    MLB_REQUIRE(valid_world(world), "mlb_ctx_create_rank: world must be 1, 2, 4 or 8 (got %d)", world);
    MLB_REQUIRE(rank >= 0 && rank < world, "mlb_ctx_create_rank: bad rank %d of %d", rank, world);
    MLB_REQUIRE(world == 1 || nccl_unique_id128, "mlb_ctx_create_rank: NCCL unique id required for world > 1");
    int available = 0;
    MLB_CUDA(cudaGetDeviceCount(&available));
    MLB_REQUIRE(device >= 0 && device < available, "mlb_ctx_create_rank: device %d not available (%d visible)", device, available);
    auto* ctx = new mlb_ctx;
    ctx->world = world;
    ctx->rank_mode = true;
    g_ranks_on_host = world;
    ctx->gpus.resize(1);
    ctx->gpus[0].device = device;
    ctx->gpus[0].rank = rank;
    int rc = init_gpu(ctx->gpus[0]);
    if (rc != MLB_OK) { delete ctx; return rc; }
    if (world > 1) {
        ncclUniqueId id;
        std::memcpy(&id, nccl_unique_id128, sizeof(id));
        const NcclApi* api = nccl();
        if (!api) { delete ctx; return MLB_ENCCL; }
        ncclResult_t r = api->CommInitRank(&ctx->gpus[0].comm, world, id, rank);
        if (r != ncclSuccess) {
            set_error("ncclCommInitRank failed: %s", api->GetErrorString(r));
            delete ctx;
            return MLB_ENCCL;
        }
    }
    *out = ctx;
    return MLB_OK;
}

int mlb_ctx_destroy(mlb_ctx* ctx)
{
    if (!ctx) return MLB_OK;
    for (Gpu& gpu : ctx->gpus) {
        cudaSetDevice(gpu.device);
        if (gpu.stream) cudaStreamSynchronize(gpu.stream);
        if (gpu.comm && nccl()) nccl()->CommDestroy(gpu.comm);
        if (gpu.ev0) cudaEventDestroy(gpu.ev0);
        if (gpu.ev1) cudaEventDestroy(gpu.ev1);
        for (int i = 0; i < 2 * kCopyThreadsMax; ++i) {
            if (gpu.bounce[i]) cudaFreeHost(gpu.bounce[i]);
            if (gpu.bounce_ev[i]) cudaEventDestroy(gpu.bounce_ev[i]);
        }
        if (gpu.stream) cudaStreamDestroy(gpu.stream);
        if (gpu.pool) cudaMemPoolDestroy(gpu.pool);
    }
    delete ctx;
    return MLB_OK;
}

int mlb_ctx_world(const mlb_ctx* ctx, int* world, int* n_local, int* first_rank)
{
    MLB_REQUIRE(ctx, "mlb_ctx_world: null context");
    if (world) *world = ctx->world;
    if (n_local) *n_local = static_cast<int>(ctx->gpus.size());
    if (first_rank) *first_rank = ctx->gpus[0].rank;
    return MLB_OK;
}

int mlb_ctx_synchronize(mlb_ctx* ctx)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx, "mlb_ctx_synchronize: null context");
    return for_each_gpu(ctx, [&](int, Gpu& gpu) -> int {
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        return MLB_OK;
    });
}

int mlb_ctx_sum_int64(mlb_ctx* ctx, int64_t local, int64_t* total)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx && total, "mlb_ctx_sum_int64: null argument");
    if (!ctx->rank_mode || ctx->world == 1) {
        *total = local;
        return MLB_OK;
    }
    Gpu& gpu = ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    MLB_NCCL_API(api);
    int64_t* dev = nullptr;
    MLB_CUDA(cudaMallocFromPoolAsync(&dev, sizeof(int64_t) * ctx->world, gpu.pool, gpu.stream));
    std::vector<int64_t> host(static_cast<size_t>(ctx->world), 0);
    int rc = MLB_OK;
    auto body = [&]() -> int {
        MLB_CUDA(cudaMemcpyAsync(dev + gpu.rank, &local, sizeof(int64_t), cudaMemcpyHostToDevice, gpu.stream));
        MLB_NCCL(api, api->AllGather(dev + gpu.rank, dev, 1, ncclInt64, gpu.comm, gpu.stream));
        MLB_CUDA(cudaMemcpyAsync(host.data(), dev, sizeof(int64_t) * ctx->world, cudaMemcpyDeviceToHost, gpu.stream));
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        return MLB_OK;
    };
    rc = body();
    cudaFreeAsync(dev, gpu.stream);
    MLB_TRY(rc);
    int64_t sum = 0;
    for (int64_t v : host) sum += v;
    *total = sum;
    return MLB_OK;
}

int mlb_ctx_timer_start(mlb_ctx* ctx)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx, "mlb_ctx_timer_start: null context");
    return for_each_gpu(ctx, [&](int, Gpu& gpu) -> int {
        MLB_CUDA(cudaEventRecord(gpu.ev0, gpu.stream));
        return MLB_OK;
    });
}

int mlb_ctx_timer_stop(mlb_ctx* ctx, double* elapsed_ms)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx && elapsed_ms, "mlb_ctx_timer_stop: null argument");
    MLB_TRY(for_each_gpu(ctx, [&](int, Gpu& gpu) -> int {
        MLB_CUDA(cudaEventRecord(gpu.ev1, gpu.stream));
        return MLB_OK;
    }));
    double worst = 0;
    MLB_TRY(for_each_gpu(ctx, [&](int, Gpu& gpu) -> int {
        MLB_CUDA(cudaEventSynchronize(gpu.ev1));
        float ms = 0;
        MLB_CUDA(cudaEventElapsedTime(&ms, gpu.ev0, gpu.ev1));
        worst = std::max(worst, static_cast<double>(ms));
        return MLB_OK;
    }));
    *elapsed_ms = worst;
    return MLB_OK;
}

int mlb_shard_range(int64_t n_total, int world, int rank, int64_t* begin, int64_t* end)
{
    MLB_REQUIRE(n_total >= 0 && valid_world(world) && rank >= 0 && rank < world, "mlb_shard_range: bad arguments");
    const Layout lay = Layout::make(n_total);
    const int vpg = kVirtualShards / world;
    if (begin) *begin = lay.point_begin(rank * vpg);
    if (end) *end = lay.point_begin((rank + 1) * vpg);
    return MLB_OK;
}

// ======================================================================= C-ABI: data

static int make_shards(mlb_ctx* ctx, int64_t n_total, int d, mlb_data** out)
{
    auto* data = new mlb_data;
    data->ctx = ctx;
    data->d = d;
    data->lay = Layout::make(n_total);
    const int vpg = ctx->vshards_per_gpu();
    data->shards.resize(ctx->gpus.size());
    for (size_t g = 0; g < ctx->gpus.size(); ++g) {
        const int rank = ctx->gpus[g].rank;
        DataShard& sh = data->shards[g];
        sh.chunk_begin = data->lay.vshard_chunk[rank * vpg];
        sh.chunk_end = data->lay.vshard_chunk[(rank + 1) * vpg];
        sh.begin = data->lay.point_begin(rank * vpg);
        sh.end = data->lay.point_begin((rank + 1) * vpg);
    }
    *out = data;
    return MLB_OK;
}

int mlb_data_free(mlb_data* data)
{
    MLB_ENTER(data ? data->ctx : nullptr);
    if (!data) return MLB_OK;
    for (size_t g = 0; g < data->shards.size(); ++g) {
        cudaSetDevice(data->ctx->gpus[g].device);
        cudaStreamSynchronize(data->ctx->gpus[g].stream);
        if (data->shards[g].owned && data->shards[g].x) cudaFreeAsync(data->shards[g].x, data->ctx->gpus[g].stream);
        if (data->shards[g].shift) cudaFreeAsync(data->shards[g].shift, data->ctx->gpus[g].stream);
        if (data->shards[g].nearest) cudaFreeAsync(data->shards[g].nearest, data->ctx->gpus[g].stream);
        if (data->shards[g].seed_centroid) cudaFreeAsync(data->shards[g].seed_centroid, data->ctx->gpus[g].stream);
    }
    delete data;
    return MLB_OK;
}

int mlb_data_upload(mlb_ctx* ctx, const double* x, int64_t n, int64_t n_total, int d, int64_t ld, mlb_data** out)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx && x && out, "mlb_data_upload: null argument");
    MLB_REQUIRE(d >= 1, "mlb_data_upload: at least one dimension required");
    MLB_REQUIRE(ld >= d, "mlb_data_upload: outer stride %lld smaller than d=%d", static_cast<long long>(ld), d);
    MLB_REQUIRE(n_total >= 1 && n_total < (1ll << 32), "mlb_data_upload: n_total out of range");
    mlb_data* data = nullptr;
    MLB_TRY(make_shards(ctx, n_total, d, &data));
    const int64_t host_begin = ctx->rank_mode ? data->shards[0].begin : 0;
    const int64_t expect = ctx->rank_mode ? data->shards[0].n() : n_total;
    if (n != expect) {
        set_error("mlb_data_upload: got %lld points, expected %lld for this context", static_cast<long long>(n), static_cast<long long>(expect));
        mlb_data_free(data);
        return MLB_EINVAL;
    }
    int rc = for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        DataShard& sh = data->shards[g];
        MLB_CUDA(cudaMallocFromPoolAsync(&sh.x, sizeof(double) * std::max<int64_t>(1, sh.n()) * d, gpu.pool, gpu.stream));
        if (sh.n() > 0) {
            const double* src = x + (sh.begin - host_begin) * ld;
            MLB_TRY(staged_h2d(gpu, sh.x, src, static_cast<size_t>(sh.n()), sizeof(double) * d, sizeof(double) * ld));
        }
        return MLB_OK;
    });
    if (rc == MLB_OK) rc = compute_shift(data);
    if (rc != MLB_OK) {
        mlb_data_free(data);
        return rc;
    }
    *out = data;
    return MLB_OK;
}

int mlb_data_wrap_device(mlb_ctx* ctx, const double* x_device, int64_t n, int d, mlb_data** out)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx && x_device && out, "mlb_data_wrap_device: null argument");
    MLB_REQUIRE(ctx->world == 1, "mlb_data_wrap_device: 1-GPU contexts only");
    MLB_REQUIRE(d >= 1 && n >= 1 && n < (1ll << 32), "mlb_data_wrap_device: bad shape");
    mlb_data* data = nullptr;
    MLB_TRY(make_shards(ctx, n, d, &data));
    data->shards[0].x = const_cast<double*>(x_device);
    data->shards[0].owned = false;
    int rc = compute_shift(data);
    if (rc != MLB_OK) {
        mlb_data_free(data);
        return rc;
    }
    *out = data;
    return MLB_OK;
}

int mlb_data_generate_gmm(mlb_ctx* ctx, int64_t n_total, int d, int k_true, uint64_t seed, double spread,
                          double* true_means, mlb_data** out)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx && out, "mlb_data_generate_gmm: null argument");
    MLB_REQUIRE(d >= 1 && d <= kMaxGenDim && k_true >= 1 && n_total >= 1 && n_total < (1ll << 32), "mlb_data_generate_gmm: bad shape");
    // Mixture parameters: a pure function of (seed, d, k_true), drawn on the host.
    std::mt19937_64 rng(seed * 0x9E3779B97F4A7C15ull + 12345u);
    auto unif = [&]() { return (static_cast<double>(rng() >> 11) + 0.5) * (1.0 / 9007199254740992.0); };
    auto normal = [&]() {
        const double u1 = unif(), u2 = unif();
        return std::sqrt(-2.0 * std::log(u1)) * std::cos(6.283185307179586 * u2);
    };
    std::vector<double> means(static_cast<size_t>(k_true) * d), chol(static_cast<size_t>(k_true) * d * d, 0.0), cum(k_true);
    for (double& m : means) m = spread * (2.0 * unif() - 1.0);
    std::vector<double> a(static_cast<size_t>(d) * d), cov(static_cast<size_t>(d) * d);
    for (int c = 0; c < k_true; ++c) {
        for (double& v : a) v = normal();
        for (int i = 0; i < d; ++i)
            for (int j = 0; j < d; ++j) {
                double s = 0;
                for (int l = 0; l < d; ++l) s += a[i * d + l] * a[j * d + l];
                cov[i * d + j] = s / d + (i == j ? 0.5 : 0.0);
            }
        double* l = chol.data() + static_cast<size_t>(c) * d * d;
        for (int j = 0; j < d; ++j) {
            double s = cov[j * d + j];
            for (int t = 0; t < j; ++t) s -= l[j * d + t] * l[j * d + t];
            l[j * d + j] = std::sqrt(s);
            for (int i = j + 1; i < d; ++i) {
                double v = cov[i * d + j];
                for (int t = 0; t < j; ++t) v -= l[i * d + t] * l[j * d + t];
                l[i * d + j] = v / l[j * d + j];
            }
        }
    }
    {
        // Dirichlet(5)-like weights: normalised sums of 5 unit exponentials (= Gamma(5, 1)).
        double total = 0;
        for (int c = 0; c < k_true; ++c) {
            double g = 0;
            for (int j = 0; j < 5; ++j) g -= std::log(unif());
            cum[c] = g;
            total += g;
        }
        double run = 0;
        for (int c = 0; c < k_true; ++c) {
            run += cum[c] / total;
            cum[c] = run;
        }
        cum[k_true - 1] = 1.0;
    }
    if (true_means) std::memcpy(true_means, means.data(), sizeof(double) * means.size());
    mlb_data* data = nullptr;
    MLB_TRY(make_shards(ctx, n_total, d, &data));
    int rc = for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        DataShard& sh = data->shards[g];
        MLB_CUDA(cudaMallocFromPoolAsync(&sh.x, sizeof(double) * std::max<int64_t>(1, sh.n()) * d, gpu.pool, gpu.stream));
        double *dm = nullptr, *dl = nullptr, *dw = nullptr;
        MLB_CUDA(cudaMallocFromPoolAsync(&dm, sizeof(double) * means.size(), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dl, sizeof(double) * chol.size(), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dw, sizeof(double) * cum.size(), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemcpyAsync(dm, means.data(), sizeof(double) * means.size(), cudaMemcpyHostToDevice, gpu.stream));
        MLB_CUDA(cudaMemcpyAsync(dl, chol.data(), sizeof(double) * chol.size(), cudaMemcpyHostToDevice, gpu.stream));
        MLB_CUDA(cudaMemcpyAsync(dw, cum.data(), sizeof(double) * cum.size(), cudaMemcpyHostToDevice, gpu.stream));
        if (sh.n() > 0) {
            const unsigned blocks = static_cast<unsigned>((sh.n() + 127) / 128);
            generate_gmm_kernel<<<blocks, 128, 0, gpu.stream>>>(sh.x, sh.begin, sh.n(), d, k_true, seed, dm, dl, dw);
            MLB_CUDA(cudaGetLastError());
        }
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        MLB_CUDA(cudaFreeAsync(dm, gpu.stream));
        MLB_CUDA(cudaFreeAsync(dl, gpu.stream));
        MLB_CUDA(cudaFreeAsync(dw, gpu.stream));
        return MLB_OK;
    });
    if (rc == MLB_OK) rc = compute_shift(data);
    if (rc != MLB_OK) {
        mlb_data_free(data);
        return rc;
    }
    *out = data;
    return MLB_OK;
}

int mlb_data_download(mlb_data* data, int64_t begin, int64_t count, double* out)
{
    MLB_ENTER(data ? data->ctx : nullptr);
    MLB_REQUIRE(data && out, "mlb_data_download: null argument");
    MLB_REQUIRE(begin >= 0 && count >= 0 && begin + count <= data->lay.n_total, "mlb_data_download: range out of bounds");
    const int d = data->d;
    int64_t covered = 0;
    MLB_TRY(for_each_gpu(data->ctx, [&](int g, Gpu& gpu) -> int {
        const DataShard& sh = data->shards[g];
        const int64_t lo = std::max(begin, sh.begin), hi = std::min(begin + count, sh.end);
        if (lo < hi) {
            MLB_TRY(staged_d2h(gpu, out + (lo - begin) * d, sh.x + (lo - sh.begin) * d, sizeof(double) * (hi - lo) * d));
            covered += hi - lo;
        }
        return MLB_OK;
    }));
    MLB_REQUIRE(covered == count, "mlb_data_download: range is not held by this context");
    return MLB_OK;
}

int mlb_data_shape(const mlb_data* data, int64_t* n_total, int64_t* n_local, int* d)
{
    MLB_REQUIRE(data, "mlb_data_shape: null data");
    if (n_total) *n_total = data->lay.n_total;
    if (n_local) {
        int64_t n = 0;
        for (const DataShard& sh : data->shards) n += sh.n();
        *n_local = n;
    }
    if (d) *d = data->d;
    return MLB_OK;
}

int mlb_standardise_features(mlb_ctx* ctx, const double* x, int64_t n, int d, int64_t ld, double* out, int64_t ld_out)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx && x && out, "mlb_standardise_features: null argument");
    MLB_REQUIRE(n >= 1 && d >= 1 && d <= 1024 && ld >= d && ld_out >= d, "mlb_standardise_features: bad shape (n=%lld, d=%d)", static_cast<long long>(n), d);
    Gpu& gpu = ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    double *xd = nullptr, *partials = nullptr, *mean = nullptr, *sd = nullptr;
    const int threads = std::max(d, 256 / d * d);
    const int64_t rows_per_block = 4096;
    const int nblocks = static_cast<int>((n + rows_per_block - 1) / rows_per_block);
    auto body = [&]() -> int {
        MLB_CUDA(cudaMallocFromPoolAsync(&xd, sizeof(double) * n * d, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&partials, sizeof(double) * nblocks * d, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&mean, sizeof(double) * d, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&sd, sizeof(double) * d, gpu.pool, gpu.stream));
        MLB_TRY(staged_h2d(gpu, xd, x, static_cast<size_t>(n), sizeof(double) * d, sizeof(double) * ld));
        standardise_partial_kernel<<<nblocks, threads, sizeof(double) * threads, gpu.stream>>>(xd, n, d, rows_per_block, nullptr, partials);
        MLB_CUDA(cudaGetLastError());
        standardise_finish_kernel<<<(d + 127) / 128, 128, 0, gpu.stream>>>(partials, nblocks, d, n, 0, mean);
        MLB_CUDA(cudaGetLastError());
        if (n > 1) {   // utils.py:25-27: the division happens only with more than one row
            standardise_partial_kernel<<<nblocks, threads, sizeof(double) * threads, gpu.stream>>>(xd, n, d, rows_per_block, mean, partials);
            MLB_CUDA(cudaGetLastError());
            standardise_finish_kernel<<<(d + 127) / 128, 128, 0, gpu.stream>>>(partials, nblocks, d, n, 1, sd);
            MLB_CUDA(cudaGetLastError());
        }
        const int64_t total = n * d;
        standardise_apply_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, gpu.stream>>>(xd, total, d, mean, sd, n > 1 ? 1 : 0);
        MLB_CUDA(cudaGetLastError());
        if (ld_out == d) {
            MLB_TRY(staged_d2h(gpu, out, xd, sizeof(double) * total));
        } else {
            MLB_TRY(staged_d2h_2d(gpu, out, sizeof(double) * ld_out, xd, sizeof(double) * d, static_cast<size_t>(n), sizeof(double) * d));
        }
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        return MLB_OK;
    };
    const int rc = body();
    cudaStreamSynchronize(gpu.stream);
    for (double* ptr : {xd, partials, mean, sd})
        if (ptr) cudaFreeAsync(ptr, gpu.stream);
    return rc;
}

}  // extern "C"
