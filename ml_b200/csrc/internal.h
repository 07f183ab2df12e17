// Internal structures shared by the translation units of libmlb200.so.  Not part of the C-ABI.
#pragma once

#include <cuda_runtime.h>
#include <nccl.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/mlb200.h"

namespace mlb {

void set_error(const char* fmt, ...);

#define MLB_CUDA(expr)                                                                          \
    do {                                                                                        \
        cudaError_t mlb_e_ = (expr);                                                            \
        if (mlb_e_ != cudaSuccess) {                                                            \
            ::mlb::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(mlb_e_)); \
            return (mlb_e_ == cudaErrorMemoryAllocation) ? MLB_ENOMEM : MLB_ECUDA;              \
        }                                                                                       \
    } while (0)

// NCCL is bound at run time (dlopen), never at link time: a process that also hosts PyTorch must end up
// with ONE libnccl.so.2, and torch ships a newer one than the system's.  nccl() prefers a copy that is
// already loaded, then $MLB200_NCCL_LIB, then the loader's default libnccl.so.2.  Single-GPU contexts never
// touch it.  Returns nullptr (with the error text set) when no usable NCCL is found.
struct NcclApi {
    ncclResult_t (*GetUniqueId)(ncclUniqueId*);
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*);
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
    ncclResult_t (*CommDestroy)(ncclComm_t);
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t);
    ncclResult_t (*GroupStart)();
    ncclResult_t (*GroupEnd)();
    const char* (*GetErrorString)(ncclResult_t);
    ncclResult_t (*GetVersion)(int*);
};
const NcclApi* nccl();

#define MLB_NCCL_API(api)                \
    const ::mlb::NcclApi* api = ::mlb::nccl(); \
    if (!api) return MLB_ENCCL

#define MLB_NCCL(api, expr)                                                                     \
    do {                                                                                        \
        ncclResult_t mlb_n_ = (expr);                                                           \
        if (mlb_n_ != ncclSuccess) {                                                            \
            ::mlb::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, (api)->GetErrorString(mlb_n_)); \
            return MLB_ENCCL;                                                                   \
        }                                                                                       \
    } while (0)

#define MLB_TRY(expr)                   \
    do {                                \
        int mlb_rc_ = (expr);           \
        if (mlb_rc_ != MLB_OK) return mlb_rc_; \
    } while (0)

#define MLB_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            ::mlb::set_error(__VA_ARGS__); \
            return MLB_EINVAL;            \
        }                                 \
    } while (0)

constexpr int kVirtualShards = MLB_VIRTUAL_SHARDS;
constexpr int kCopyThreadsMax = 8;   // host threads that pack / unpack the pinned bounce buffers of one large copy
constexpr int kSmCount = 148;  // B200

// e / d for 0 <= e < 65536 and 1 <= d <= 128 without the ~30-instruction integer division the compiler emits for a
// run-time divisor: (e + 0.5) / d is at least 0.5 / d away from an integer, far more than the float rounding error.
struct FastDiv {
    int d;
    float inv;
    __host__ __device__ explicit FastDiv(int divisor) : d(divisor), inv(1.0f / static_cast<float>(divisor)) {}
    __device__ __forceinline__ int div(int e) const { return __float2int_rz((static_cast<float>(e) + 0.5f) * inv); }
};

// How the N points are cut up.  A pure function of n_total, so that every GPU count sees the same
// chunks and therefore the same summation tree (bitwise G-invariance).
struct Layout {
    int64_t n_total = 0;
    int chunk = 0;                            // points per chunk (multiple of 128)
    int64_t n_chunks = 0;                     // ceil(n_total / chunk)
    int64_t vshard_chunk[kVirtualShards + 1]; // chunk boundaries of the virtual shards

    static Layout make(int64_t n_total);
    int64_t point_begin(int vshard) const { return std::min<int64_t>(vshard_chunk[vshard] * chunk, n_total); }
};

// One local GPU of a context.
struct Gpu {
    int device = 0;
    int rank = 0;  // global rank of this GPU in [0, world)
    cudaStream_t stream = nullptr;
    cudaMemPool_t pool = nullptr;  // the context's own stream-ordered allocation pool on this device
    ncclComm_t comm = nullptr;  // null when world == 1
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // pinned bounce buffers for copies from / to pageable host memory (staged_h2d, staged_d2h): two per copy thread
    void* bounce[2 * kCopyThreadsMax] = {};
    cudaEvent_t bounce_ev[2 * kCopyThreadsMax] = {};
};

}  // namespace mlb

struct mlb_ctx {
    int world = 1;          // total GPUs in the job
    bool rank_mode = false; // one process per GPU
    std::vector<mlb::Gpu> gpus;  // the local ones, consecutive ranks
    // Every C-ABI entry point that enqueues work holds this for its whole duration: the context owns ONE stream and
    // ONE set of pinned bounce buffers per GPU, and EM captures its step into a CUDA graph on that stream, so two
    // host threads driving two models (cppyml releases the GIL inside fit) must not interleave inside a call.
    // Recursive: entry points call each other (mlb_em_step -> mlb_em_run_steps -> mlb_ctx_synchronize).
    std::recursive_mutex mu;
    int vshards_per_gpu() const { return mlb::kVirtualShards / world; }
};

// First statement of every C-ABI entry point that touches a context (ctx_ may be null: the argument checks that follow
// report it): serialises on the context and restores the caller's current CUDA device on return.
#define MLB_ENTER(ctx_)                                        \
    ::mlb::DeviceRestore mlb_dev_;                             \
    std::unique_lock<std::recursive_mutex> mlb_lock_;          \
    if (mlb_ctx* mlb_c_ = (ctx_)) mlb_lock_ = std::unique_lock<std::recursive_mutex>(mlb_c_->mu)

namespace mlb {

// The slice of the data one local GPU holds.
struct DataShard {
    double* x = nullptr;       // point-contiguous, d doubles per point
    bool owned = true;
    int64_t begin = 0, end = 0;           // global point range
    int64_t chunk_begin = 0, chunk_end = 0;  // global chunk range
    double* shift = nullptr;   // d doubles: the global data mean (device copy)
    double* nearest = nullptr;        // K-means++ seeding: squared distance to the nearest chosen centroid, per local point (seeding.cu)
    double* seed_centroid = nullptr;  // d doubles: the newest centroid of the seeding pass
    int64_t n() const { return end - begin; }
    int64_t n_chunks() const { return chunk_end - chunk_begin; }
};

}  // namespace mlb

struct mlb_data {
    mlb_ctx* ctx = nullptr;
    mlb::Layout lay;
    int d = 0;
    std::vector<mlb::DataShard> shards;  // one per local GPU
    std::vector<double> shift;           // host copy of the global data mean
    int64_t launches = 0;                // kernels launched on this object after its creation (seeding passes)
};

namespace mlb {

// Restores the caller's current CUDA device when a C-ABI call returns (the library switches devices internally).
struct DeviceRestore {
    int saved = -1;
    DeviceRestore() { if (cudaGetDevice(&saved) != cudaSuccess) { saved = -1; cudaGetLastError(); } }
    ~DeviceRestore() { if (saved >= 0) cudaSetDevice(saved); }
};

// Runs body(g, gpu) for every local GPU with that GPU's device made current.
template <class F>
int for_each_gpu(mlb_ctx* ctx, F&& body)
{
    for (size_t g = 0; g < ctx->gpus.size(); ++g) {
        MLB_CUDA(cudaSetDevice(ctx->gpus[g].device));
        MLB_TRY(body(static_cast<int>(g), ctx->gpus[g]));
    }
    return MLB_OK;
}

// Level-1 group sums of reduce_and_exchange, one buffer per local GPU, grown on demand.  Owned by the object whose
// statistics are reduced (mlb_em, mlb_km), never shared: EM replays its step from a CUDA graph that has the buffer's
// address baked in, so nobody else may reallocate it.
struct ReduceScratch {
    std::vector<double*> ptr;
    std::vector<size_t> len;
    void release(mlb_ctx* ctx);
};

// Reduces per-chunk partial vectors to the 8 virtual-shard vectors and exchanges them.
//   partials[g]: device, [local chunks of GPU g][s]
//   vsum[g]:     device, [8][s]; on return every GPU holds all 8 shard vectors.
// Fixed summation order => deterministic and independent of the GPU count.
int reduce_and_exchange(mlb_data* data, const std::vector<double*>& partials, const std::vector<double*>& vsum, int s, ReduceScratch& scratch);
// The same for partial vectors per "unit" other than the chunk (the direct EM kernels' super-chunks): bounds[0..8] are the
// global unit boundaries of the 8 virtual shards (a function of N only), partials[g] holds the units of GPU g's shards.
int reduce_and_exchange_units(mlb_data* data, const std::vector<double*>& partials, const std::vector<double*>& vsum, int s, ReduceScratch& scratch,
                              const int64_t* bounds);

// Copies between host memory that is probably pageable (a numpy array, a std::vector, an Eigen matrix) and the device.
// A direct cudaMemcpy of pageable memory runs at ~10 GB/s host -> device and ~4 GB/s device -> host on these boxes (one
// driver thread staging through its own pinned buffer; first-touch page faults on fresh destination pages).  Large
// copies are therefore cut into 4 MB pieces that up to four host threads pack into / unpack from pinned bounce buffers
// (two per thread: the DMA of one piece overlaps the CPU copy of the next), so the DMA engine, not a single memcpy, is
// the bound.  Pinned (page-locked) host memory and small copies go straight to cudaMemcpyAsync.
//
// staged_h2d: the source is `rows` rows of `row_bytes` bytes, `src_stride` bytes apart (src_stride == row_bytes: one
// contiguous block); the destination is dense.  The DMAs are ordered on gpu.stream like any other work.  A pageable
// source has been read completely on return; a PINNED source is read by the DMA engine asynchronously, so the caller
// must synchronise the stream (every C-ABI entry point does, on all of its exit paths) before the buffer may go away.
int staged_h2d(Gpu& gpu, void* dst_device, const void* src, size_t rows, size_t row_bytes, size_t src_stride);
// staged_d2h: synchronous; on return dst holds the data.
int staged_d2h(Gpu& gpu, void* dst, const void* src_device, size_t bytes);
// The same for `rows` rows of `row_bytes` bytes, `src_stride` apart on the device and `dst_stride` apart on the host
// (one column block of a column-major matrix per row): all rows share the copy threads.
int staged_d2h_2d(Gpu& gpu, void* dst, size_t dst_stride, const void* src_device, size_t src_stride, size_t rows, size_t row_bytes);

// Event pairs around the launches of one kernel on one stream (roofline timing for bench.py).
struct KernelTimer {
    bool enabled = false;
    std::vector<cudaEvent_t> events;  // pairs
    size_t used = 0;                  // events recorded
    static constexpr size_t kMaxLaunches = 4096;
    int begin(cudaStream_t stream);
    int end(cudaStream_t stream);
    int total(double* total_ms, int64_t* launches);
    void reset() { used = 0; }
    void destroy();
};

// Host-side fixed tree over the 8 virtual-shard vectors: ((0+1)+(2+3))+((4+5)+(6+7)).
__host__ __device__ inline double tree8(const double* v, int64_t stride)
{
    return ((v[0] + v[stride]) + (v[2 * stride] + v[3 * stride])) + ((v[4 * stride] + v[5 * stride]) + (v[6 * stride] + v[7 * stride]));
}

}  // namespace mlb
