// K-means (Lloyd) on B200 (sm_100a), FP64.  Replaces the loops of ML/KMeans.cpp:
//     assignment_step + assign_label   KMeans.cpp:153-178     km_assign_kernel
//     update_step                      KMeans.cpp:180-192     km_stats_sorted_kernel / km_stats_small_kernel + km_update_kernel
//
// Assignment = filter + exact refinement (DESIGN.md "K-means").
//   filter:  d2_ik = |z_i|^2 + |c'_k|^2 - 2 z_i . c'_k  (z = x - shift, c' = c - shift) for all K centroids as a
//            [points x D] x [D x K] product on the FP64 tensor pipe (mma.sync.m8n8k4.f64), tracking the best and
//            second-best score per point on 32-bit integer keys (the high word of the non-negative double);
//   refine:  the winner's squared distance is recomputed exactly as the reference does ((x - c).squaredNorm(),
//            sequential over the dimensions) so labels, distances and inertia are the reference's; a point whose two
//            best keys cannot be separated (key truncation + FP64 rounding bound) is re-assigned by the exact scan
//            over all K (strict <, lowest k wins).
// Every warp works on its own 16-point sub-tiles (own cp.async double buffer), so one warp's refinement overlaps the
// other warps' filter.  Update statistics (per-cluster count and sum of z) are a separate kernel: for K > 32 a counting
// sort of the chunk by label, then every cluster's points added in index order; for K <= 32 a one-hot tensor-pipe product.
// No floating-point atomics anywhere: bitwise reproducible, and identical for every GPU count.
#include <algorithm>
#include <cmath>

#include "internal.h"

namespace mlb {

constexpr int kKmTile = 64;      // points per CTA tile of the assignment kernel
constexpr int kKmThreads = 128;  // 4 warps, 16 points each
constexpr int kKmGroup = 32;     // centroids per accumulator group (4 n-tiles)

struct KmArgs {
    const double* x;
    long long n_local;
    int d, k, KP;
    const double* shift;
    const double* cfrag;    // [DP/4][KP/16][32][2] image of -2 c'
    const double* cnorm;    // [KP] |c'_k|^2 (+inf for padding)
    const double* craw;     // D x K centroids as the host sees them
    const double* cmax;     // [1] max_k |c'_k|
    unsigned* labels;       // in: previous labels, out: new labels
    double* partials;       // [n_chunks][SV]: K x (D+1) sums and counts, inertia, changed
    int chunk, n_chunks;
    unsigned* counter;
    double* dist_out;       // optional: the squared distance of every point to its centroid (mlb_km_predict, centroid blocks)
    int pstride;            // statistics: doubles between the partial vectors of consecutive chunks
    int k_lo;               // statistics: first cluster of the block this launch accumulates (KP clusters from k_lo)
    int stat_off;           // statistics: extra offset (doubles) of this launch's K x (D+1) block inside a chunk's partial vector (start sets)
    // start sets (km_assign_kernel<..., MULTI = true>, mlb_kms): n_sets centroid sets of k centroids each against the same
    // points in one pass.  cfrag is [n_sets][DP * KP], cnorm [n_sets][KP], craw [n_sets][D x K], cmax [n_sets], labels
    // [n_sets][label_stride]; a chunk's partial vector is [n_sets][KP x (D+1)] followed by (inertia, changed) per set.
    int n_sets;
    unsigned active;        // bit s: set s takes part in this pass (a converged start is frozen)
    long long label_stride;
};

__device__ __forceinline__ void km_dmma(double (&acc)[2], double a, double b)
{
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(acc[0]), "+d"(acc[1]) : "d"(a), "d"(b));
}

__host__ __device__ inline int km_sv(int d, int KP) { return KP * (d + 1) + 8; }

// nw = warps per CTA of the assignment kernel (16 points each)
inline size_t km_smem_bytes(int DP, int KP, int nw = 4)
{
    return sizeof(double) * (static_cast<size_t>(DP) * KP + KP + 2 * static_cast<size_t>(nw) * 16 * (DP + 4) + DP + 32) + sizeof(int) * 3 * nw * 16;
}
// the same with ns centroid sets resident at once and a per-thread (inertia, changed) accumulator per set
inline size_t km_sets_smem_bytes(int DP, int KP, int nw, int ns)
{
    return km_smem_bytes(DP, KP, nw) + sizeof(double) * (static_cast<size_t>(ns - 1) * (static_cast<size_t>(DP) * KP + KP) + static_cast<size_t>(ns) * nw * 32)
           + sizeof(int) * static_cast<size_t>(ns) * nw * 32;
}

// (x - c).squaredNorm() exactly as KMeans.cpp:158 evaluates it (sequential, fused multiply-add).
// The centroid row comes from global memory (L1/L2): its loads are issued 8 at a time ahead of the dependent FMA chain.
__device__ __forceinline__ double exact_distance(const double* x, const double* __restrict__ c, int d)
{
    double s = 0.0;
    for (int l0 = 0; l0 < d; l0 += 8) {
        double cv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) cv[u] = l0 + u < d ? __ldg(c + l0 + u) : 0.0;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (l0 + u < d) {
                const double t = x[l0 + u] - cv[u];
                s = fma(t, t, s);
            }
        }
    }
    return s;
}

__device__ __forceinline__ void km_cp_async8(void* smem, const void* gmem)
{
    const unsigned a = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(a), "l"(gmem));
}
__device__ __forceinline__ void km_cp_async16(void* smem, const void* gmem)
{
    const unsigned a = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(a), "l"(gmem));
}
__device__ __forceinline__ void km_cp_async4(void* smem, const void* gmem)
{
    const unsigned a = static_cast<unsigned>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(a), "l"(gmem));
}
__device__ __forceinline__ void km_cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void km_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// ---------------------------------------------------------------- assignment (KMeans.cpp:153-178)
// Writes the labels and, per chunk, the inertia and the number of changed labels (slots KP*(d+1) and +1 of the partial).
// Every warp works on its own 16-point sub-tiles (its own cp.async double buffer, only __syncwarp inside a chunk), so the
// exact refinement of one warp (global loads of centroid rows) overlaps the tensor-pipe filter of the others.
constexpr int kKmSub = 16;   // points per warp sub-tile

// COMPACT: the chunk's 8 scalars go to partials[chunk * 8] (centroid blocks, prediction) instead of to their slots in the
// chunk's full statistics vector.  A template parameter, not run-time addressing: with the addressing made generic ptxas
// allocates the main loop differently (125 instead of 149 registers at D = 32) and the kernel is 5 % slower on C5.
// NW = warps per CTA.  The centroid image is shared by the whole CTA, so when it is what limits the CTAs per SM (64 KB at
// D = 32, K = 256: two CTAs of four warps, 8 warps per SM) one wide CTA keeps twice the warps resident on the same image
// (NW = 16: 4 per sub-partition), which is what hides the fixed issue latency between a warp's DMMAs and the global loads
// of the refinement (ncu r01j: 36 % of the stall samples were `wait`, 14.5 % long scoreboard, the FP64 pipe 69 % busy).
// MULTI: p.n_sets centroid sets ("starts" of a multi-start fit, KMeans.cpp:29-47) against the same points in one pass: the
// point sub-tile is staged and turned into A fragments once, then filter + refinement run per set on that set's image,
// labels and (inertia, changed) accumulators.  Per set the arithmetic and its order are those of the one-set kernel, so a
// set's labels, inertia and changed count are bit for bit what a fit of that start alone produces.  A template parameter:
// the one-set instantiations are instruction for instruction the measured ones.
template <int DP, bool COMPACT, int NW, bool MULTI = false>
__global__ void __launch_bounds__(NW * 32) km_assign_kernel(const KmArgs p)
{
    constexpr int DQ = DP / 4, XS = DP + 4, kKmTile = NW * 16, kKmThreads = NW * 32;
    static_assert(!(MULTI && COMPACT), "start sets write full statistics vectors");
    extern __shared__ __align__(16) double sm[];
    const int KP = p.KP, d = p.d, SD = d + 1;
    const int NS = MULTI ? p.n_sets : 1;
    double* Bf = sm;                                  // [NS] DP * KP
    double* nrm = Bf + static_cast<size_t>(NS) * DP * KP;  // [NS] KP
    double* Xb = nrm + NS * KP;                       // [4 warps][2 buffers][16][XS], raw coordinates (padding columns zero)
    double* sh = Xb + 2 * kKmTile * XS;               // DP
    double* red = sh + DP;                            // 32
    int* labs_all = reinterpret_cast<int*>(red + 32); // [NW][16]: the filter's verdict (~label: ambiguous under its rounding bound)
    unsigned* oldl_all = reinterpret_cast<unsigned*>(labs_all + kKmTile);  // [NW][2][16]: previous labels
    // MULTI: every thread's running (inertia, changed) of the chunk, per set (the one-set kernel keeps them in registers)
    double* set_inertia = reinterpret_cast<double*>(oldl_all + 2 * kKmTile);   // [NS][threads]
    int* set_changed = reinterpret_cast<int*>(set_inertia + (MULTI ? NS * kKmThreads : 0));   // [NS][threads]
    __shared__ int s_next;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, c = lane & 3;

    if (MULTI) {
        for (int i = tid; i < NS * DP * KP; i += kKmThreads) Bf[i] = p.cfrag[i];
        for (int i = tid; i < NS * KP; i += kKmThreads) nrm[i] = p.cnorm[i];
    } else {
        for (int i = tid; i < DP * KP + KP; i += kKmThreads) sm[i] = i < DP * KP ? p.cfrag[i] : p.cnorm[i - DP * KP];
    }
    for (int i = tid; i < 2 * kKmTile * XS; i += kKmThreads) Xb[i] = 0.0;
    if (tid < DP) sh[tid] = tid < d ? p.shift[tid] : 0.0;
    __syncthreads();
    double shc[DQ];
#pragma unroll
    for (int j = 0; j < DQ; ++j) shc[j] = sh[4 * j + c];
    const double u_bound = 8.0 * (d + 4) * 1.1102230246251565e-16;
    const double cmax1 = *p.cmax;
    double* Xw = Xb + warp * (2 * kKmSub * XS);
    int* labs = labs_all + warp * kKmSub;
    unsigned* oldw = oldl_all + warp * (2 * kKmSub);

    // Asynchronous copy of one sub-tile of points (and their previous labels) into the warp's buffer `buf`; rows past the
    // end are zeroed.
    const FastDiv by_d(d);
    auto stage = [&](long long tile0, int nvalid, int buf) {
        double* X = Xw + buf * (kKmSub * XS);
        const double* xg = p.x + tile0 * d;
        const int nel = nvalid * d;
        if (d == DP) {
            // rows are 16-byte aligned on both sides: two coordinates per copy, row index by a shift
            for (int e2 = lane; e2 < kKmSub * (DP / 2); e2 += 32) {
                const int pt = e2 / (DP / 2), q = e2 - pt * (DP / 2);
                if (2 * e2 < nel) km_cp_async16(X + pt * XS + 2 * q, xg + 2 * e2);
                else *reinterpret_cast<double2*>(X + pt * XS + 2 * q) = make_double2(0.0, 0.0);
            }
        } else {
            for (int e = lane; e < kKmSub * d; e += 32) {
                const int pt = by_d.div(e), dm = e - pt * d;
                if (e < nel) km_cp_async8(X + pt * XS + dm, xg + e);
                else X[pt * XS + dm] = 0.0;
            }
        }
        if (lane < nvalid) km_cp_async4(oldw + buf * kKmSub + lane, p.labels + tile0 + lane);
        km_cp_async_commit();
    };

    for (;;) {
        __syncthreads();
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        __syncthreads();
        const int chunk = s_next;
        if (chunk >= p.n_chunks) break;
        const long long p_begin = static_cast<long long>(chunk) * p.chunk;
        const long long p_end = p_begin + p.chunk < p.n_local ? p_begin + p.chunk : p.n_local;
        const int nsubs = static_cast<int>((p_end - p_begin + kKmSub - 1) / kKmSub);
        double inertia_acc = 0.0;
        int changed_acc = 0;
        if (MULTI)
            for (int s = 0; s < NS; ++s) { set_inertia[s * kKmThreads + tid] = 0.0; set_changed[s * kKmThreads + tid] = 0; }

        // warp w takes the sub-tiles w, w + NW, w + 2 NW, ... of the chunk
        auto sub_begin = [&](int t) { return p_begin + static_cast<long long>(t) * kKmSub; };
        auto sub_valid = [&](int t) { const long long left = p_end - sub_begin(t); return static_cast<int>(left < kKmSub ? left : kKmSub); };
        if (warp < nsubs) stage(sub_begin(warp), sub_valid(warp), 0);
        int it = 0;
        for (int t = warp; t < nsubs; t += NW, ++it) {
            const long long tile0 = sub_begin(t);
            const int nvalid = sub_valid(t);
            if (t + NW < nsubs) {
                stage(sub_begin(t + NW), sub_valid(t + NW), (it + 1) & 1);
                km_cp_async_wait<1>();
            } else {
                km_cp_async_wait<0>();
            }
            __syncwarp();
            const double* X = Xw + (it & 1) * (kKmSub * XS);
            const unsigned* old_labels = oldw + (it & 1) * kKmSub;

            // ---------------- filter: scores of this warp's 16 points against all centroids
            const double* x0 = X + g * XS;
            const double* x1 = x0 + 8 * XS;
            double z0[DQ], z1[DQ];
            double zz0 = 0.0, zz1 = 0.0;
#pragma unroll
            for (int j = 0; j < DQ; ++j) {
                z0[j] = x0[4 * j + c] - shc[j];
                z1[j] = x1[4 * j + c] - shc[j];
                zz0 = fma(z0[j], z0[j], zz0);
                zz1 = fma(z1[j], z1[j], zz1);
            }
            zz0 += __shfl_xor_sync(0xffffffffu, zz0, 1);
            zz0 += __shfl_xor_sync(0xffffffffu, zz0, 2);
            zz1 += __shfl_xor_sync(0xffffffffu, zz1, 1);
            zz1 += __shfl_xor_sync(0xffffffffu, zz1, 2);
            // Best / second-best tracking on 32-bit keys.  The accumulators start at |c'|^2 + |z|^2, so a score IS the squared
            // distance (>= 0 up to rounding) and the high word of the double, read as an integer, orders like the value
            // with 20 mantissa bits: three integer min/max, a compare and a select per score instead of IEEE fmin/fmax
            // chains.  What the truncation (and FP64 rounding) cannot separate is sent to the exact scan below.
            const double zz[2] = {zz0, zz1};
            for (int set = 0; set < NS; ++set) {
            if (MULTI && !((p.active >> set) & 1u)) continue;
            const double* Bfs = MULTI ? Bf + static_cast<size_t>(set) * DP * KP : Bf;
            const double* nrms = MULTI ? nrm + set * KP : nrm;
            const double* craws = MULTI ? p.craw + static_cast<long long>(set) * d * p.k : p.craw;
            const double cmax = MULTI ? p.cmax[set] : cmax1;
            int bestk[2] = {0x7fffffff, 0x7fffffff}, secondk[2] = {0x7fffffff, 0x7fffffff};
            int bk[2] = {0, 0};
            for (int grp = 0; grp < KP / kKmGroup; ++grp) {
                double acc[2][4][2];
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) {
                    const double2 nn = *reinterpret_cast<const double2*>(nrms + grp * kKmGroup + 8 * nt + 2 * c);
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        acc[mt][nt][0] = nn.x + zz[mt];
                        acc[mt][nt][1] = nn.y + zz[mt];
                    }
                }
#pragma unroll
                for (int j = 0; j < DQ; ++j) {
                    const double2* bp = reinterpret_cast<const double2*>(Bfs) + (static_cast<size_t>(j) * (KP / 16) + grp * 2) * 32 + lane;
                    const double2 b01 = bp[0], b23 = bp[32];
                    km_dmma(acc[0][0], z0[j], b01.x); km_dmma(acc[1][0], z1[j], b01.x);
                    km_dmma(acc[0][1], z0[j], b01.y); km_dmma(acc[1][1], z1[j], b01.y);
                    km_dmma(acc[0][2], z0[j], b23.x); km_dmma(acc[1][2], z1[j], b23.x);
                    km_dmma(acc[0][3], z0[j], b23.y); km_dmma(acc[1][3], z1[j], b23.y);
                }
#pragma unroll
                for (int mt = 0; mt < 2; ++mt)
#pragma unroll
                    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int key = max(__double2hiint(acc[mt][nt][e]), 0);
                            secondk[mt] = min(secondk[mt], max(key, bestk[mt]));
                            if (key < bestk[mt]) bk[mt] = grp * kKmGroup + 8 * nt + 2 * c + e;
                            bestk[mt] = min(bestk[mt], key);
                        }
            }
            // ---------------- merge over the 4 lanes of a point; the filter's verdict goes to shared memory
#pragma unroll
            for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
                for (int off = 1; off <= 2; off <<= 1) {
                    const int ob = __shfl_xor_sync(0xffffffffu, bestk[mt], off);
                    const int os = __shfl_xor_sync(0xffffffffu, secondk[mt], off);
                    const int ok = __shfl_xor_sync(0xffffffffu, bk[mt], off);
                    secondk[mt] = min(min(secondk[mt], os), max(bestk[mt], ob));
                    if (ob < bestk[mt] || (ob == bestk[mt] && ok < bk[mt])) { bestk[mt] = ob; bk[mt] = ok; }
                }
                const int pl = mt * 8 + g;
                if (c == 0) {
                    // best score <= best_hi, second score >= second_lo; tau bounds the FP64 rounding of a score
                    const double best_hi = __hiloint2double(bestk[mt] + 1, 0);
                    const double second_lo = secondk[mt] == 0x7fffffff ? INFINITY : __hiloint2double(secondk[mt], 0);
                    const double root = sqrt(zz[mt]) + cmax;
                    const double tau = u_bound * root * root;
                    labs[pl] = second_lo > best_hi + tau ? bk[mt] : ~bk[mt];
                }
            }
            __syncwarp();
            // ---------------- exact refinement: two lanes per point.  The reference's sum runs over the dimensions in order
            // (KMeans.cpp:158); lane 2i takes the first half of the dimensions, hands its partial sum to lane 2i + 1, which
            // continues the same fused-multiply-add chain over the second half: the same value, with the centroid row's
            // global loads of both halves in flight together.
            {
                const int pl = lane >> 1, half = lane & 1;
                const bool valid = pl < nvalid;
                const double* xr = X + pl * XS;
                const int hd = (d + 1) / 2;
                const int l_lo = half ? hd : 0, l_hi = half ? d : hd;
                int label = valid ? labs[pl] : 0;
                const bool ambiguous = label < 0;
                if (ambiguous) label = ~label;
                constexpr int HD = DP / 2;
                double tv[HD];
                const double* cr = craws + static_cast<long long>(label) * d;
#pragma unroll
                for (int u = 0; u < HD; ++u) tv[u] = l_lo + u < l_hi ? __ldg(cr + l_lo + u) : 0.0;
#pragma unroll
                for (int u = 0; u < HD; ++u) tv[u] = l_lo + u < l_hi ? xr[l_lo + u] - tv[u] : 0.0;
                double part = 0.0;
                if (!half) {
#pragma unroll
                    for (int u = 0; u < HD; ++u)
                        if (u < l_hi - l_lo) part = fma(tv[u], tv[u], part);
                }
                const double first = __shfl_sync(0xffffffffu, part, lane & ~1);
                if (half) {
                    part = first;
#pragma unroll
                    for (int u = 0; u < HD; ++u)
                        if (u < l_hi - l_lo) part = fma(tv[u], tv[u], part);
                }
                double d2 = __shfl_sync(0xffffffffu, part, lane | 1);
                if (valid && ambiguous && !half) {
                    // ambiguous under the filter's rounding bound: the reference's scan (KMeans.cpp:153-165)
                    d2 = INFINITY;
                    label = 0;
                    for (int kk = 0; kk < p.k; ++kk) {
                        const double sq = exact_distance(xr, craws + static_cast<long long>(kk) * d, d);
                        if (sq < d2) { d2 = sq; label = kk; }
                    }
                }
                if (!half && valid) {
                    if (MULTI) {
                        unsigned* lab_s = p.labels + static_cast<long long>(set) * p.label_stride + tile0 + pl;
                        set_inertia[set * kKmThreads + tid] += d2;
                        if (*lab_s != static_cast<unsigned>(label)) ++set_changed[set * kKmThreads + tid];
                        *lab_s = static_cast<unsigned>(label);
                    } else {
                        inertia_acc += d2;
                        if (old_labels[pl] != static_cast<unsigned>(label)) ++changed_acc;
                        p.labels[tile0 + pl] = static_cast<unsigned>(label);
                        if (COMPACT && p.dist_out) p.dist_out[tile0 + pl] = d2;
                    }
                }
            }
            __syncwarp();   // the buffer and the verdicts are rewritten two sub-tiles later / by the next sub-tile / by the next set
            }   // set
        }

        // ---------------- the chunk's inertia and changed-label count: fixed order inside the warp and across the warps
        double* out = COMPACT ? p.partials + static_cast<long long>(chunk) * 8 - KP * SD
                      : MULTI ? p.partials + static_cast<long long>(chunk) * p.pstride + (NS - 1) * KP * SD   // scalars after the NS statistics blocks
                              : p.partials + static_cast<long long>(chunk) * km_sv(d, KP);
        for (int set = 0; set < NS; ++set) {
            if (MULTI) {
                inertia_acc = set_inertia[set * kKmThreads + tid];
                changed_acc = set_changed[set * kKmThreads + tid];
                __syncthreads();   // red[] of the previous set has been read
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                inertia_acc += __shfl_xor_sync(0xffffffffu, inertia_acc, off);
                changed_acc += __shfl_xor_sync(0xffffffffu, changed_acc, off);
            }
            if (lane == 0) { red[warp] = inertia_acc; red[16 + warp] = static_cast<double>(changed_acc); }
            __syncthreads();
            if (tid == 0) {
                // fixed pairwise tree over the NW warps
                double a[NW], b[NW];
#pragma unroll
                for (int w = 0; w < NW; ++w) { a[w] = red[w]; b[w] = red[16 + w]; }
#pragma unroll
                for (int span = 1; span < NW; span <<= 1)
#pragma unroll
                    for (int w = 0; w + span < NW; w += 2 * span) { a[w] += a[w + span]; b[w] += b[w + span]; }
                out[KP * SD + 2 * set] = a[0];
                out[KP * SD + 2 * set + 1] = b[0];
            }
        }
        if (tid >= 2 * NS && tid < 8) out[KP * SD + tid] = 0.0;
    }
}

// ---------------------------------------------------------------- assignment for D > 64: the reference's scan
// The filter above keeps a point's coordinates in registers (DQ = D / 4 per lane and sub-tile), which stops paying beyond
// D = 64.  Wider points take KMeans.cpp:153-165 as written: every point against every centroid, (x - c).squaredNorm() as
// the sequential fused multiply-add chain, strict <, lowest index wins.  One thread per point; the point tile and a block
// of 32 centroids sit in shared memory (rows of the tile padded to an odd stride, centroid reads are broadcasts).  Same
// outputs as km_assign_kernel: labels, per chunk the inertia and the number of changed labels, optionally the distances.
constexpr int kKmExactTile = 128;
constexpr int kKmExactBlock = 32;

inline size_t km_exact_smem_bytes(int d)
{
    return sizeof(double) * (static_cast<size_t>(kKmExactTile) * (d | 1) + static_cast<size_t>(kKmExactBlock) * d + 2 * kKmExactTile);
}
// The block-capacity bound of the exact path: a centroid block of KB is at most what a KB x (D + 1) block of sums and a
// 128-point tile leave of one CTA's shared memory.  It fixes KB at D > 64 (288 at D = 65, 128 at D = 100), and with it
// the number of statistics launches per step.
inline size_t km_exact_block_bytes(int d, int KB)
{
    return sizeof(double) * (static_cast<size_t>(KB) * (d + 1) + static_cast<size_t>(128) * d + d) + sizeof(int) * 128;
}

template <bool COMPACT>
__global__ void __launch_bounds__(kKmExactTile) km_assign_exact_kernel(const KmArgs p)
{
    extern __shared__ __align__(16) double sm[];
    const int d = p.d, XS = d | 1, KP = p.KP, SD = d + 1;
    double* X = sm;                                            // [128][XS]
    double* C = X + static_cast<size_t>(kKmExactTile) * XS;    // [32][d]
    double* red = C + static_cast<size_t>(kKmExactBlock) * d;  // [2][128]
    __shared__ int s_next;
    const int tid = threadIdx.x;
    const FastDiv by_d(d);

    for (;;) {
        __syncthreads();
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        __syncthreads();
        const int chunk = s_next;
        if (chunk >= p.n_chunks) break;
        const long long p_begin = static_cast<long long>(chunk) * p.chunk;
        const long long p_end = p_begin + p.chunk < p.n_local ? p_begin + p.chunk : p.n_local;
        double inertia_acc = 0.0, changed_acc = 0.0;
        for (long long tile0 = p_begin; tile0 < p_end; tile0 += kKmExactTile) {
            const int nvalid = static_cast<int>(p_end - tile0 < kKmExactTile ? p_end - tile0 : kKmExactTile);
            __syncthreads();   // the previous tile has been consumed
            const double* xg = p.x + tile0 * d;
            for (int e = tid; e < nvalid * d; e += kKmExactTile) {
                const int pt = by_d.div(e);
                X[pt * XS + (e - pt * d)] = __ldg(xg + e);
            }
            const double* row = X + tid * XS;
            double best = INFINITY;
            unsigned label = 0;
            for (int c0 = 0; c0 < p.k; c0 += kKmExactBlock) {
                const int cb = min(kKmExactBlock, p.k - c0);
                __syncthreads();   // the previous centroid block has been consumed (first pass: the tile is complete)
                for (int e = tid; e < cb * d; e += kKmExactTile) C[e] = __ldg(p.craw + static_cast<long long>(c0) * d + e);
                __syncthreads();
                if (tid < nvalid) {
                    for (int kk = 0; kk < cb; ++kk) {
                        const double* cr = C + kk * d;
                        double s = 0.0;
#pragma unroll 4
                        for (int l = 0; l < d; ++l) {
                            const double t = row[l] - cr[l];
                            s = fma(t, t, s);
                        }
                        if (s < best) { best = s; label = static_cast<unsigned>(c0 + kk); }
                    }
                }
            }
            if (tid < nvalid) {
                inertia_acc += best;
                if (p.labels[tile0 + tid] != label) changed_acc += 1.0;
                p.labels[tile0 + tid] = label;
                if (COMPACT && p.dist_out) p.dist_out[tile0 + tid] = best;
            }
        }
        // the chunk's inertia and changed-label count: a fixed tree over the 128 threads
        __syncthreads();
        red[tid] = inertia_acc;
        red[kKmExactTile + tid] = changed_acc;
        __syncthreads();
        for (int s = kKmExactTile / 2; s > 0; s >>= 1) {
            if (tid < s) {
                red[tid] += red[tid + s];
                red[kKmExactTile + tid] += red[kKmExactTile + tid + s];
            }
            __syncthreads();
        }
        double* out = COMPACT ? p.partials + static_cast<long long>(chunk) * 8 - KP * SD : p.partials + static_cast<long long>(chunk) * km_sv(d, KP);
        if (tid == 0) {
            out[KP * SD] = red[0];
            out[KP * SD + 1] = red[kKmExactTile];
        }
        if (tid >= 2 && tid < 8) out[KP * SD + tid] = 0.0;
    }
}

// ---------------------------------------------------------------- distances to every centroid (mlb_km_transform)
// out[i + k ld] = (x_i - c_k).squaredNorm() as exact_distance and km_assign_exact_kernel evaluate it (the sequential
// fused multiply-add chain over the dimensions from 0.0, raw coordinates), or its square root, for every point of the
// tile and every centroid.  The shape of km_assign_exact_kernel: one thread per point, a 128-point tile (odd row stride)
// and a block of centroids in shared memory; the block is stored dimension-major, so the kKmTrGroup centroids a thread
// advances together are read as broadcast double2 loads.  A warp's stores along a column are 256 contiguous bytes.  Its
// own argument struct: a field added to KmArgs would move the register allocation of the fit's kernels.
constexpr int kKmTrBlock = 32;   // centroids per shared-memory block
constexpr int kKmTrGroup = 8;    // independent distance chains per thread

struct KmTransformArgs {
    const double* x;      // n x D, point-major
    long long n;
    int d, k;
    const double* craw;   // D x K
    double* out;          // column-major n x K with leading dimension ld
    long long ld;
    int squared;          // 0: Euclidean distances, else squared
};

inline size_t km_transform_smem_bytes(int d)
{
    return sizeof(double) * (static_cast<size_t>(kKmExactTile) * (d | 1) + static_cast<size_t>(kKmTrBlock) * d);
}

__global__ void __launch_bounds__(kKmExactTile) km_transform_kernel(const KmTransformArgs p)
{
    extern __shared__ __align__(16) double sm[];
    const int d = p.d, XS = d | 1, tid = threadIdx.x;
    double* X = sm;                                            // [128][XS]
    double* C = X + static_cast<size_t>(kKmExactTile) * XS;    // [d][32]: C[l * 32 + kk] = coordinate l of centroid c0 + kk
    const long long tile0 = static_cast<long long>(blockIdx.x) * kKmExactTile;
    const int nvalid = static_cast<int>(p.n - tile0 < kKmExactTile ? p.n - tile0 : kKmExactTile);
    const FastDiv by_d(d);
    const double* xg = p.x + tile0 * d;
    for (int e = tid; e < nvalid * d; e += kKmExactTile) {
        const int pt = by_d.div(e);
        X[pt * XS + (e - pt * d)] = __ldg(xg + e);
    }
    const double* row = X + tid * XS;
    double* out = p.out + tile0 + tid;
    for (int c0 = 0; c0 < p.k; c0 += kKmTrBlock) {
        const int cb = min(kKmTrBlock, p.k - c0);
        __syncthreads();   // the previous block has been consumed (first pass: the tile is complete)
        for (int e = tid; e < kKmTrBlock * d; e += kKmExactTile) {
            const int kk = by_d.div(e), l = e - kk * d;
            C[l * kKmTrBlock + kk] = kk < cb ? __ldg(p.craw + static_cast<long long>(c0) * d + e) : 0.0;
        }
        __syncthreads();
        if (tid >= nvalid) continue;
        for (int g0 = 0; g0 < cb; g0 += kKmTrGroup) {
            double s[kKmTrGroup];
#pragma unroll
            for (int u = 0; u < kKmTrGroup; ++u) s[u] = 0.0;
            for (int l = 0; l < d; ++l) {
                const double xv = row[l];
                const double2* cp = reinterpret_cast<const double2*>(C + l * kKmTrBlock + g0);
#pragma unroll
                for (int h = 0; h < kKmTrGroup / 2; ++h) {
                    const double2 cv = cp[h];
                    const double t0 = xv - cv.x, t1 = xv - cv.y;
                    s[2 * h] = fma(t0, t0, s[2 * h]);
                    s[2 * h + 1] = fma(t1, t1, s[2 * h + 1]);
                }
            }
#pragma unroll
            for (int u = 0; u < kKmTrGroup; ++u)
                if (g0 + u < cb) out[static_cast<long long>(c0 + g0 + u) * p.ld] = p.squared ? s[u] : sqrt(s[u]);
        }
    }
}

// ---------------------------------------------------------------- update statistics (KMeans.cpp:180-192)
// Per chunk and cluster: the count and the sum of z = x - shift over the chunk's points carrying that label, added in
// index order: no floating-point atomics, bitwise reproducible.  A separate kernel (it re-reads the points and the fresh
// labels, 8D + 4 bytes per point) so that the assignment kernel keeps its shared memory for the centroids and runs several
// CTAs per SM.  A CTA takes a whole chunk (<= 4096 points) at a time:
//   1. stable counting sort of the chunk's point indices by label: every warp ranks its own contiguous 1/8 of the chunk
//      with __match_any_sync (32 points per step) into a per-warp count table, a thread per cluster turns the 8 counts into
//      bases, one warp scans the cluster totals, every point's slot is start[label] + base[warp][label] + rank;
//   2. the clusters are dealt to the 8 warps in contiguous runs of about chunk/8 points; a warp walks its clusters'
//      points in index order, lane = coordinate, gathering the rows straight from global memory (a row is D contiguous
//      doubles: full sectors, every row of the chunk is read exactly once) into a register sum that goes out to the
//      chunk's partial vector with one coalesced store.  No shared-memory statistics at all (10 KB per CTA: the SM fills
//      up with warps, which is what the gathers need), no read-modify-write per point.
// It replaced a kernel in which the warp owning a cluster added that cluster's points into shared memory (the same terms
// in the same order): ~43 warp instructions per point, 99 KB per CTA, 1.51 ms against 0.673 ms per 12.5M points at C5
// (ncu r02h, r02q).
// BLOCKED: the launch accumulates the KP clusters from p.k_lo on (centroid blocks, start sets) into their slots of the
// chunk's full statistics vector; a template parameter so that the one-block kernel stays exactly the measured one.
constexpr int kSsThreads = 256;
constexpr int kSsMaxChunk = 4096;

constexpr int kSsRows = 8;         // rows per gather group (two groups in flight per warp)

inline size_t km_stats_sorted_smem_bytes(int DP, int KP, int chunk)
{
    const size_t dps = static_cast<size_t>(DP < 32 ? 32 : DP);
    return sizeof(double) * (8 * 2 * kSsRows * dps) + sizeof(unsigned short) * (8 * static_cast<size_t>(KP) + 3 * static_cast<size_t>(chunk))
           + sizeof(int) * (static_cast<size_t>(KP) + 1 + 8);
}

template <int DP, bool BLOCKED>
__global__ void __launch_bounds__(kSsThreads) km_stats_sorted_kernel(const KmArgs p)
{
    constexpr int NJ = (DP + 31) / 32;   // coordinates per lane
    extern __shared__ __align__(16) unsigned char smraw[];
    const int KP = p.KP, d = p.d, SD = d + 1, T = p.chunk;
    constexpr int DPS = DP < 32 ? 32 : DP;                                          // doubles per staged row
    double* stage = reinterpret_cast<double*>(smraw) + (threadIdx.x >> 5) * (2 * kSsRows * DPS);   // [8 warps][2][kSsRows][DPS] gathered rows
    int* start = reinterpret_cast<int*>(reinterpret_cast<double*>(smraw) + 8 * 2 * kSsRows * DPS);   // [KP + 1] first slot of every cluster in `sorted`
    unsigned short* cnt = reinterpret_cast<unsigned short*>(start + KP + 1 + 8);   // [8][KP] per-warp counts, then exclusive bases
    unsigned short* labs = cnt + 8 * KP;                                            // [T] label of every point (0xffff: not in this block)
    unsigned short* rank = labs + T;                                                // [T] rank among the warp's points of the same label
    unsigned short* sorted = rank + T;                                              // [T] point indices ordered by (label, index)
    __shared__ int s_next;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per_warp = T / 8;   // T is a multiple of 128
    double shv[NJ];
#pragma unroll
    for (int j = 0; j < NJ; ++j) shv[j] = lane + 32 * j < d ? p.shift[lane + 32 * j] : 0.0;

    for (;;) {
        __syncthreads();   // the previous chunk's tables have been read
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        for (int i = tid; i < 4 * KP; i += kSsThreads) reinterpret_cast<unsigned*>(cnt)[i] = 0u;
        __syncthreads();
        const int chunk = s_next;
        if (chunk >= p.n_chunks) break;
        const long long p_begin = static_cast<long long>(chunk) * p.chunk;
        const int nvalid = static_cast<int>(p_begin + p.chunk < p.n_local ? p.chunk : p.n_local - p_begin);

        // ---- 1a. every warp ranks its own points, 32 at a time in index order
        unsigned short* cw = cnt + warp * KP;
        const int w_end = (warp + 1) * per_warp;   // per_warp is a multiple of 16, not always of 32
        for (int i0 = warp * per_warp; i0 < w_end; i0 += 32) {
            const int i = i0 + lane;
            int lab = -1;
            if (i < w_end && i < nvalid) {
                lab = static_cast<int>(p.labels[p_begin + i]) - (BLOCKED ? p.k_lo : 0);
                if (lab < 0 || lab >= KP) lab = -1;
            }
            const unsigned same = __match_any_sync(0xffffffffu, lab >= 0 ? lab : -1 - lane);
            const int before = __popc(same & ((1u << lane) - 1u));
            const int base = lab >= 0 ? cw[lab] : 0;
            __syncwarp();
            if (lab >= 0 && before == 0) cw[lab] = static_cast<unsigned short>(base + __popc(same));
            __syncwarp();
            if (i < w_end) {
                labs[i] = lab >= 0 ? static_cast<unsigned short>(lab) : 0xffffu;
                rank[i] = static_cast<unsigned short>(base + before);
            }
        }
        __syncthreads();
        // ---- 1b. per cluster: the warps' counts become exclusive bases, the total goes to start[]
        for (int kk = tid; kk < KP; kk += kSsThreads) {
            int run = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                const int c = cnt[w * KP + kk];
                cnt[w * KP + kk] = static_cast<unsigned short>(run);
                run += c;
            }
            start[kk] = run;
        }
        __syncthreads();
        // ---- 1c. exclusive scan of the totals (warp 0; KP is a multiple of 32)
        if (warp == 0) {
            const int per = KP / 32;
            int local = 0;
            for (int j = 0; j < per; ++j) local += start[lane * per + j];
            int incl = local;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, off);
                if (lane >= off) incl += v;
            }
            int run = incl - local;
            for (int j = 0; j < per; ++j) {
                const int c = start[lane * per + j];
                start[lane * per + j] = run;
                run += c;
            }
            if (lane == 31) start[KP] = run;
        }
        __syncthreads();
        // ---- 1d. placement
        for (int i = tid; i < T; i += kSsThreads) {
            const unsigned lab = labs[i];
            if (lab != 0xffffu) sorted[start[lab] + cnt[(i / per_warp) * KP + lab] + rank[i]] = static_cast<unsigned short>(i);
        }
        __syncthreads();
        // ---- 2. clusters in contiguous runs of about total / 8 points per warp: first cluster whose start is >= the share
        const int total = start[KP];
        auto first_cluster = [&](int w) {
            if (w >= 8) return KP;
            const int target = static_cast<int>((static_cast<long long>(total) * w) / 8);
            int lo = 0, hi = KP;   // first kk in [0, KP] with start[kk] >= target, but never beyond a cluster with points
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (start[mid] >= target) hi = mid; else lo = mid + 1;
            }
            return w == 0 ? 0 : lo;
        };
        const int c_lo = first_cluster(warp), c_hi = first_cluster(warp + 1);
        double* out = BLOCKED ? p.partials + static_cast<long long>(chunk) * p.pstride + static_cast<long long>(p.k_lo) * SD + p.stat_off
                              : p.partials + static_cast<long long>(chunk) * km_sv(d, KP);
        const double* xg = p.x + p_begin * d;
        // The warp walks the sorted points of its clusters 32 at a time: every lane fetches one entry's row offset and
        // label and whether it is the LAST row of its cluster; the rows are gathered 8 at a time with cp.async into the warp's
        // two staging buffers (16 rows in flight per warp: the pass is bound by memory-level parallelism, 3.25 GB of rows at
        // C5; plain loads were sunk next to their uses by ptxas, one row in flight) and added in order; after a cluster's
        // last row the sum goes out with a predicated store and the accumulator restarts.
        constexpr int NB = kSsRows;
        double acc[NJ];
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[j] = 0.0;
        const int s_w = start[c_lo], e_w = start[c_hi];
        for (int jb = s_w; jb < e_w; jb += 32) {
            const int pos = jb + lane;
            const bool ok = pos < e_w;
            const int pt = ok ? sorted[pos] : 0;
            const int lab = ok ? labs[pt] : -1;
            int next_lab = __shfl_down_sync(0xffffffffu, lab, 1);
            if (lane == 31) next_lab = pos + 1 < e_w ? labs[sorted[pos + 1]] : -1;
            const unsigned last_mask = __ballot_sync(0xffffffffu, ok && lab != next_lab);
            const int off = pt * d;                    // < 4096 * 128
            const int row_out = lab * SD;              // where this entry's cluster goes in the partial vector
            const int n = e_w - jb < 32 ? e_w - jb : 32;
            // rows of group h / NB -> the warp's staging buffer (h / NB) & 1, asynchronously: every lane copies the
            // coordinates it will add itself, so a lane only ever waits for its own copies
            auto gather = [&](int h) {
                double* dst = stage + ((h / NB) & 1) * (NB * DPS);
#pragma unroll
                for (int u = 0; u < NB; ++u) {
                    const int o = __shfl_sync(0xffffffffu, off, h + u);
                    if (h + u < n) {
#pragma unroll
                        for (int j = 0; j < NJ; ++j)
                            if (lane + 32 * j < d) km_cp_async8(dst + u * DPS + lane + 32 * j, xg + o + lane + 32 * j);
                    }
                }
                km_cp_async_commit();
            };
            gather(0);
#pragma unroll 1
            for (int h = 0; h < n; h += NB) {
                if (h + NB < n) {
                    gather(h + NB);
                    km_cp_async_wait<1>();
                } else {
                    km_cp_async_wait<0>();
                }
                __syncwarp();   // also keeps the compiler from reading the buffer above the wait
                const double* src = stage + ((h / NB) & 1) * (NB * DPS);
#pragma unroll
                for (int u = 0; u < NB; ++u) {
                    const int ro = __shfl_sync(0xffffffffu, row_out, h + u);
                    const bool flush = (last_mask >> (h + u)) & 1u;
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const double v = (h + u < n && lane + 32 * j < d) ? src[u * DPS + lane + 32 * j] : shv[j];   // shv: adds zero
                        acc[j] += v - shv[j];
                        if (flush && lane + 32 * j < d) out[ro + lane + 32 * j] = acc[j];
                        acc[j] = flush ? 0.0 : acc[j];
                    }
                }
            }
        }
        // counts, and zeros for the clusters without points in this chunk: a lane per cluster
        for (int kk = c_lo + lane; kk < c_hi; kk += 32) {
            const int count = start[kk + 1] - start[kk];
            double* row = out + static_cast<long long>(kk) * SD;
            row[d] = static_cast<double>(count);
            if (count == 0)
                for (int dim = 0; dim < d; ++dim) row[dim] = 0.0;
        }
    }
}

// ---------------------------------------------------------------- update statistics, K <= 32
// With few clusters, splitting the work by cluster leaves most warps idle (K = 3: one warp does everything).  Here the
// statistics are a tensor-pipe product instead: S[k][col] = sum_i onehot(label_i == k) * [z_i, 1][col], a
// [32 x points] x [points x (D+1)] DMMA with the one-hot operand made from the labels in registers.  Every warp runs
// its own 16-point sub-tiles; the order of the additions is the hardware's fixed one, so the result is reproducible;
// the four warps' accumulators are combined in a fixed order at the end of a chunk.  2 * 32 * (D + 1) flops per point.
template <int DP>
__global__ void __launch_bounds__(kKmThreads) km_stats_small_kernel(const KmArgs p)
{
    constexpr int NTD = (DP + 1 + 7) / 8, ZS = 8 * NTD + 4, XR = (kKmSub * DP + 31) / 32;
    extern __shared__ __align__(16) double sm[];
    const int d = p.d, SD = d + 1;
    double* Zw = sm;                                  // [4][16][ZS]: z, then the constant 1 (0 past the end), zero padding
    double* redbuf = Zw + 4 * kKmSub * ZS;            // [32][8 * NTD] chunk-end combination
    double* sh = redbuf + 32 * 8 * NTD;               // DP
    __shared__ int s_next;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, c = lane & 3;

    for (int i = tid; i < 4 * kKmSub * ZS; i += kKmThreads) Zw[i] = 0.0;
    if (tid < DP) sh[tid] = tid < d ? p.shift[tid] : 0.0;
    __syncthreads();
    double* Z = Zw + warp * kKmSub * ZS;
    const FastDiv by_d(d);

    for (;;) {
        __syncthreads();
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        __syncthreads();
        const int chunk = s_next;
        if (chunk >= p.n_chunks) break;
        const long long p_begin = static_cast<long long>(chunk) * p.chunk;
        const long long p_end = p_begin + p.chunk < p.n_local ? p_begin + p.chunk : p.n_local;
        const int nsubs = static_cast<int>((p_end - p_begin + kKmSub - 1) / kKmSub);
        double acc[4][NTD][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < NTD; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

        for (int t = warp; t < nsubs; t += 4) {
            const long long tile0 = p_begin + static_cast<long long>(t) * kKmSub;
            const int nvalid = static_cast<int>(p_end - tile0 < kKmSub ? p_end - tile0 : kKmSub);
            const double* xg = p.x + tile0 * d;
            const int nel = nvalid * d;
            double xr[XR];
#pragma unroll
            for (int r = 0; r < XR; ++r) {
                const int e = lane + 32 * r;
                xr[r] = e < nel ? __ldg(xg + e) : 0.0;
            }
            const int label = lane < nvalid ? static_cast<int>(p.labels[tile0 + lane]) : -1;
            __syncwarp();
#pragma unroll
            for (int r = 0; r < XR; ++r) {
                const int e = lane + 32 * r;
                if (e < kKmSub * d) {
                    const int pt = (d == DP) ? e / DP : by_d.div(e);
                    const int dm = e - pt * d;
                    Z[pt * ZS + dm] = e < nel ? xr[r] - sh[dm] : 0.0;
                }
            }
            if (lane < kKmSub) Z[lane * ZS + d] = lane < nvalid ? 1.0 : 0.0;   // the count column sits right after the coordinates
            __syncwarp();
#pragma unroll
            for (int s = 0; s < kKmSub / 4; ++s) {
                const int lab = __shfl_sync(0xffffffffu, label, 4 * s + c);
                const double* zp = Z + (4 * s + c) * ZS + g;
                double bf[NTD];
#pragma unroll
                for (int j = 0; j < NTD; ++j) bf[j] = zp[8 * j];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const double onehot = lab == 8 * i + g ? 1.0 : 0.0;
#pragma unroll
                    for (int j = 0; j < NTD; ++j) km_dmma(acc[i][j], onehot, bf[j]);
                }
            }
        }
        // ---------------- the four warps' statistics in the fixed order ((w0 + w1) + w2) + w3, then out[k][0..d] = sums, count
        for (int w = 0; w < 4; ++w) {
            __syncthreads();
            if (warp == w) {
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < NTD; ++j) {
                        double2* cell = reinterpret_cast<double2*>(redbuf + (8 * i + g) * (8 * NTD) + 8 * j + 2 * c);
                        double2 v = make_double2(acc[i][j][0], acc[i][j][1]);
                        if (w > 0) {
                            const double2 o = *cell;
                            v.x = o.x + v.x;
                            v.y = o.y + v.y;
                        }
                        *cell = v;
                    }
            }
        }
        __syncthreads();
        double* out = p.partials + static_cast<long long>(chunk) * (p.pstride ? p.pstride : km_sv(d, p.KP)) + p.stat_off;   // pstride: start sets
        for (int i = tid; i < p.KP * SD; i += kKmThreads) {
            const int kk = i / SD, col = i - kk * SD;
            out[i] = redbuf[kk * (8 * NTD) + col];
        }
    }
}

inline size_t km_stats_small_smem_bytes(int DP)
{
    const int NTD = (DP + 1 + 7) / 8;
    return sizeof(double) * (4 * kKmSub * (8 * NTD + 4) + 32 * 8 * NTD + DP);
}

// Builds the filter's image of the centroids: -2 c' in mma B-fragment order and |c'|^2; one thread per (dimension, centroid).
struct KmPrepArgs {
    const double* craw;   // D x K
    const double* shift;
    int d, k, DP, KP;
    double* cfrag;
    double* cnorm;
    double* cmax;         // [1]
};

__global__ void km_prepare_kernel(const KmPrepArgs p)
{
    const int kk = blockIdx.x * blockDim.x + threadIdx.x;
    if (kk >= p.KP) return;
    double nn = 0.0;
    for (int dim = 0; dim < p.DP; ++dim) {
        double cp = 0.0;
        if (kk < p.k && dim < p.d) cp = p.craw[dim + static_cast<long long>(kk) * p.d] - p.shift[dim];
        nn = fma(cp, cp, nn);
        const int j = dim >> 2, c = dim & 3, nt = kk >> 3, g = kk & 7, lane = g * 4 + c;
        p.cfrag[((static_cast<long long>(j) * (p.KP / 16) + nt / 2) * 32 + lane) * 2 + (nt & 1)] = -2.0 * cp;
    }
    p.cnorm[kk] = kk < p.k ? nn : INFINITY;
}

__global__ void km_cmax_kernel(const double* cnorm, int k, double* cmax)
{
    double m = 0.0;
    for (int i = 0; i < k; ++i) m = fmax(m, cnorm[i]);
    *cmax = sqrt(m);
}

// update_step (KMeans.cpp:180-192) from the exchanged statistics: centroid = shift + sum(z)/count, an
// empty cluster goes to the origin; old centroids kept; out[0] = |C - C_old|_F^2 (KMeans.cpp:103).
struct KmUpdateArgs {
    const double* vsum;   // [8][SV]
    const double* shift;
    int d, k, KP, SV;
    double* craw;
    double* cold;
    double* out;          // [4]: shift^2, inertia, changed
};

__global__ void km_update_kernel(const KmUpdateArgs p)
{
    __shared__ double part[256];
    const int tid = threadIdx.x;
    double acc = 0.0;
    for (int e = tid; e < p.d * p.k; e += blockDim.x) {
        const int dim = e % p.d, kk = e / p.d;
        const double cnt = tree8(p.vsum + static_cast<long long>(kk) * (p.d + 1) + p.d, p.SV);
        const double sum = tree8(p.vsum + static_cast<long long>(kk) * (p.d + 1) + dim, p.SV);
        const double old = p.craw[e];
        const double now = cnt > 0.0 ? p.shift[dim] + sum / cnt : 0.0;
        p.cold[e] = old;
        p.craw[e] = now;
        const double t = now - old;
        acc = fma(t, t, acc);
    }
    part[tid] = acc;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (tid < s) part[tid] += part[tid + s];
        __syncthreads();
    }
    if (tid == 0) p.out[0] = part[0];
}

__global__ void km_scalars_kernel(const double* vsum, int SV, int base, double* out)
{
    out[1] = tree8(vsum + base, SV);
    out[2] = tree8(vsum + base + 1, SV);
}

// ---------------------------------------------------------------- centroid blocks (K beyond one CTA's shared memory)
// The centroids are cut into blocks of KB that fit; the assignment kernel runs once per block and leaves every point's
// nearest centroid WITHIN the block (lowest index on ties) and its exactly evaluated squared distance.  Folding the
// blocks in ascending order with a strict < is the reference's scan over all K (KMeans.cpp:153-165): same label, same
// distance.
__global__ void km_combine_kernel(const unsigned* __restrict__ block_labels, const double* __restrict__ block_dist, long long n, unsigned base, int first,
                                  unsigned* __restrict__ best_labels, double* __restrict__ best_dist)
{
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double dist = block_dist[i];
    if (first || dist < best_dist[i]) {
        best_dist[i] = dist;
        best_labels[i] = base + block_labels[i];
    }
}

// After the last block: labels <- winners, and per chunk the inertia and the number of changed labels, added in a fixed
// order (a thread adds its points in index order, then a fixed tree over the 256 threads).  One CTA per chunk.
__global__ void __launch_bounds__(256) km_finish_assign_kernel(const unsigned* __restrict__ best_labels, const double* __restrict__ best_dist, long long n, int chunk,
                                                               unsigned* __restrict__ labels, double* __restrict__ partials, int pstride, int poff)
{
    __shared__ double part[256];
    __shared__ double changed[256];
    const long long p_begin = static_cast<long long>(blockIdx.x) * chunk;
    const long long p_end = p_begin + chunk < n ? p_begin + chunk : n;
    double acc = 0.0, ch = 0.0;
    for (long long i = p_begin + threadIdx.x; i < p_end; i += 256) {
        const unsigned now = best_labels[i];
        acc += best_dist[i];
        if (labels[i] != now) ch += 1.0;
        labels[i] = now;
    }
    part[threadIdx.x] = acc;
    changed[threadIdx.x] = ch;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (static_cast<int>(threadIdx.x) < s) {
            part[threadIdx.x] += part[threadIdx.x + s];
            changed[threadIdx.x] += changed[threadIdx.x + s];
        }
        __syncthreads();
    }
    double* out = partials + static_cast<long long>(blockIdx.x) * pstride + poff;
    if (threadIdx.x == 0) { out[0] = part[0]; out[1] = changed[0]; }
    if (threadIdx.x >= 2 && threadIdx.x < 8) out[threadIdx.x] = 0.0;
}

using KmKernelFn = void (*)(KmArgs);

template <bool COMPACT, int NW>
static KmKernelFn km_kernel_for_nw(int DP)
{
    switch (DP) {
    case 4: return km_assign_kernel<4, COMPACT, NW>;
    case 8: return km_assign_kernel<8, COMPACT, NW>;
    case 16: return km_assign_kernel<16, COMPACT, NW>;
    case 32: return km_assign_kernel<32, COMPACT, NW>;
    case 64: return km_assign_kernel<64, COMPACT, NW>;
    default: return nullptr;
    }
}

template <bool COMPACT>
static KmKernelFn km_kernel_for(int DP, int nw)
{
    return nw == 16 ? km_kernel_for_nw<COMPACT, 16>(DP) : nw == 8 ? km_kernel_for_nw<COMPACT, 8>(DP) : km_kernel_for_nw<COMPACT, 4>(DP);
}

// Warps per CTA of the assignment kernel for a centroid block of kb centroids: the choice that keeps the most warps
// resident per SM (shared memory: one centroid image per CTA; registers: 128 per thread, 16 warps per SM), the narrowest
// CTA on ties.  A function of the shape only, so every GPU of a job makes the same choice.
static int km_warps_per_cta(int DP, int kb)
{
    constexpr size_t kSmem = 227 * 1024;
    int best_nw = 4, best_warps = 0;
    for (int nw : {4, 8, 16}) {
        const size_t bytes = km_smem_bytes(DP, kb, nw) + 1024;
        if (bytes > kSmem) continue;
        const int ctas = static_cast<int>(std::min<size_t>(kSmem / bytes, 16 / nw));
        if (ctas * nw > best_warps) { best_warps = ctas * nw; best_nw = nw; }
    }
    return best_nw;
}

static KmKernelFn km_stats_small_kernel_for(int DP)
{
    switch (DP) {
    case 4: return km_stats_small_kernel<4>;
    case 8: return km_stats_small_kernel<8>;
    case 16: return km_stats_small_kernel<16>;
    case 32: return km_stats_small_kernel<32>;
    default: return nullptr;
    }
}

template <bool BLOCKED>
static KmKernelFn km_stats_sorted_kernel_for(int DP)
{
    switch (DP) {
    case 4: return km_stats_sorted_kernel<4, BLOCKED>;
    case 8: return km_stats_sorted_kernel<8, BLOCKED>;
    case 16: return km_stats_sorted_kernel<16, BLOCKED>;
    case 32: return km_stats_sorted_kernel<32, BLOCKED>;
    case 64: return km_stats_sorted_kernel<64, BLOCKED>;
    case 128: return km_stats_sorted_kernel<128, BLOCKED>;
    default: return nullptr;
    }
}

struct KmGpu {
    double* craw = nullptr;
    double* cold = nullptr;
    double* cfrag = nullptr;
    double* cnorm = nullptr;
    double* cmax = nullptr;
    unsigned* labels = nullptr;
    double* partials = nullptr;
    double* vsum = nullptr;
    double* out = nullptr;
    unsigned* counter = nullptr;
    int grid = 0, grid_stats = 0;
    KernelTimer timer;
    // centroid blocks (nblocks > 1): per-point winners so far and the current block's results; 8 scalars per chunk
    unsigned* best_lab = nullptr;
    double* best_dist = nullptr;
    unsigned* lab_tmp = nullptr;
    double* dist_tmp = nullptr;
    double* scratch = nullptr;
};

}  // namespace mlb

using namespace mlb;

struct mlb_km {
    mlb_ctx* ctx = nullptr;
    mlb_data* data = nullptr;
    int d = 0, k = 0, DP = 0, KP = 0, SV = 0;
    int KB = 0, nblocks = 1;     // centroid blocks: KP = nblocks * KB; one block (KB == KP) whenever K fits shared memory
    std::vector<KmGpu> gpus;
    KmKernelFn fn = nullptr, fn_compact = nullptr, fn_stats = nullptr;   // fn_compact: the assignment kernel with compact per-chunk scalars
    bool stats_small = false;    // fn_stats is km_stats_small_kernel (one-hot), else km_stats_sorted_kernel (counting sort)
    bool exact = false;          // D > 64: the reference's scan (km_assign_exact_kernel) instead of the DMMA filter
    int nw = 4;                  // warps per CTA of the assignment kernel
    size_t smem = 0, smem_stats = 0;
    bool have_centroids = false, have_stats = false;
    int64_t launches = 0;
    ReduceScratch reduce_scratch;
};

namespace mlb {

static int km_prepare(mlb_km* km)
{
    if (km->exact) return MLB_OK;   // no filter image: the scan reads the centroids as they are
    return for_each_gpu(km->ctx, [&](int g, Gpu& gpu) -> int {
        KmGpu& kg = km->gpus[g];
        for (int b = 0; b < km->nblocks; ++b) {
            const int k_b = std::min(km->KB, km->k - b * km->KB);
            KmPrepArgs a{kg.craw + static_cast<size_t>(b) * km->KB * km->d, km->data->shards[g].shift, km->d, k_b, km->DP, km->KB,
                         kg.cfrag + static_cast<size_t>(b) * km->DP * km->KB, kg.cnorm + static_cast<size_t>(b) * km->KB, kg.cmax + b};
            km_prepare_kernel<<<(km->KB + 127) / 128, 128, 0, gpu.stream>>>(a);
            MLB_CUDA(cudaGetLastError());
            km_cmax_kernel<<<1, 1, 0, gpu.stream>>>(a.cnorm, k_b, a.cmax);
            MLB_CUDA(cudaGetLastError());
            km->launches += 2;
        }
        return MLB_OK;
    });
}

// The assignment of n points at x (device memory of local GPU g): labels (in: the previous labels, out: the new ones),
// per chunk the inertia and the number of changed labels at partials[chunk * pstride + poff], optionally every point's
// squared distance.  One launch when the centroids are one block; otherwise one launch per block into per-point
// temporaries (tmp_*: n entries each, owned by the caller), folded in ascending block order.
static int launch_assign(mlb_km* km, int g, const double* x, long long n, int chunk, int n_chunks, unsigned* labels, double* dist_out, double* partials,
                         int pstride, int poff, unsigned* tmp_best_lab, double* tmp_best_dist, unsigned* tmp_lab, double* tmp_dist, double* tmp_scratch)
{
    Gpu& gpu = km->ctx->gpus[g];
    KmGpu& kg = km->gpus[g];
    KmArgs a{};
    a.x = x; a.n_local = n; a.d = km->d; a.KP = km->KB;
    a.shift = km->data->shards[g].shift;
    a.chunk = chunk; a.n_chunks = n_chunks;
    a.counter = kg.counter;
    if (km->nblocks == 1 || km->exact) {
        a.k = km->k;
        a.KP = km->KP;   // == KB when the centroids are one block; the exact kernel scans all K whatever the statistics blocks
        a.cfrag = kg.cfrag; a.cnorm = kg.cnorm; a.craw = kg.craw; a.cmax = kg.cmax;
        a.labels = labels; a.partials = partials; a.dist_out = dist_out;
        // full statistics vectors (the fit: pstride == SV, scalars at KP * (d + 1)) or 8 scalars per chunk (prediction)
        const KmKernelFn fn = pstride == 8 ? km->fn_compact : km->fn;
        MLB_CUDA(cudaMemsetAsync(kg.counter, 0, sizeof(unsigned), gpu.stream));
        fn<<<std::min(kg.grid, n_chunks), km->exact ? kKmExactTile : km->nw * 32, km->smem, gpu.stream>>>(a);
        MLB_CUDA(cudaGetLastError());
        ++km->launches;
        return MLB_OK;
    }
    double* best_dist = dist_out ? dist_out : tmp_best_dist;
    for (int b = 0; b < km->nblocks; ++b) {
        a.k = std::min(km->KB, km->k - b * km->KB);
        a.cfrag = kg.cfrag + static_cast<size_t>(b) * km->DP * km->KB;
        a.cnorm = kg.cnorm + static_cast<size_t>(b) * km->KB;
        a.craw = kg.craw + static_cast<size_t>(b) * km->KB * km->d;
        a.cmax = kg.cmax + b;
        a.labels = tmp_lab; a.partials = tmp_scratch; a.dist_out = tmp_dist;
        MLB_CUDA(cudaMemsetAsync(kg.counter, 0, sizeof(unsigned), gpu.stream));
        km->fn_compact<<<std::min(kg.grid, n_chunks), km->nw * 32, km->smem, gpu.stream>>>(a);
        MLB_CUDA(cudaGetLastError());
        km_combine_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, gpu.stream>>>(tmp_lab, tmp_dist, n, static_cast<unsigned>(b) * km->KB, b == 0, tmp_best_lab, best_dist);
        MLB_CUDA(cudaGetLastError());
        km->launches += 2;
    }
    km_finish_assign_kernel<<<n_chunks, 256, 0, gpu.stream>>>(tmp_best_lab, best_dist, n, chunk, labels, partials, pstride, poff);
    MLB_CUDA(cudaGetLastError());
    ++km->launches;
    return MLB_OK;
}

constexpr int64_t kKmStage = 1 << 20;   // host points per staged batch
constexpr int kKmRun = 2048;            // chunk of the assignment kernel on host points: one inertia partial per run

// The assignment of m host points with the current centroids (mlb_km_predict, mlb_km_score), on the first local GPU, in
// staged batches of kKmStage points through the COMPACT kernels.  labels_out, sqdist_out and run_inertia (appended: the
// inertia of every kKmRun-point run, in point order) may each be null.  The fit's labels, statistics and centroids are
// not touched.
static int km_assign_host(mlb_km* km, const double* x, int64_t m, int64_t ld_x, unsigned* labels_out, double* sqdist_out, std::vector<double>* run_inertia)
{
    Gpu& gpu = km->ctx->gpus[0];
    const int d = km->d;
    MLB_CUDA(cudaSetDevice(gpu.device));
    const int64_t cap = std::min<int64_t>(m, kKmStage);
    const int64_t cap_chunks = (cap + kKmRun - 1) / kKmRun;
    double *xd = nullptr, *dist = nullptr, *partials = nullptr, *tmp_dist = nullptr, *tmp_scratch = nullptr;
    unsigned *labels = nullptr, *tmp_best_lab = nullptr, *tmp_lab = nullptr;
    std::vector<double> host_partials;
    auto body = [&]() -> int {
        MLB_CUDA(cudaMallocFromPoolAsync(&xd, sizeof(double) * cap * d, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dist, sizeof(double) * cap, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&labels, sizeof(unsigned) * cap, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&partials, sizeof(double) * 8 * cap_chunks, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(labels, 0, sizeof(unsigned) * cap, gpu.stream));   // the kernel reads the "previous" labels
        if (km->nblocks > 1) {
            MLB_CUDA(cudaMallocFromPoolAsync(&tmp_best_lab, sizeof(unsigned) * cap, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&tmp_lab, sizeof(unsigned) * cap, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&tmp_dist, sizeof(double) * cap, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&tmp_scratch, sizeof(double) * 8 * cap_chunks, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMemsetAsync(tmp_lab, 0, sizeof(unsigned) * cap, gpu.stream));
        }
        for (int64_t off = 0; off < m; off += kKmStage) {
            const int64_t n = std::min<int64_t>(kKmStage, m - off);
            const int n_chunks = static_cast<int>((n + kKmRun - 1) / kKmRun);
            MLB_TRY(staged_h2d(gpu, xd, x + off * ld_x, static_cast<size_t>(n), sizeof(double) * d, sizeof(double) * ld_x));
            MLB_TRY(launch_assign(km, 0, xd, n, kKmRun, n_chunks, labels, dist, partials, 8, 0, tmp_best_lab, nullptr, tmp_lab, tmp_dist, tmp_scratch));
            if (labels_out) MLB_TRY(staged_d2h(gpu, labels_out + off, labels, sizeof(unsigned) * n));
            if (sqdist_out) MLB_TRY(staged_d2h(gpu, sqdist_out + off, dist, sizeof(double) * n));
            if (run_inertia) {
                // the stages are whole runs, so the run partials do not depend on the staging
                host_partials.resize(static_cast<size_t>(8) * n_chunks);
                MLB_CUDA(cudaMemcpyAsync(host_partials.data(), partials, sizeof(double) * host_partials.size(), cudaMemcpyDeviceToHost, gpu.stream));
                MLB_CUDA(cudaStreamSynchronize(gpu.stream));
                for (int c = 0; c < n_chunks; ++c) run_inertia->push_back(host_partials[static_cast<size_t>(8) * c]);
            }
            MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        }
        return MLB_OK;
    };
    const int rc = body();
    for (void* ptr : {static_cast<void*>(xd), static_cast<void*>(dist), static_cast<void*>(labels), static_cast<void*>(partials), static_cast<void*>(tmp_best_lab),
                      static_cast<void*>(tmp_lab), static_cast<void*>(tmp_dist), static_cast<void*>(tmp_scratch)})
        if (ptr) cudaFreeAsync(ptr, gpu.stream);
    return rc;
}

// Points per staged batch of mlb_km_transform / mlb_km_transform_range: at most kKmStage, and at most 1 GiB of distances
// in the device buffer (K = 256: 512K points).
static int64_t km_transform_stage(int k)
{
    return std::max<int64_t>(kKmExactTile, std::min<int64_t>(kKmStage, (int64_t{1} << 27) / k / kKmExactTile * kKmExactTile));
}

// Distances of the n points at x (device memory of local GPU g) to every current centroid into out (column-major n x K,
// leading dimension ld).
static int launch_transform(mlb_km* km, int g, const double* x, long long n, int squared, double* out, long long ld)
{
    Gpu& gpu = km->ctx->gpus[g];
    const KmTransformArgs a{x, n, km->d, km->k, km->gpus[g].craw, out, ld, squared};
    const size_t smem = km_transform_smem_bytes(km->d);
    MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(km_transform_kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    km_transform_kernel<<<static_cast<unsigned>((n + kKmExactTile - 1) / kKmExactTile), kKmExactTile, smem, gpu.stream>>>(a);
    MLB_CUDA(cudaGetLastError());
    ++km->launches;
    return MLB_OK;
}

}  // namespace mlb

extern "C" {

int mlb_km_create(mlb_ctx* ctx, mlb_data* data, int k, mlb_km** out)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx && data && out, "mlb_km_create: null argument");
    MLB_REQUIRE(data->ctx == ctx, "mlb_km_create: data belongs to another context");
    MLB_REQUIRE(k >= 1, "mlb_km_create: number of clusters must be positive");
    const int d = data->d;
    int DP = 0;
    for (int cand : {4, 8, 16, 32, 64, 128})
        if (d <= cand) { DP = cand; break; }
    MLB_REQUIRE(DP, "mlb_km_create: D=%d not supported by this build (D <= 128)", d);
    const bool exact = DP > 64;   // wide points: the reference's scan instead of the DMMA filter (km_assign_exact_kernel)
    constexpr size_t kSmemLimit = 227 * 1024;
    int KP = (k + kKmGroup - 1) / kKmGroup * kKmGroup, KB = KP, nblocks = 1;
    // what bounds a centroid block: the filter's centroid image, or on the exact path its block-capacity bound
    auto block_bytes = [&](int kb) { return exact ? km_exact_block_bytes(d, kb) : km_smem_bytes(DP, kb); };
    int forced = 0;   // MLB200_KM_BLOCK: developer override (a multiple of 32) that forces small centroid blocks, for tests
    if (const char* env = std::getenv("MLB200_KM_BLOCK")) forced = std::atoi(env) / kKmGroup * kKmGroup;
    if (block_bytes(KP) > kSmemLimit || (forced >= kKmGroup && forced < KP)) {
        // Centroid blocks: the largest block that leaves room for two CTAs per SM if that is at least 128 centroids,
        // else the largest that fits at all.  The exact path keeps no centroid image: its largest block within the bound.
        auto largest = [&](size_t limit) {
            int kb = 0;
            for (int cand = kKmGroup; cand <= 4096; cand += kKmGroup)
                if (block_bytes(cand) <= (exact ? kSmemLimit : limit)) kb = cand;
            return kb;
        };
        KB = largest(kSmemLimit / 2 - 1024);
        if (KB < 128) KB = largest(kSmemLimit);
        if (forced >= kKmGroup) KB = std::min(KB, forced);
        MLB_REQUIRE(KB >= kKmGroup, "mlb_km_create: D=%d leaves no room for a block of centroids in shared memory", d);
        nblocks = (k + KB - 1) / KB;
        KP = nblocks * KB;
    }
    const int nw = exact ? 4 : km_warps_per_cta(DP, KB);
    const bool stats_small = nblocks == 1 && KP == kKmGroup && DP <= 32;   // K <= 32: one-hot tensor-pipe statistics (its accumulators fit the registers up to D = 32)
    const int chunk = data->lay.chunk;
    MLB_REQUIRE(stats_small || (chunk <= kSsMaxChunk && KB < 0xffff), "mlb_km_create: the statistics kernel takes chunks of at most %d points and blocks of fewer than 65535 centroids (chunk %d, block %d)", kSsMaxChunk, chunk, KB);
    const size_t smem = exact ? km_exact_smem_bytes(d) : km_smem_bytes(DP, KB, nw);
    auto* km = new mlb_km;
    km->ctx = ctx; km->data = data; km->d = d; km->k = k; km->DP = DP; km->KP = KP; km->SV = km_sv(d, KP);
    km->KB = KB; km->nblocks = nblocks;
    km->exact = exact;
    km->nw = nw;
    km->fn = exact ? km_assign_exact_kernel<false> : km_kernel_for<false>(DP, nw);
    km->fn_compact = exact ? km_assign_exact_kernel<true> : km_kernel_for<true>(DP, nw);
    km->stats_small = stats_small;
    km->fn_stats = stats_small ? km_stats_small_kernel_for(DP) : nblocks == 1 ? km_stats_sorted_kernel_for<false>(DP) : km_stats_sorted_kernel_for<true>(DP);
    km->smem = smem;
    km->smem_stats = stats_small ? km_stats_small_smem_bytes(DP) : km_stats_sorted_smem_bytes(DP, KB, chunk);
    km->gpus.resize(ctx->gpus.size());
    int rc = for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        KmGpu& kg = km->gpus[g];
        const DataShard& sh = data->shards[g];
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.craw, sizeof(double) * d * k, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.cold, sizeof(double) * d * k, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.cfrag, sizeof(double) * DP * KP, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.cnorm, sizeof(double) * KP, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.cmax, sizeof(double) * km->nblocks, gpu.pool, gpu.stream));
        if (km->nblocks > 1) {
            const int64_t n = std::max<int64_t>(1, sh.n());
            MLB_CUDA(cudaMallocFromPoolAsync(&kg.best_lab, sizeof(unsigned) * n, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&kg.best_dist, sizeof(double) * n, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&kg.lab_tmp, sizeof(unsigned) * n, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&kg.dist_tmp, sizeof(double) * n, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&kg.scratch, sizeof(double) * 8 * std::max<int64_t>(1, sh.n_chunks()), gpu.pool, gpu.stream));
            MLB_CUDA(cudaMemsetAsync(kg.lab_tmp, 0, sizeof(unsigned) * n, gpu.stream));
        }
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.labels, sizeof(unsigned) * std::max<int64_t>(1, sh.n()), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.partials, sizeof(double) * std::max<int64_t>(1, sh.n_chunks()) * km->SV, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.vsum, sizeof(double) * kVirtualShards * km->SV, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.out, sizeof(double) * 4, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.counter, sizeof(unsigned), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(kg.labels, 0, sizeof(unsigned) * std::max<int64_t>(1, sh.n()), gpu.stream));   // labels_.resize(): zeros
        MLB_CUDA(cudaMemsetAsync(kg.vsum, 0, sizeof(double) * kVirtualShards * km->SV, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(kg.cold, 0, sizeof(double) * d * k, gpu.stream));
        MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(km->fn), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(km->fn_compact), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        int per_sm = 0, sms = 0;
        MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void*>(km->fn), exact ? kKmExactTile : nw * 32, smem));
        MLB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, gpu.device));
        MLB_REQUIRE(per_sm >= 1, "mlb_km_create: K-means kernel does not fit on an SM");
        kg.grid = per_sm * sms;
        MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(km->fn_stats), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(km->smem_stats)));
        MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void*>(km->fn_stats), km->stats_small ? kKmThreads : kSsThreads, km->smem_stats));
        MLB_REQUIRE(per_sm >= 1, "mlb_km_create: K-means statistics kernel does not fit on an SM");
        kg.grid_stats = per_sm * sms;
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        return MLB_OK;
    });
    if (rc != MLB_OK) { mlb_km_destroy(km); return rc; }
    *out = km;
    return MLB_OK;
}

int mlb_km_destroy(mlb_km* km)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    if (!km) return MLB_OK;
    for (size_t g = 0; g < km->gpus.size(); ++g) {
        cudaSetDevice(km->ctx->gpus[g].device);
        cudaStreamSynchronize(km->ctx->gpus[g].stream);
        KmGpu& kg = km->gpus[g];
        kg.timer.destroy();
        for (void* ptr : {static_cast<void*>(kg.craw), static_cast<void*>(kg.cold), static_cast<void*>(kg.cfrag), static_cast<void*>(kg.cnorm),
                          static_cast<void*>(kg.cmax), static_cast<void*>(kg.labels), static_cast<void*>(kg.partials), static_cast<void*>(kg.vsum),
                          static_cast<void*>(kg.out), static_cast<void*>(kg.counter), static_cast<void*>(kg.best_lab), static_cast<void*>(kg.best_dist),
                          static_cast<void*>(kg.lab_tmp), static_cast<void*>(kg.dist_tmp), static_cast<void*>(kg.scratch)})
            if (ptr) cudaFreeAsync(ptr, km->ctx->gpus[g].stream);
    }
    km->reduce_scratch.release(km->ctx);
    delete km;
    return MLB_OK;
}

int mlb_km_set_centroids(mlb_km* km, const double* centroids)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && centroids, "mlb_km_set_centroids: null argument");
    MLB_TRY(for_each_gpu(km->ctx, [&](int g, Gpu& gpu) -> int {
        MLB_CUDA(cudaMemcpyAsync(km->gpus[g].craw, centroids, sizeof(double) * km->d * km->k, cudaMemcpyHostToDevice, gpu.stream));
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        return MLB_OK;
    }));
    MLB_TRY(km_prepare(km));
    km->have_centroids = true;
    km->have_stats = false;
    return MLB_OK;
}

int mlb_km_get_centroids(mlb_km* km, double* centroids)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && centroids, "mlb_km_get_centroids: null argument");
    if (!km->have_centroids) { set_error("mlb_km_get_centroids: centroids not set"); return MLB_ESTATE; }
    Gpu& gpu = km->ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    MLB_CUDA(cudaMemcpyAsync(centroids, km->gpus[0].craw, sizeof(double) * km->d * km->k, cudaMemcpyDeviceToHost, gpu.stream));
    MLB_CUDA(cudaStreamSynchronize(gpu.stream));
    return MLB_OK;
}

int mlb_km_assign(mlb_km* km, double* inertia, int64_t* n_changed)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km, "mlb_km_assign: null argument");
    if (!km->have_centroids) { set_error("mlb_km_assign: centroids not set"); return MLB_ESTATE; }
    mlb_ctx* ctx = km->ctx;
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        KmGpu& kg = km->gpus[g];
        const DataShard& sh = km->data->shards[g];
        const int chunk = km->data->lay.chunk, n_chunks = static_cast<int>(sh.n_chunks());
        if (n_chunks > 0) {
            MLB_TRY(kg.timer.begin(gpu.stream));
            MLB_TRY(launch_assign(km, g, sh.x, sh.n(), chunk, n_chunks, kg.labels, nullptr, kg.partials, km->SV, km->KP * (km->d + 1),
                                  kg.best_lab, kg.best_dist, kg.lab_tmp, kg.dist_tmp, kg.scratch));
            // statistics of the fresh labels, one launch per centroid block
            KmArgs a{};
            a.x = sh.x; a.n_local = sh.n(); a.d = km->d; a.k = km->k; a.KP = km->KB;
            a.shift = sh.shift; a.labels = kg.labels; a.partials = kg.partials; a.pstride = km->SV;
            a.chunk = chunk; a.n_chunks = n_chunks; a.counter = kg.counter;
            for (int b = 0; b < km->nblocks; ++b) {
                a.k_lo = b * km->KB;
                MLB_CUDA(cudaMemsetAsync(kg.counter, 0, sizeof(unsigned), gpu.stream));
                km->fn_stats<<<std::min(kg.grid_stats, n_chunks), km->stats_small ? kKmThreads : kSsThreads, km->smem_stats, gpu.stream>>>(a);
                MLB_CUDA(cudaGetLastError());
                ++km->launches;
            }
            MLB_TRY(kg.timer.end(gpu.stream));
        }
        return MLB_OK;
    }));
    std::vector<double*> partials, vsum;
    for (KmGpu& kg : km->gpus) { partials.push_back(kg.partials); vsum.push_back(kg.vsum); }
    MLB_TRY(reduce_and_exchange(km->data, partials, vsum, km->SV, km->reduce_scratch));
    km->launches += static_cast<int64_t>(ctx->gpus.size());
    double host[4] = {0, 0, 0, 0};
    {
        Gpu& gpu = ctx->gpus[0];
        MLB_CUDA(cudaSetDevice(gpu.device));
        km_scalars_kernel<<<1, 1, 0, gpu.stream>>>(km->gpus[0].vsum, km->SV, km->KP * (km->d + 1), km->gpus[0].out);
        MLB_CUDA(cudaGetLastError());
        ++km->launches;
        MLB_CUDA(cudaMemcpyAsync(host, km->gpus[0].out, sizeof(double) * 4, cudaMemcpyDeviceToHost, gpu.stream));
    }
    MLB_TRY(mlb_ctx_synchronize(ctx));
    if (inertia) *inertia = host[1];
    if (n_changed) *n_changed = static_cast<int64_t>(host[2]);
    km->have_stats = true;
    return MLB_OK;
}

int mlb_km_update(mlb_km* km, double* centroid_shift_sq)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km, "mlb_km_update: null argument");
    if (!km->have_stats) { set_error("mlb_km_update: no assignment to update from"); return MLB_ESTATE; }
    MLB_TRY(for_each_gpu(km->ctx, [&](int g, Gpu& gpu) -> int {
        KmGpu& kg = km->gpus[g];
        KmUpdateArgs a{kg.vsum, km->data->shards[g].shift, km->d, km->k, km->KP, km->SV, kg.craw, kg.cold, kg.out};
        km_update_kernel<<<1, 256, 0, gpu.stream>>>(a);
        MLB_CUDA(cudaGetLastError());
        ++km->launches;
        return MLB_OK;
    }));
    MLB_TRY(km_prepare(km));
    double host = 0.0;
    Gpu& gpu = km->ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    MLB_CUDA(cudaMemcpyAsync(&host, km->gpus[0].out, sizeof(double), cudaMemcpyDeviceToHost, gpu.stream));
    MLB_TRY(mlb_ctx_synchronize(km->ctx));
    if (centroid_shift_sq) *centroid_shift_sq = host;
    km->have_stats = false;
    return MLB_OK;
}

int mlb_km_predict(mlb_km* km, const double* x, int64_t m, int64_t ld_x, unsigned int* labels_out, double* sqdist_out)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && x && labels_out, "mlb_km_predict: null argument");
    MLB_REQUIRE(m >= 0 && ld_x >= km->d, "mlb_km_predict: bad shape (m=%lld, ld_x=%lld, D=%d)", static_cast<long long>(m), static_cast<long long>(ld_x), km->d);
    if (!km->have_centroids) { set_error("mlb_km_predict: centroids not set"); return MLB_ESTATE; }
    if (m == 0) return MLB_OK;
    return km_assign_host(km, x, m, ld_x, labels_out, sqdist_out, nullptr);
}

int mlb_km_score(mlb_km* km, const double* x, int64_t m, int64_t ld_x, double* sqdist_out, double* inertia_out)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && x && inertia_out, "mlb_km_score: null argument");
    MLB_REQUIRE(m >= 0 && ld_x >= km->d, "mlb_km_score: bad shape (m=%lld, ld_x=%lld, D=%d)", static_cast<long long>(m), static_cast<long long>(ld_x), km->d);
    if (!km->have_centroids) { set_error("mlb_km_score: centroids not set"); return MLB_ESTATE; }
    *inertia_out = 0.0;
    if (m == 0) return MLB_OK;
    std::vector<double> runs;
    MLB_TRY(km_assign_host(km, x, m, ld_x, nullptr, sqdist_out, &runs));
    double total = 0.0;
    for (double v : runs) total += v;   // in point order
    *inertia_out = total;
    return MLB_OK;
}

int mlb_km_score_fitted(mlb_km* km, double* inertia_out)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && inertia_out, "mlb_km_score_fitted: null argument");
    if (!km->have_centroids) { set_error("mlb_km_score_fitted: centroids not set"); return MLB_ESTATE; }
    mlb_ctx* ctx = km->ctx;
    const size_t ng = ctx->gpus.size();
    // The assignment of mlb_km_assign (same kernels, same chunks) into scratch labels and 8 scalars per chunk; the chunk
    // inertias take the step's reduction (8 virtual shards, one exchange, fixed tree), so the sum is bitwise the inertia
    // the next mlb_km_assign reports, for any GPU count.  The fit's labels, statistics, centroids and timer are not touched;
    // the temporaries of the centroid-block path are rewritten by every assignment before they are read.
    std::vector<unsigned*> labels(ng, nullptr);
    std::vector<double*> part(ng, nullptr), vsum(ng, nullptr);
    ReduceScratch scratch;
    double host_vsum[kVirtualShards * 8] = {};
    auto body = [&]() -> int {
        MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
            KmGpu& kg = km->gpus[g];
            const DataShard& sh = km->data->shards[g];
            const int n_chunks = static_cast<int>(sh.n_chunks());
            MLB_CUDA(cudaMallocFromPoolAsync(&labels[g], sizeof(unsigned) * std::max<int64_t>(1, sh.n()), gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&part[g], sizeof(double) * 8 * std::max(1, n_chunks), gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&vsum[g], sizeof(double) * kVirtualShards * 8, gpu.pool, gpu.stream));
            if (n_chunks > 0)
                MLB_TRY(launch_assign(km, g, sh.x, sh.n(), km->data->lay.chunk, n_chunks, labels[g], nullptr, part[g], 8, 0, kg.best_lab, kg.best_dist, kg.lab_tmp,
                                      kg.dist_tmp, kg.scratch));
            return MLB_OK;
        }));
        MLB_TRY(reduce_and_exchange(km->data, part, vsum, 8, scratch));
        km->launches += static_cast<int64_t>(ng);
        Gpu& gpu0 = ctx->gpus[0];
        MLB_CUDA(cudaSetDevice(gpu0.device));
        MLB_CUDA(cudaMemcpyAsync(host_vsum, vsum[0], sizeof(host_vsum), cudaMemcpyDeviceToHost, gpu0.stream));
        return MLB_OK;
    };
    int rc = body();
    const int rc_sync = mlb_ctx_synchronize(ctx);
    if (rc == MLB_OK) rc = rc_sync;
    for (size_t g = 0; g < ng; ++g) {
        cudaSetDevice(ctx->gpus[g].device);
        for (void* ptr : {static_cast<void*>(labels[g]), static_cast<void*>(part[g]), static_cast<void*>(vsum[g])})
            if (ptr) cudaFreeAsync(ptr, ctx->gpus[g].stream);
    }
    scratch.release(ctx);
    if (rc == MLB_OK) *inertia_out = tree8(host_vsum, 8);
    return rc;
}

int mlb_km_transform(mlb_km* km, const double* x, int64_t m, int64_t ld_x, int squared, double* dist_out, int64_t ld_out)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && x && dist_out, "mlb_km_transform: null argument");
    MLB_REQUIRE(m >= 0 && ld_x >= km->d && ld_out >= m, "mlb_km_transform: bad shape (m=%lld, ld_x=%lld, ld_out=%lld, D=%d)", static_cast<long long>(m),
                static_cast<long long>(ld_x), static_cast<long long>(ld_out), km->d);
    if (!km->have_centroids) { set_error("mlb_km_transform: centroids not set"); return MLB_ESTATE; }
    if (m == 0) return MLB_OK;
    Gpu& gpu = km->ctx->gpus[0];
    const int d = km->d;
    MLB_CUDA(cudaSetDevice(gpu.device));
    const int64_t stage = km_transform_stage(km->k), cap = std::min(m, stage);
    double *xd = nullptr, *out = nullptr;
    auto body = [&]() -> int {
        MLB_CUDA(cudaMallocFromPoolAsync(&xd, sizeof(double) * cap * d, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&out, sizeof(double) * cap * km->k, gpu.pool, gpu.stream));
        for (int64_t off = 0; off < m; off += stage) {
            const int64_t n = std::min(stage, m - off);
            MLB_TRY(staged_h2d(gpu, xd, x + off * ld_x, static_cast<size_t>(n), sizeof(double) * d, sizeof(double) * ld_x));
            MLB_TRY(launch_transform(km, 0, xd, n, squared, out, cap));
            MLB_TRY(staged_d2h_2d(gpu, dist_out + off, sizeof(double) * ld_out, out, sizeof(double) * cap, static_cast<size_t>(km->k), sizeof(double) * n));
            MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        }
        return MLB_OK;
    };
    const int rc = body();
    for (double* ptr : {xd, out})
        if (ptr) cudaFreeAsync(ptr, gpu.stream);
    return rc;
}

int mlb_km_transform_range(mlb_km* km, int64_t begin, int64_t count, int squared, double* dist_out, int64_t ld_out)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && dist_out, "mlb_km_transform_range: null argument");
    MLB_REQUIRE(begin >= 0 && count >= 0 && begin + count <= km->data->lay.n_total, "mlb_km_transform_range: range out of bounds");
    MLB_REQUIRE(ld_out >= count, "mlb_km_transform_range: leading dimension smaller than the row count");
    if (!km->have_centroids) { set_error("mlb_km_transform_range: centroids not set"); return MLB_ESTATE; }
    if (count == 0) return MLB_OK;
    mlb_ctx* ctx = km->ctx;
    const size_t ng = ctx->gpus.size();
    std::vector<int64_t> cap(ng, 0);
    int64_t covered = 0;
    const int64_t stage = km_transform_stage(km->k);
    for (size_t g = 0; g < ng; ++g) {
        const DataShard& sh = km->data->shards[g];
        const int64_t held = std::max<int64_t>(0, std::min(begin + count, sh.end) - std::max(begin, sh.begin));
        covered += held;
        cap[g] = std::min(held, stage);
    }
    MLB_REQUIRE(covered == count, "mlb_km_transform_range: range is not held by this context");
    std::vector<double*> out(ng, nullptr);
    auto body = [&]() -> int {
        MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
            if (cap[g] > 0) MLB_CUDA(cudaMallocFromPoolAsync(&out[g], sizeof(double) * cap[g] * km->k, gpu.pool, gpu.stream));
            return MLB_OK;
        }));
        // stage by stage: up to `stage` points per GPU at a time through its device buffer
        for (int64_t off = 0;; off += stage) {
            bool any = false;
            MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
                const DataShard& sh = km->data->shards[g];
                const int64_t lo = std::max(begin, sh.begin) + off, hi = std::min(begin + count, sh.end);
                const int64_t n = std::min(stage, hi - lo);
                if (n <= 0) return MLB_OK;
                any = true;
                MLB_TRY(launch_transform(km, g, sh.x + (lo - sh.begin) * km->d, n, squared, out[g], cap[g]));
                return staged_d2h_2d(gpu, dist_out + (lo - begin), sizeof(double) * ld_out, out[g], sizeof(double) * cap[g], static_cast<size_t>(km->k), sizeof(double) * n);
            }));
            if (!any) break;
        }
        return MLB_OK;
    };
    int rc = body();
    const int rc_sync = mlb_ctx_synchronize(ctx);
    if (rc == MLB_OK) rc = rc_sync;
    for (size_t g = 0; g < ng; ++g)
        if (out[g]) {
            cudaSetDevice(ctx->gpus[g].device);
            cudaFreeAsync(out[g], ctx->gpus[g].stream);
        }
    return rc;
}

int mlb_km_get_labels(mlb_km* km, unsigned int* labels)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && labels, "mlb_km_get_labels: null argument");
    const int64_t host_begin = km->ctx->rank_mode ? km->data->shards[0].begin : 0;
    MLB_TRY(for_each_gpu(km->ctx, [&](int g, Gpu& gpu) -> int {
        const DataShard& sh = km->data->shards[g];
        if (sh.n() > 0) MLB_TRY(staged_d2h(gpu, labels + (sh.begin - host_begin), km->gpus[g].labels, sizeof(unsigned) * sh.n()));
        return MLB_OK;
    }));
    return mlb_ctx_synchronize(km->ctx);
}

int mlb_km_set_kernel_timing(mlb_km* km, int enabled)
{
    MLB_REQUIRE(km, "mlb_km_set_kernel_timing: null argument");
    for (KmGpu& kg : km->gpus) {
        kg.timer.enabled = enabled != 0;
        kg.timer.reset();
    }
    return MLB_OK;
}

int mlb_km_kernel_time_ms(mlb_km* km, double* total_ms, int64_t* launches)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km, "mlb_km_kernel_time_ms: null argument");
    MLB_CUDA(cudaSetDevice(km->ctx->gpus[0].device));
    return km->gpus[0].timer.total(total_ms, launches);
}

int mlb_km_launch_count(const mlb_km* km, int64_t* launches)
{
    MLB_REQUIRE(km && launches, "mlb_km_launch_count: null argument");
    *launches = km->launches;
    return MLB_OK;
}

int mlb_km_kernel_config(const mlb_km* km, int out[8])
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && out, "mlb_km_kernel_config: null argument");
    out[0] = km->DP;
    out[1] = km->KP;
    out[2] = km->KB;
    out[3] = km->nblocks;
    out[4] = km->nw;
    out[5] = km->exact ? 1 : 0;
    out[6] = km->stats_small ? 0 : 1;
    out[7] = km->data->lay.chunk;
    return MLB_OK;
}

}  // extern "C"

// ======================================================================= start sets (multi-start K-means, KMeans.cpp:29-47)
// The reference runs the number_initialisations_ starts of a fit one after the other, each a full Lloyd loop over the data.
// Here up to kKmsMaxSets starts advance in lockstep: ONE pass of the assignment kernel stages every point sub-tile once and
// scores it against all the sets' centroid images (km_assign_kernel<..., MULTI>), the per-set statistics land side by side in
// a chunk's partial vector ([set][K x (D+1)], then (inertia, changed) per set), so one reduction / exchange, one read-back
// and two host synchronisations per iteration serve all the starts.  A start that has converged is frozen (its bit leaves
// the active mask: no scoring, no statistics, no update), which is what keeps every start's trajectory the one it has alone.

namespace mlb {

constexpr int kKmsMaxSets = 4;   // the 8 scalar slots of a partial vector hold (inertia, changed) for four sets

template <int NW>
static KmKernelFn kms_kernel_for_nw(int DP)
{
    switch (DP) {
    case 4: return km_assign_kernel<4, false, NW, true>;
    case 8: return km_assign_kernel<8, false, NW, true>;
    case 16: return km_assign_kernel<16, false, NW, true>;
    case 32: return km_assign_kernel<32, false, NW, true>;
    case 64: return km_assign_kernel<64, false, NW, true>;
    default: return nullptr;
    }
}

// out[4 s + 1] = inertia of set s, out[4 s + 2] = its changed-label count (the layout mlb_km uses, one group of 4 per set)
__global__ void kms_scalars_kernel(const double* vsum, int SV, int base, int n_sets, double* out)
{
    const int s = threadIdx.x;
    if (s >= n_sets) return;
    out[4 * s + 1] = tree8(vsum + base + 2 * s, SV);
    out[4 * s + 2] = tree8(vsum + base + 2 * s + 1, SV);
}

struct KmsGpu {
    double* craw = nullptr;    // [S][D x K]
    double* cold = nullptr;
    double* cfrag = nullptr;   // [S][DP * KP]
    double* cnorm = nullptr;   // [S][KP]
    double* cmax = nullptr;    // [S]
    unsigned* labels = nullptr;  // [S][n_local]
    double* partials = nullptr;  // [n_chunks][SV]
    double* vsum = nullptr;      // [8][SV]
    double* out = nullptr;       // [4 S]
    unsigned* counter = nullptr;
    int grid = 0, grid_stats = 0;
};

}  // namespace mlb

struct mlb_kms {
    mlb_ctx* ctx = nullptr;
    mlb_data* data = nullptr;
    int d = 0, k = 0, DP = 0, KP = 0, n_sets = 0, SV = 0, nw = 4;
    std::vector<mlb::KmsGpu> gpus;
    mlb::KmKernelFn fn = nullptr, fn_stats = nullptr;
    bool stats_small = false;
    size_t smem = 0, smem_stats = 0;
    unsigned have_centroids = 0, have_stats = 0;   // bit per set
    int64_t launches = 0;
    mlb::ReduceScratch reduce_scratch;
};

namespace mlb {

static int kms_prepare(mlb_kms* km, unsigned sets)
{
    return for_each_gpu(km->ctx, [&](int g, Gpu& gpu) -> int {
        KmsGpu& kg = km->gpus[g];
        for (int s = 0; s < km->n_sets; ++s) {
            if (!((sets >> s) & 1u)) continue;
            KmPrepArgs a{kg.craw + static_cast<size_t>(s) * km->d * km->k, km->data->shards[g].shift, km->d, km->k, km->DP, km->KP,
                         kg.cfrag + static_cast<size_t>(s) * km->DP * km->KP, kg.cnorm + static_cast<size_t>(s) * km->KP, kg.cmax + s};
            km_prepare_kernel<<<(km->KP + 127) / 128, 128, 0, gpu.stream>>>(a);
            MLB_CUDA(cudaGetLastError());
            km_cmax_kernel<<<1, 1, 0, gpu.stream>>>(a.cnorm, km->k, a.cmax);
            MLB_CUDA(cudaGetLastError());
            km->launches += 2;
        }
        return MLB_OK;
    });
}

}  // namespace mlb

extern "C" {

int mlb_kms_supported(const mlb_data* data, int k, int n_sets)
{
    if (!data || k < 1 || n_sets < 1 || n_sets > kKmsMaxSets) return 0;
    int DP = 0;
    for (int cand : {4, 8, 16, 32, 64})
        if (data->d <= cand) { DP = cand; break; }
    if (!DP) return 0;   // wider points take the exact scan, one start at a time
    const int KP = (k + kKmGroup - 1) / kKmGroup * kKmGroup;
    constexpr size_t kSmemLimit = 227 * 1024;
    return km_sets_smem_bytes(DP, KP, 4, n_sets) + 1024 <= kSmemLimit;
}

int mlb_kms_create(mlb_ctx* ctx, mlb_data* data, int k, int n_sets, mlb_kms** out)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx && data && out, "mlb_kms_create: null argument");
    MLB_REQUIRE(data->ctx == ctx, "mlb_kms_create: data belongs to another context");
    MLB_REQUIRE(k >= 1, "mlb_kms_create: number of clusters must be positive");
    MLB_REQUIRE(n_sets >= 1 && n_sets <= kKmsMaxSets, "mlb_kms_create: 1 to %d start sets per object (got %d)", kKmsMaxSets, n_sets);
    MLB_REQUIRE(mlb_kms_supported(data, k, n_sets), "mlb_kms_create: %d sets of K=%d centroids at D=%d do not fit one CTA's shared memory (or D > 64): run the starts one at a time", n_sets, k, data->d);
    const int d = data->d;
    int DP = 0;
    for (int cand : {4, 8, 16, 32, 64})
        if (d <= cand) { DP = cand; break; }
    const int KP = (k + kKmGroup - 1) / kKmGroup * kKmGroup;
    constexpr size_t kSmemLimit = 227 * 1024;
    // Warps per CTA: the one-start kernel's choice for this shape whenever the sets' images leave room for it (a chunk's
    // inertia partial is summed per warp, so with the same number of warps it is bit for bit the one-start value; labels,
    // changed counts and statistics do not depend on it), else the choice that keeps the most warps resident per SM.
    int nw = km_warps_per_cta(DP, KP);
    if (km_sets_smem_bytes(DP, KP, nw, n_sets) + 1024 > kSmemLimit) {
        int best_warps = 0;
        nw = 4;
        for (int cand : {4, 8, 16}) {
            const size_t bytes = km_sets_smem_bytes(DP, KP, cand, n_sets) + 1024;
            if (bytes > kSmemLimit) continue;
            const int ctas = static_cast<int>(std::min<size_t>(kSmemLimit / bytes, 16 / cand));
            if (ctas * cand > best_warps) { best_warps = ctas * cand; nw = cand; }
        }
    }
    const bool stats_small = KP == kKmGroup && DP <= 32;
    const int chunk = data->lay.chunk;
    MLB_REQUIRE(stats_small || (chunk <= kSsMaxChunk && KP < 0xffff), "mlb_kms_create: the statistics kernel takes chunks of at most %d points and blocks of fewer than 65535 centroids (chunk %d, K %d)", kSsMaxChunk, chunk, KP);
    auto* km = new mlb_kms;
    km->ctx = ctx; km->data = data; km->d = d; km->k = k; km->DP = DP; km->KP = KP; km->n_sets = n_sets;
    km->SV = n_sets * KP * (d + 1) + 8;
    km->nw = nw;
    km->fn = nw == 16 ? kms_kernel_for_nw<16>(DP) : nw == 8 ? kms_kernel_for_nw<8>(DP) : kms_kernel_for_nw<4>(DP);
    km->smem = km_sets_smem_bytes(DP, KP, nw, n_sets);
    km->stats_small = stats_small;
    km->fn_stats = stats_small ? km_stats_small_kernel_for(DP) : km_stats_sorted_kernel_for<true>(DP);
    km->smem_stats = stats_small ? km_stats_small_smem_bytes(DP) : km_stats_sorted_smem_bytes(DP, KP, chunk);
    km->gpus.resize(ctx->gpus.size());
    const size_t S = static_cast<size_t>(n_sets);
    int rc = for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        KmsGpu& kg = km->gpus[g];
        const DataShard& sh = data->shards[g];
        const size_t n = static_cast<size_t>(std::max<int64_t>(1, sh.n()));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.craw, sizeof(double) * S * d * k, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.cold, sizeof(double) * S * d * k, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.cfrag, sizeof(double) * S * DP * KP, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.cnorm, sizeof(double) * S * KP, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.cmax, sizeof(double) * S, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.labels, sizeof(unsigned) * S * n, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.partials, sizeof(double) * std::max<int64_t>(1, sh.n_chunks()) * km->SV, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.vsum, sizeof(double) * kVirtualShards * km->SV, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.out, sizeof(double) * 4 * S, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&kg.counter, sizeof(unsigned), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(kg.labels, 0, sizeof(unsigned) * S * n, gpu.stream));   // labels_.resize(): zeros
        MLB_CUDA(cudaMemsetAsync(kg.partials, 0, sizeof(double) * std::max<int64_t>(1, sh.n_chunks()) * km->SV, gpu.stream));   // frozen sets are never written
        MLB_CUDA(cudaMemsetAsync(kg.vsum, 0, sizeof(double) * kVirtualShards * km->SV, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(kg.cold, 0, sizeof(double) * S * d * k, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(kg.cfrag, 0, sizeof(double) * S * DP * KP, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(kg.cnorm, 0, sizeof(double) * S * KP, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(kg.cmax, 0, sizeof(double) * S, gpu.stream));
        MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(km->fn), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(km->smem)));
        int per_sm = 0, sms = 0;
        MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void*>(km->fn), nw * 32, km->smem));
        MLB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, gpu.device));
        MLB_REQUIRE(per_sm >= 1, "mlb_kms_create: K-means kernel does not fit on an SM");
        kg.grid = per_sm * sms;
        MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(km->fn_stats), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(km->smem_stats)));
        MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void*>(km->fn_stats), km->stats_small ? kKmThreads : kSsThreads, km->smem_stats));
        MLB_REQUIRE(per_sm >= 1, "mlb_kms_create: K-means statistics kernel does not fit on an SM");
        kg.grid_stats = per_sm * sms;
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        return MLB_OK;
    });
    if (rc != MLB_OK) { mlb_kms_destroy(km); return rc; }
    *out = km;
    return MLB_OK;
}

int mlb_kms_destroy(mlb_kms* km)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    if (!km) return MLB_OK;
    for (size_t g = 0; g < km->gpus.size(); ++g) {
        cudaSetDevice(km->ctx->gpus[g].device);
        cudaStreamSynchronize(km->ctx->gpus[g].stream);
        KmsGpu& kg = km->gpus[g];
        for (void* ptr : {static_cast<void*>(kg.craw), static_cast<void*>(kg.cold), static_cast<void*>(kg.cfrag), static_cast<void*>(kg.cnorm),
                          static_cast<void*>(kg.cmax), static_cast<void*>(kg.labels), static_cast<void*>(kg.partials), static_cast<void*>(kg.vsum),
                          static_cast<void*>(kg.out), static_cast<void*>(kg.counter)})
            if (ptr) cudaFreeAsync(ptr, km->ctx->gpus[g].stream);
    }
    km->reduce_scratch.release(km->ctx);
    delete km;
    return MLB_OK;
}

int mlb_kms_set_centroids(mlb_kms* km, int set, const double* centroids)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && centroids, "mlb_kms_set_centroids: null argument");
    MLB_REQUIRE(set >= 0 && set < km->n_sets, "mlb_kms_set_centroids: set %d out of range", set);
    MLB_TRY(for_each_gpu(km->ctx, [&](int g, Gpu& gpu) -> int {
        MLB_CUDA(cudaMemcpyAsync(km->gpus[g].craw + static_cast<size_t>(set) * km->d * km->k, centroids, sizeof(double) * km->d * km->k, cudaMemcpyHostToDevice, gpu.stream));
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        return MLB_OK;
    }));
    MLB_TRY(kms_prepare(km, 1u << set));
    km->have_centroids |= 1u << set;
    km->have_stats &= ~(1u << set);
    return MLB_OK;
}

int mlb_kms_get_centroids(mlb_kms* km, int set, double* centroids)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && centroids, "mlb_kms_get_centroids: null argument");
    MLB_REQUIRE(set >= 0 && set < km->n_sets, "mlb_kms_get_centroids: set %d out of range", set);
    if (!((km->have_centroids >> set) & 1u)) { set_error("mlb_kms_get_centroids: centroids not set"); return MLB_ESTATE; }
    Gpu& gpu = km->ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    MLB_CUDA(cudaMemcpyAsync(centroids, km->gpus[0].craw + static_cast<size_t>(set) * km->d * km->k, sizeof(double) * km->d * km->k, cudaMemcpyDeviceToHost, gpu.stream));
    MLB_CUDA(cudaStreamSynchronize(gpu.stream));
    return MLB_OK;
}

int mlb_kms_assign(mlb_kms* km, unsigned int active, double* inertia, int64_t* n_changed)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km, "mlb_kms_assign: null argument");
    MLB_REQUIRE(active != 0 && (active >> km->n_sets) == 0, "mlb_kms_assign: active mask 0x%x names no set or a set beyond %d", active, km->n_sets);
    if ((km->have_centroids & active) != active) { set_error("mlb_kms_assign: centroids not set for an active set"); return MLB_ESTATE; }
    mlb_ctx* ctx = km->ctx;
    const int SD = km->d + 1;
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        KmsGpu& kg = km->gpus[g];
        const DataShard& sh = km->data->shards[g];
        const int chunk = km->data->lay.chunk, n_chunks = static_cast<int>(sh.n_chunks());
        if (n_chunks == 0) return MLB_OK;
        KmArgs a{};
        a.x = sh.x; a.n_local = sh.n(); a.d = km->d; a.k = km->k; a.KP = km->KP;
        a.shift = sh.shift;
        a.cfrag = kg.cfrag; a.cnorm = kg.cnorm; a.craw = kg.craw; a.cmax = kg.cmax;
        a.labels = kg.labels; a.partials = kg.partials; a.pstride = km->SV;
        a.chunk = chunk; a.n_chunks = n_chunks; a.counter = kg.counter;
        a.n_sets = km->n_sets; a.active = active; a.label_stride = std::max<int64_t>(1, sh.n());
        MLB_CUDA(cudaMemsetAsync(kg.counter, 0, sizeof(unsigned), gpu.stream));
        km->fn<<<std::min(kg.grid, n_chunks), km->nw * 32, km->smem, gpu.stream>>>(a);
        MLB_CUDA(cudaGetLastError());
        ++km->launches;
        // statistics of the fresh labels: one launch per active set into that set's block of the partial vectors
        for (int s = 0; s < km->n_sets; ++s) {
            if (!((active >> s) & 1u)) continue;
            KmArgs b{};
            b.x = sh.x; b.n_local = sh.n(); b.d = km->d; b.k = km->k; b.KP = km->KP;
            b.shift = sh.shift; b.labels = kg.labels + static_cast<size_t>(s) * a.label_stride; b.partials = kg.partials; b.pstride = km->SV;
            b.chunk = chunk; b.n_chunks = n_chunks; b.counter = kg.counter;
            b.k_lo = 0; b.stat_off = s * km->KP * SD;
            MLB_CUDA(cudaMemsetAsync(kg.counter, 0, sizeof(unsigned), gpu.stream));
            km->fn_stats<<<std::min(kg.grid_stats, n_chunks), km->stats_small ? kKmThreads : kSsThreads, km->smem_stats, gpu.stream>>>(b);
            MLB_CUDA(cudaGetLastError());
            ++km->launches;
        }
        return MLB_OK;
    }));
    std::vector<double*> partials, vsum;
    for (KmsGpu& kg : km->gpus) { partials.push_back(kg.partials); vsum.push_back(kg.vsum); }
    MLB_TRY(reduce_and_exchange(km->data, partials, vsum, km->SV, km->reduce_scratch));
    km->launches += static_cast<int64_t>(ctx->gpus.size());
    double host[4 * kKmsMaxSets] = {};
    {
        Gpu& gpu = ctx->gpus[0];
        MLB_CUDA(cudaSetDevice(gpu.device));
        kms_scalars_kernel<<<1, 32, 0, gpu.stream>>>(km->gpus[0].vsum, km->SV, km->n_sets * km->KP * SD, km->n_sets, km->gpus[0].out);
        MLB_CUDA(cudaGetLastError());
        ++km->launches;
        MLB_CUDA(cudaMemcpyAsync(host, km->gpus[0].out, sizeof(double) * 4 * km->n_sets, cudaMemcpyDeviceToHost, gpu.stream));
    }
    MLB_TRY(mlb_ctx_synchronize(ctx));
    for (int s = 0; s < km->n_sets; ++s) {
        if (!((active >> s) & 1u)) continue;
        if (inertia) inertia[s] = host[4 * s + 1];
        if (n_changed) n_changed[s] = static_cast<int64_t>(host[4 * s + 2]);
    }
    km->have_stats |= active;
    return MLB_OK;
}

int mlb_kms_update(mlb_kms* km, unsigned int active, double* centroid_shift_sq)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km, "mlb_kms_update: null argument");
    MLB_REQUIRE(active != 0 && (active >> km->n_sets) == 0, "mlb_kms_update: active mask 0x%x names no set or a set beyond %d", active, km->n_sets);
    if ((km->have_stats & active) != active) { set_error("mlb_kms_update: no assignment to update an active set from"); return MLB_ESTATE; }
    const int SD = km->d + 1;
    MLB_TRY(for_each_gpu(km->ctx, [&](int g, Gpu& gpu) -> int {
        KmsGpu& kg = km->gpus[g];
        for (int s = 0; s < km->n_sets; ++s) {
            if (!((active >> s) & 1u)) continue;
            const size_t c_off = static_cast<size_t>(s) * km->d * km->k;
            KmUpdateArgs a{kg.vsum + static_cast<size_t>(s) * km->KP * SD, km->data->shards[g].shift, km->d, km->k, km->KP, km->SV, kg.craw + c_off, kg.cold + c_off, kg.out + 4 * s};
            km_update_kernel<<<1, 256, 0, gpu.stream>>>(a);
            MLB_CUDA(cudaGetLastError());
            ++km->launches;
        }
        return MLB_OK;
    }));
    MLB_TRY(kms_prepare(km, active));
    double host[4 * kKmsMaxSets] = {};
    Gpu& gpu = km->ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    MLB_CUDA(cudaMemcpyAsync(host, km->gpus[0].out, sizeof(double) * 4 * km->n_sets, cudaMemcpyDeviceToHost, gpu.stream));
    MLB_TRY(mlb_ctx_synchronize(km->ctx));
    for (int s = 0; s < km->n_sets; ++s)
        if (((active >> s) & 1u) && centroid_shift_sq) centroid_shift_sq[s] = host[4 * s];
    km->have_stats &= ~active;
    return MLB_OK;
}

int mlb_kms_get_labels(mlb_kms* km, int set, unsigned int* labels)
{
    MLB_ENTER(km ? km->ctx : nullptr);
    MLB_REQUIRE(km && labels, "mlb_kms_get_labels: null argument");
    MLB_REQUIRE(set >= 0 && set < km->n_sets, "mlb_kms_get_labels: set %d out of range", set);
    const int64_t host_begin = km->ctx->rank_mode ? km->data->shards[0].begin : 0;
    MLB_TRY(for_each_gpu(km->ctx, [&](int g, Gpu& gpu) -> int {
        const DataShard& sh = km->data->shards[g];
        const size_t stride = static_cast<size_t>(std::max<int64_t>(1, sh.n()));
        if (sh.n() > 0) MLB_TRY(staged_d2h(gpu, labels + (sh.begin - host_begin), km->gpus[g].labels + static_cast<size_t>(set) * stride, sizeof(unsigned) * sh.n()));
        return MLB_OK;
    }));
    return mlb_ctx_synchronize(km->ctx);
}

int mlb_kms_launch_count(const mlb_kms* km, int64_t* launches)
{
    MLB_REQUIRE(km && launches, "mlb_kms_launch_count: null argument");
    *launches = km->launches;
    return MLB_OK;
}

}  // extern "C"
