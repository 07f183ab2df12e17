// Gaussian-mixture EM on B200 (sm_100a), FP64.  Replaces the loops of ML/EM.cpp:
//     expectation_step   EM.cpp:190-219      maximisation_step   EM.cpp:221-263
//     process_covariances EM.cpp:274-287     calculate_labels    EM.cpp:289-304
//     calculate_sample_covariance EM.cpp:265-272
//
// Formulation (DESIGN.md "EM kernels").  With z = x - c (c = the global data mean, held per data
// set) every point has a feature vector phi(z) = [1, z_a, z_a z_b (a <= b)].  Then
//   E-step:  log(pi_k N_k(x)) + D/2 log(2 pi) = phi(z) . theta_k        -- a [points x F] x [F x K] product
//   M-step:  S[f][k] = sum_i phi_f(z_i) r_ik                             -- a [F x points] x [points x K] product
// where theta_k packs -1/2 Sigma_k^-1, Sigma_k^-1 (mu_k - c) and the constant, and S packs the
// weighted count, first and second moments about c.  Both products run on the FP64 tensor pipe
// (mma.sync.m8n8k4.f64 -> DMMA.8x8x4), the features are generated in registers from the point
// tile in shared memory.  Three kernel families share this formulation, the partial-statistics
// layout, the reduction and the parameter refresh below:
//     em_small_kernel (em_small.cuh)  D <= 8,  K <= 32   fused E+M, every warp on its own 16-point sub-tiles
//     em_kernel       (this file)     D <= 16, K <= 32   fused E+M, 64-point tiles, M-step split over the warps
//     em_split_*      (em_split.cuh)  D <= 64, K <= 256  E kernel + M kernel, Theta streamed, R resident in HBM
// The fused kernels read X exactly once per iteration and the responsibilities never leave the SM.
//
// Determinism: per-chunk partial statistics in a fixed layout, chunks are a function of N only,
// fixed-order reduction (context.cu), no floating-point atomics anywhere.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>

#include "em_direct.cuh"
#include "em_split.cuh"
#include "fastmath.cuh"
#include "internal.h"

namespace mlb {

constexpr int kTile = 64;        // points per CTA tile
constexpr int kEmThreads = 128;  // 4 warps
constexpr int kLogBatch = 16;    // tiles between two log() calls of the log-likelihood partial

#ifdef MLB_EM_LIBM_EXP
#define MLB_EM_EXP(x) exp(x)
#else
#define MLB_EM_EXP(x) exp_nonpositive((x), etab)
#endif
#ifndef MLB_EM_MINB_SMALL
#define MLB_EM_MINB_SMALL 4
#endif

// ---- compile-time shape helpers -------------------------------------------------------------
// E-step contraction steps.  One step feeds 4 features (one per lane c = lane & 3 of a quad) of 8 points to a
// DMMA.8x8x4.  With the D coordinates cut into DQ = DP/4 blocks of 4, the D(D+1)/2 + D features are packed as
//   off-diagonal block pairs (ma < mb), 4 steps each:  lane c holds z_a * z_{4 mb + c},  a = 4 ma + i
//   diagonal blocks, "rotations" of the quad:          r = 0: z_{4m+c}^2
//                                                      r = 1: z_{4m+c} * z_{4m+(c+1)%4}
//                                                      r = 2: only 2 distinct products per block, so two blocks
//                                                             share a step (lanes 0,1: block 2h; lanes 2,3: block 2h+1)
//   linear terms:                                      lane c holds z_{4m+c}
// which is exactly D(D+1)/2 + D slots when DQ is even: no padding products, unlike a square 4x4 tiling of the
// diagonal blocks (which spends 16 slots on 10 distinct products).
__host__ __device__ constexpr int em_ne_offdiag(int DP) { return 4 * (DP / 4) * (DP / 4 - 1) / 2; }
__host__ __device__ constexpr int em_ne(int DP) { return em_ne_offdiag(DP) + 2 * (DP / 4) + (DP / 4 + 1) / 2 + DP / 4; }
// index of the first off-diagonal step of coordinate a = 4 ma + i against block mb > ma
__host__ __device__ constexpr int em_estep_offdiag(int DP, int a, int mb)
{
    const int DQ = DP / 4, ma = a / 4, i = a % 4;
    int n = 0;
    for (int m = 0; m < ma; ++m) n += 4 * (DQ - 1 - m);
    return n + i * (DQ - 1 - ma) + (mb - ma - 1);
}
// M-step features: 1, z_a, z_a z_b (a <= b), padded to a multiple of 8 rows.
__host__ __device__ constexpr int em_fm_raw(int DP) { return 1 + DP + DP * (DP + 1) / 2; }
__host__ __device__ constexpr int em_nm(int DP) { return (em_fm_raw(DP) + 7) / 8; }
__host__ __device__ constexpr int em_sv(int DP, int KP) { return em_nm(DP) * 8 * KP + 8; }
__host__ __device__ constexpr int em_theta_len(int DP, int KP) { return em_ne(DP) * (KP / 8) * 32 + KP; }

constexpr size_t em_smem_bytes(int DP, int KP)
{
    return sizeof(double) * (em_theta_len(DP, KP) + 2 * kTile * (DP + 4) + kTile * (KP + 4) + 8 + DP + kExpTableSize);
}

struct EmArgs {
    const double* x;       // local points, d doubles each
    long long n_local;
    int d, k;
    const double* shift;   // d
    const double* theta;   // E-step image: [NE][NT/2][32 lanes][2] (or [NE][32] for NT == 1), then KP constants
    const int2* feat_m;    // [NM*8] Z-row offsets (ia, ib) of each M-step feature
    double* partials;      // [n_chunks][SV]
    int chunk;             // points per chunk
    int n_chunks;
    unsigned* counter;     // dynamic chunk scheduler
    const double* r_in;    // MODE 1: responsibilities, column-major local rows
    long long r_ld;
    double* r_out;         // MODE 2: responsibilities of [range_begin, range_begin + range_count), column-major
    long long r_out_ld;
    unsigned* labels_out;  // MODE 2
    long long range_begin, range_count;
};

__device__ __forceinline__ long long min64(long long a, long long b) { return a < b ? a : b; }

__device__ __forceinline__ void dmma(double (&acc)[2], double a, double b)
{
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(acc[0]), "+d"(acc[1]) : "d"(a), "d"(b));
}

template <int NT>
__device__ __forceinline__ void load_theta_frag(const double* thE, int j, int lane, double (&bf)[NT])
{
    if constexpr (NT == 1) {
        bf[0] = thE[j * 32 + lane];
    } else {
#pragma unroll
        for (int h = 0; h < NT / 2; ++h) {
            const double2 v = reinterpret_cast<const double2*>(thE)[(j * (NT / 2) + h) * 32 + lane];
            bf[2 * h] = v.x;
            bf[2 * h + 1] = v.y;
        }
    }
}

// MODE 0: fused E+M step.  MODE 1: M-step from given responsibilities.  MODE 2: E-step only,
// writing responsibilities and labels (the "emit" pass).
template <int DP, int KP, int MODE>
__global__ void __launch_bounds__(kEmThreads, (DP * KP <= 128 || MODE == 2) ? MLB_EM_MINB_SMALL : 2) em_kernel(const EmArgs p)
{
    constexpr int NT = KP / 8, DQ = DP / 4, NE = em_ne(DP), NM = em_nm(DP);
    constexpr int ZS = DP + 4, RS = KP + 4;
    constexpr int WN = (NM >= 8 || NT == 1) ? 1 : 2, WM = 4 / WN;
    constexpr int MW = (NM + WM - 1) / WM, NW = NT / WN;
    constexpr int SV = em_sv(DP, KP);
    constexpr int XR = kTile * DP / kEmThreads;

    extern __shared__ __align__(16) double sm[];
    double* thE = sm;
    double* cE = thE + NE * NT * 32;
    double* Zb = cE + KP;
    double* R = Zb + 2 * kTile * ZS;
    double* wl = R + kTile * RS;
    double* sh = wl + 8;
    double* etab = sh + DP;   // 2^(j/32) for exp_nonpositive
    __shared__ int s_next;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, c = lane & 3;
    const int d = p.d;

    if (MODE != 1)
        for (int i = tid; i < em_theta_len(DP, KP); i += kEmThreads) sm[i] = p.theta[i];
    for (int i = tid; i < 2 * kTile * ZS; i += kEmThreads) Zb[i] = 0.0;
    for (int i = tid; i < kTile * RS; i += kEmThreads) R[i] = 0.0;
    if (tid < DP) sh[tid] = tid < d ? p.shift[tid] : 0.0;
    load_exp_table(etab);

    // M-step ownership: warp (wm, wn) holds feature tiles wm*MW .. wm*MW+MW-1 x component tiles wn*NW .. +NW-1.
    const int wm = warp / WN, wn = warp % WN;
    int ia[MW], ib[MW];
    double sacc[MW][NW][2];
    if (MODE != 2) {
#pragma unroll
        for (int i = 0; i < MW; ++i) {
            const int mt = wm * MW + i;
            const int2 f = mt < NM ? p.feat_m[mt * 8 + g] : make_int2(DP + 1, DP + 1);
            ia[i] = f.x;
            ib[i] = f.y;
        }
    }

    double xr[XR];
    auto load_tile = [&](long long point0, int nvalid) {
        const double* xg = p.x + point0 * d;
        const int nel = nvalid * d;
#pragma unroll
        for (int r = 0; r < XR; ++r) {
            const int e = tid + kEmThreads * r;
            xr[r] = e < nel ? xg[e] : 0.0;
        }
    };
    auto store_tile = [&](double* Z, int nvalid) {
        const int nel = nvalid * d;
#pragma unroll
        for (int r = 0; r < XR; ++r) {
            const int e = tid + kEmThreads * r;
            if (e < kTile * d) {
                const int pt = (d == DP) ? e / DP : FastDiv(d).div(e);
                const int dm = e - pt * d;
                Z[pt * ZS + dm] = e < nel ? xr[r] - sh[dm] : 0.0;
            }
        }
        if (tid < kTile) Z[tid * ZS + DP] = tid < nvalid ? 1.0 : 0.0;
    };

    const long long work_begin = MODE == 2 ? p.range_begin : 0;
    const long long work_end = MODE == 2 ? p.range_begin + p.range_count : p.n_local;

    for (;;) {
        __syncthreads();
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        __syncthreads();
        const int chunk = s_next;
        if (chunk >= p.n_chunks) break;
        const long long p_begin = work_begin + static_cast<long long>(chunk) * p.chunk;
        const long long p_end = min64(p_begin + p.chunk, work_end);
        const int ntiles = static_cast<int>((p_end - p_begin + kTile - 1) / kTile);

        if (MODE != 2) {
#pragma unroll
            for (int i = 0; i < MW; ++i)
#pragma unroll
                for (int nt = 0; nt < NW; ++nt) sacc[i][nt][0] = sacc[i][nt][1] = 0.0;
        }
        // log-likelihood partial: sum_i (max_i + log(sum_i)).  The sums (each in [1, K]) are multiplied up over
        // kLogBatch tiles and logged once, so the log costs 1/kLogBatch per point (2^(5*2*kLogBatch) at most).
        double ll_acc = 0.0, ll_prod = 1.0;

        load_tile(p_begin, static_cast<int>(min64(kTile, p_end - p_begin)));
        store_tile(Zb, static_cast<int>(min64(kTile, p_end - p_begin)));
        __syncthreads();

        for (int t = 0; t < ntiles; ++t) {
            double* Z = Zb + (t & 1) * kTile * ZS;
            const long long tile0 = p_begin + static_cast<long long>(t) * kTile;
            const int nvalid = static_cast<int>(min64(kTile, p_end - tile0));
            const int nvalid_next = t + 1 < ntiles ? static_cast<int>(min64(kTile, p_end - tile0 - kTile)) : 0;
            if (t + 1 < ntiles) load_tile(tile0 + kTile, nvalid_next);

            if (MODE == 1) {
                // responsibilities given by the caller (maximise_first, EM.cpp:120-125)
                for (int idx = tid; idx < kTile * p.k; idx += kEmThreads) {
                    const int pt = idx % kTile, kk = idx / kTile;
                    R[pt * RS + kk] = pt < nvalid ? p.r_in[tile0 + pt + kk * p.r_ld] : 0.0;
                }
            } else {
                // ---------------- E-step: Q = Phi(Z) . Theta for this warp's 16 points x all components
                const double* z0 = Z + (warp * 16 + g) * ZS;
                const double* z1 = z0 + 8 * ZS;
                double acc[2][NT][2];
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const double2 cc = *reinterpret_cast<const double2*>(cE + 8 * nt + 2 * c);
                    acc[0][nt][0] = acc[1][nt][0] = cc.x;
                    acc[0][nt][1] = acc[1][nt][1] = cc.y;
                }
                double zc0[DQ], zc1[DQ];
#pragma unroll
                for (int m = 0; m < DQ; ++m) {
                    zc0[m] = z0[4 * m + c];
                    zc1[m] = z1[4 * m + c];
                }
                auto estep = [&](int j, double a0, double a1) {
                    double bf[NT];
                    load_theta_frag<NT>(thE, j, lane, bf);
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        dmma(acc[0][nt], a0, bf[nt]);
                        dmma(acc[1][nt], a1, bf[nt]);
                    }
                };
                // off-diagonal block pairs
#pragma unroll
                for (int a = 0; a < DP - 4; ++a) {
                    const double za0 = z0[a], za1 = z1[a];
#pragma unroll
                    for (int m = a / 4 + 1; m < DQ; ++m) estep(em_estep_offdiag(DP, a, m), za0 * zc0[m], za1 * zc1[m]);
                }
                // diagonal blocks: squares, first rotation, paired second rotation
                constexpr int J0 = em_ne_offdiag(DP);
#pragma unroll
                for (int m = 0; m < DQ; ++m) estep(J0 + m, zc0[m] * zc0[m], zc1[m] * zc1[m]);
#pragma unroll
                for (int m = 0; m < DQ; ++m) {
                    const int o = 4 * m + ((c + 1) & 3);
                    estep(J0 + DQ + m, zc0[m] * z0[o], zc1[m] * z1[o]);
                }
#pragma unroll
                for (int h = 0; h < (DQ + 1) / 2; ++h) {
                    const int mx = 2 * h + (c >> 1);                 // lanes 2,3 take the odd block of the pair
                    const int o = 4 * mx + c, o2 = 4 * mx + ((c + 2) & 3);
                    const bool live = mx < DQ;                        // DQ odd: the last pair has no second block
                    const double u0 = live ? z0[o] * z0[o2] : 0.0, u1 = live ? z1[o] * z1[o2] : 0.0;
                    estep(J0 + 2 * DQ + h, u0, u1);
                }
                // linear terms
#pragma unroll
                for (int m = 0; m < DQ; ++m) estep(NE - DQ + m, zc0[m], zc1[m]);
                // ---------------- log-sum-exp over the 4 lanes that share a point
                double mxs[2], sums[2];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
#ifdef MLB_EM_FMAX_SHIFT
                    double mx = -INFINITY;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) mx = fmax(mx, fmax(acc[mt][nt][0], acc[mt][nt][1]));
                    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
                    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
#else
                    int mkey = lse_key(acc[mt][0][0]);
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) mkey = max(mkey, max(lse_key(acc[mt][nt][0]), lse_key(acc[mt][nt][1])));
                    mkey = max(mkey, __shfl_xor_sync(0xffffffffu, mkey, 1));
                    mkey = max(mkey, __shfl_xor_sync(0xffffffffu, mkey, 2));
                    const double mx = lse_shift_of_key(mkey);   // within 2^-20 of the largest term (fastmath.cuh)
#endif
                    double sum = 0.0;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        acc[mt][nt][0] = MLB_EM_EXP(acc[mt][nt][0] - mx);
                        acc[mt][nt][1] = MLB_EM_EXP(acc[mt][nt][1] - mx);
                        sum += acc[mt][nt][0] + acc[mt][nt][1];
                    }
                    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                    mxs[mt] = mx;
                    sums[mt] = sum;
                }
                // One reciprocal per lane instead of two: the four lanes of a quad hold the same two sums, so the even lanes
                // invert the first point's and the odd lanes the second point's, and a shuffle hands both to everybody.
                const double inv_mine = reciprocal_of_sum((c & 1) ? sums[1] : sums[0]);
                const double invs[2] = {__shfl_sync(0xffffffffu, inv_mine, lane & ~1), __shfl_sync(0xffffffffu, inv_mine, lane | 1)};
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    const int pl = warp * 16 + mt * 8 + g;
                    const double inv = invs[mt];
                    if (c == 0 && pl < nvalid) {
                        ll_acc += mxs[mt];
                        ll_prod *= sums[mt];
                    }
                    if (MODE == 0) {
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt)
                            *reinterpret_cast<double2*>(R + pl * RS + 8 * nt + 2 * c) = make_double2(acc[mt][nt][0] * inv, acc[mt][nt][1] * inv);
                    } else {
                        // emit: responsibilities_ (EM.cpp:213-218) and labels_ (EM.cpp:289-304, first maximum wins)
                        double best = -1.0;
                        unsigned best_k = 0xffffffffu;
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const int kk = 8 * nt + 2 * c + e;
                                const double r = acc[mt][nt][e] * inv;
                                if (kk < p.k) {
                                    if (pl < nvalid && p.r_out) p.r_out[(tile0 - p.range_begin) + pl + kk * p.r_out_ld] = r;
                                    if (r > best) { best = r; best_k = kk; }
                                }
                            }
#pragma unroll
                        for (int off = 1; off <= 2; off <<= 1) {
                            const double ob = __shfl_xor_sync(0xffffffffu, best, off);
                            const unsigned ok = __shfl_xor_sync(0xffffffffu, best_k, off);
                            if (ob > best || (ob == best && ok < best_k)) { best = ob; best_k = ok; }
                        }
                        if (c == 0 && pl < nvalid && p.labels_out) p.labels_out[(tile0 - p.range_begin) + pl] = best_k;
                    }
                }
            }
            if (MODE != 2) {
                __syncthreads();
                // ---------------- M-step: S += Phi(Z)^T . R over the tile's 64 points
#pragma unroll 4
                for (int s = 0; s < kTile / 4; ++s) {
                    const double* zp = Z + (4 * s + c) * ZS;
                    const double* rp = R + (4 * s + c) * RS + wn * NW * 8 + g;
                    double bf[NW];
#pragma unroll
                    for (int nt = 0; nt < NW; ++nt) bf[nt] = rp[8 * nt];
#pragma unroll
                    for (int i = 0; i < MW; ++i) {
                        if (wm * MW + i < NM) {
                            const double af = zp[ia[i]] * zp[ib[i]];
#pragma unroll
                            for (int nt = 0; nt < NW; ++nt) dmma(sacc[i][nt], af, bf[nt]);
                        }
                    }
                }
            }
            if (MODE != 1 && ((t & (kLogBatch - 1)) == kLogBatch - 1 || t + 1 == ntiles)) {
                ll_acc += log(ll_prod);
                ll_prod = 1.0;
            }
            if (t + 1 < ntiles) store_tile(Zb + ((t + 1) & 1) * kTile * ZS, nvalid_next);
            __syncthreads();
        }

        if (MODE != 2) {
            double* out = p.partials + static_cast<long long>(chunk) * SV;
#pragma unroll
            for (int i = 0; i < MW; ++i) {
                const int mt = wm * MW + i;
                if (mt < NM) {
#pragma unroll
                    for (int nt = 0; nt < NW; ++nt)
                        *reinterpret_cast<double2*>(out + (mt * 8 + g) * KP + (wn * NW + nt) * 8 + 2 * c) = make_double2(sacc[i][nt][0], sacc[i][nt][1]);
                }
            }
            // log-likelihood partial: fixed butterfly inside the warp, fixed order across warps
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) ll_acc += __shfl_xor_sync(0xffffffffu, ll_acc, off);
            if (lane == 0) wl[warp] = ll_acc;
            __syncthreads();
            if (tid == 0) out[NM * 8 * KP] = (wl[0] + wl[1]) + (wl[2] + wl[3]);
            if (tid >= 1 && tid < 8) out[NM * 8 * KP + tid] = 0.0;
        }
    }
}

#include "em_small.cuh"

// ---------------------------------------------------------------- parameter refresh (replicated on every GPU)
//
// One block per (padded) component.  Stage 1 (vsum != nullptr): fixed-tree sum of the 8 virtual
// shard vectors, then mean / covariance / weight (EM.cpp:238-257) from moments about the shift c:
//     mu = c + m1/s,   Sigma = m2/s - (m1/s)(m1/s)^T + 1e-15 I,   pi = s/N.
// Stage 2: process_covariances (EM.cpp:274-287): Cholesky, inverse by solving against the identity,
// sqrt|Sigma| = prod L_ii; then the E-step image theta for the next iteration.
struct EmFinalizeArgs {
    const double* vsum;   // feature-path statistics [8][SV] (moments about the shift c), or nullptr
    const double* dstats; // direct-path statistics [8][dSV] (augmented moments about each component's old mean), or nullptr
    const double* shift;
    int d, k, DP, KP, SV;
    int DPd, dSV;         // direct path: D padded to 8, length of a statistics vector
    long long n_total;
    const int2* feat_m;   // [NM*8]
    const int2* feat_e;   // [NE*4]: (a, b); b == DP: linear term a; a < 0: unused slot
    int nm8, ne;
    double* means;        // D x K
    double* covs;         // K x (D x D)
    double* weights;      // K
    double* inv_covs;     // K x (D x D)
    double* sqrt_dets;    // K
    double* theta_out;    // E-step image of the feature kernels, or nullptr (shapes only the direct kernels take)
    double* dimg_out;     // E-step images of the direct kernels [k][dr_img_len(DPd)], or nullptr
    double* kappa_out;    // [k] delta^T P delta: how far (in its own standard deviations, squared) a component sits from the shift
    int p_in_smem;        // the inverse covariance fits next to the factor in shared memory
    double* ll_ring;      // ring of log-likelihoods of the E-steps whose statistics these are (nullptr: skip)
    unsigned long long* ll_counter;   // device-side step counter: the ring slot written is *ll_counter % ring, then it is incremented
    int ll_ring_len;
};

__global__ void em_finalize_kernel(const EmFinalizeArgs p)
{
    extern __shared__ double fs[];
    const int d = p.d, DP = p.DP, KP = p.KP, NT = KP / 8;
    double* A = fs;            // covariance, column-major d x d, factorised in place
    double* L = A;             // Cholesky factor (lower)
    double* delta = A + d * d; // mean - shift
    double* m1 = delta + d;
    double* v = m1 + d;        // P delta
    const int kc = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
    double* P = p.p_in_smem ? v + d : p.inv_covs + static_cast<long long>(kc < p.k ? kc : 0) * d * d;   // inverse covariance
    __shared__ double s_count, s_const;
    const bool real = kc < p.k;
    double weight = 0.0;

    if (real) {
        if (p.vsum) {
            for (int f = tid; f < p.nm8; f += nthr) {
                const int2 ab = p.feat_m[f];
                const double val = tree8(p.vsum + static_cast<long long>(f) * KP + kc, p.SV);
                if (ab.x == DP && ab.y == DP) s_count = val;
                else if (ab.y == DP && ab.x < d) m1[ab.x] = val;
                else if (ab.x < d && ab.y < d) { A[ab.x + ab.y * d] = val; A[ab.y + ab.x * d] = val; }
            }
            __syncthreads();
            const double s = s_count;
            for (int a = tid; a < d; a += nthr) delta[a] = m1[a] / s;
            __syncthreads();
            for (int e = tid; e < d * d; e += nthr) {
                const int a = e % d, b = e / d;
                double cv = A[e] / s - delta[a] * delta[b];
                if (a == b) cv += 1e-15;   // EM.cpp:250-256
                A[e] = cv;
                p.covs[static_cast<long long>(kc) * d * d + e] = cv;
            }
            weight = s / static_cast<double>(p.n_total);
            for (int a = tid; a < d; a += nthr) p.means[a + kc * d] = p.shift[a] + delta[a];
            if (tid == 0) p.weights[kc] = weight;
        } else if (p.dstats) {
            // Moments about the component's own previous mean (em_direct.cuh): s, m1 = sum r w, m2 = sum r w w^T with
            // w = x - mu_old.  mu_new = mu_old + m1/s, Sigma = m2/s - (m1/s)(m1/s)^T + 1e-15 I (EM.cpp:238-257).
            const int NBa = p.DPd / 8 + 1, NB = NBa - 1;
            const double* st = p.dstats + static_cast<long long>(kc) * dr_stat_len(p.DPd);
            if (tid == 0) s_count = tree8(st + dr_tile_index(NBa, NB, NB) * 64, p.dSV);
            for (int a = tid; a < d; a += nthr) m1[a] = tree8(st + dr_tile_index(NBa, a / 8, NB) * 64 + (a % 8) * 8, p.dSV);
            for (int e = tid; e < d * d; e += nthr) {
                const int a = e % d, b = e / d;
                if (a <= b) {   // the tile entry (a, b) only: (r w_a) w_b and (r w_b) w_a round differently
                    const double val = tree8(st + dr_tile_index(NBa, a / 8, b / 8) * 64 + (a % 8) * 8 + (b % 8), p.dSV);
                    A[a + b * d] = val;
                    A[b + a * d] = val;
                }
            }
            __syncthreads();
            const double s = s_count;
            for (int a = tid; a < d; a += nthr) m1[a] = m1[a] / s;
            __syncthreads();
            for (int e = tid; e < d * d; e += nthr) {
                const int a = e % d, b = e / d;
                double cv = A[e] / s - m1[a] * m1[b];
                if (a == b) cv += 1e-15;
                A[e] = cv;
                p.covs[static_cast<long long>(kc) * d * d + e] = cv;
            }
            weight = s / static_cast<double>(p.n_total);
            for (int a = tid; a < d; a += nthr) {
                const double mean = p.means[a + kc * d] + m1[a];
                p.means[a + kc * d] = mean;
                delta[a] = mean - p.shift[a];
            }
            if (tid == 0) p.weights[kc] = weight;
        } else {
            for (int e = tid; e < d * d; e += nthr) A[e] = p.covs[static_cast<long long>(kc) * d * d + e];
            for (int a = tid; a < d; a += nthr) delta[a] = p.means[a + kc * d] - p.shift[a];
            weight = p.weights[kc];
        }
        __syncthreads();
        // Unblocked left-looking Cholesky in place, sequential inner sums (same order as the oracle's restatement of Eigen::LLT).
        for (int j = 0; j < d; ++j) {
            if (tid == 0) {
                double x = L[j + j * d];
                double sq = 0.0;
                for (int t = 0; t < j; ++t) sq += L[j + t * d] * L[j + t * d];
                if (j > 0) x -= sq;
                L[j + j * d] = sqrt(x);
            }
            __syncthreads();
            const double ljj = L[j + j * d];
            for (int i = j + 1 + tid; i < d; i += nthr) {
                double dot = 0.0;
                for (int t = 0; t < j; ++t) dot += L[i + t * d] * L[j + t * d];
                double val = L[i + j * d];
                if (j > 0) val -= dot;
                L[i + j * d] = val / ljj;
            }
            __syncthreads();
        }
        // llt.solve(Identity): forward then backward substitution, one column per thread (only the lower triangle of L is read).
        for (int col = tid; col < d; col += nthr) {
            double* x = P + col * d;
            for (int i = 0; i < d; ++i) x[i] = i == col ? 1.0 : 0.0;
            for (int i = 0; i < d; ++i) {
                double val = x[i];
                for (int j = 0; j < i; ++j) val -= L[i + j * d] * x[j];
                x[i] = val / L[i + i * d];
            }
            for (int i = d - 1; i >= 0; --i) {
                double val = x[i];
                for (int j = i + 1; j < d; ++j) val -= L[j + i * d] * x[j];
                x[i] = val / L[i + i * d];
            }
        }
        __syncthreads();
        if (p.p_in_smem)
            for (int e = tid; e < d * d; e += nthr) p.inv_covs[static_cast<long long>(kc) * d * d + e] = P[e];
        // v = P_sym delta using the upper triangle only, as xAx_symmetric does (LinearAlgebra.cpp:17-29)
        for (int a = tid; a < d; a += nthr) {
            double acc = 0.0;
            for (int b = 0; b < d; ++b) acc += (b >= a ? P[a + b * d] : P[b + a * d]) * delta[b];
            v[a] = acc;
        }
        __syncthreads();
        if (tid == 0) {
            double sqrt_det = 1.0;
            for (int i = 0; i < d; ++i) sqrt_det *= L[i + i * d];
            p.sqrt_dets[kc] = sqrt_det;
            double dv = 0.0;
            for (int a = 0; a < d; ++a) dv += delta[a] * v[a];
            s_const = log(weight / sqrt_det) - 0.5 * dv;
            if (p.kappa_out) p.kappa_out[kc] = dv;
            if (p.dimg_out) p.dimg_out[static_cast<long long>(kc) * dr_img_len(p.DPd) + dr_steps(p.DPd / 8) * 32 + p.DPd] = log(weight / sqrt_det);
        }
        __syncthreads();
        if (p.dimg_out) {
            // Direct-kernel image: the DMMA steps of P' (block upper triangle; 2 P above the diagonal blocks), then delta.
            const int NB = p.DPd / 8, SPC = dr_steps(NB);
            double* im = p.dimg_out + static_cast<long long>(kc) * dr_img_len(p.DPd);
            for (int idx = tid; idx < SPC * 32; idx += nthr) {
                const int step = idx >> 5, lane = idx & 31, g = lane >> 2, c = lane & 3;
                int B = 0;
                while ((B + 1) * (B + 2) <= step) ++B;        // steps before block column B: B (B + 1)
                const int s2 = step - B * (B + 1);
                const int a = 4 * s2 + c, n = 8 * B + g;
                double val = 0.0;
                if (a < d && n < d) {
                    val = a <= n ? P[a + n * d] : P[n + a * d];
                    if (a / 8 != B) val *= 2.0;
                }
                im[idx] = val;
            }
            for (int a = tid; a < p.DPd; a += nthr) im[SPC * 32 + a] = a < d ? delta[a] : 0.0;
            if (tid >= 1 && tid < 8) im[SPC * 32 + p.DPd + tid] = 0.0;
        }
    }
    // E-step image of the feature kernels
    if (p.theta_out) {
        const int nt = kc / 8, row = kc % 8;
        for (int idx = tid; idx < p.ne * 4; idx += nthr) {
            const int j = idx >> 2, c = idx & 3;
            const int2 ab = p.feat_e[idx];
            double val = 0.0;
            if (real && ab.x >= 0 && ab.x < d) {
                if (ab.y == DP) val = v[ab.x];
                else if (ab.y < d) val = ab.x == ab.y ? -0.5 * P[ab.x + ab.x * d] : -P[ab.x + ab.y * d];
            }
            const int lane = row * 4 + c;
            if (NT == 1) p.theta_out[j * 32 + lane] = val;
            else p.theta_out[((j * (NT / 2) + nt / 2) * 32 + lane) * 2 + (nt & 1)] = val;
        }
        if (tid == 0 && kc < KP) p.theta_out[p.ne * NT * 32 + kc] = real ? s_const : -INFINITY;
    }
    if (p.ll_ring && (p.vsum || p.dstats) && kc == 0 && tid == 0) {
        const double ll_sum = p.vsum ? tree8(p.vsum + (p.SV - 8), p.SV) : tree8(p.dstats + (p.dSV - 8), p.dSV);
        // mean over points minus D log(2 pi) / 2 (EM.cpp:197-211).  The slot comes from a device-side counter so that
        // the launch arguments are the same for every step (the step is replayed from a CUDA graph).
        const unsigned long long idx = *p.ll_counter;
        p.ll_ring[idx % p.ll_ring_len] = ll_sum / static_cast<double>(p.n_total) - 0.5 * d * log(2.0 * 3.14159265358979323846);
        *p.ll_counter = idx + 1;
    }
}

__global__ void selftest_exp_kernel(const double* x, long long n, double* out)
{
    __shared__ double etab[kExpTableSize];
    load_exp_table(etab);
    __syncthreads();
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = exp_nonpositive(x[i], etab);
}

// ---------------------------------------------------------------- dispatch

using EmKernelFn = void (*)(EmArgs);

template <int MODE>
static EmKernelFn em_kernel_for(int DP, int KP)
{
#define MLB_EM_CASE(D_, K_) if (DP == D_ && KP == K_) return em_kernel<D_, K_, MODE>;
#define MLB_EM_SMALL_CASE(D_, K_) if (DP == D_ && KP == K_) return em_small_kernel<D_, K_, MODE>;
    MLB_EM_SMALL_CASE(4, 8) MLB_EM_SMALL_CASE(4, 16) MLB_EM_SMALL_CASE(4, 32)
    MLB_EM_SMALL_CASE(8, 8) MLB_EM_SMALL_CASE(8, 16) MLB_EM_SMALL_CASE(8, 32)
    MLB_EM_CASE(16, 8) MLB_EM_CASE(16, 16) MLB_EM_CASE(16, 32)
#undef MLB_EM_CASE
#undef MLB_EM_SMALL_CASE
    return nullptr;
}

struct EmGpu {
    double* theta[2] = {nullptr, nullptr};
    double* params = nullptr;  // means | covs | weights | inv_covs | sqrt_dets
    double* partials = nullptr;
    double* vsum = nullptr;
    double* ll = nullptr;      // ring of log-likelihoods
    unsigned long long* ll_counter = nullptr;   // device-side count of completed steps (selects the ring slot)
    int2* feat_m = nullptr;
    int2* feat_e = nullptr;
    unsigned* counter = nullptr;
    double* stage = nullptr;   // emit / responsibilities staging
    unsigned* stage_labels = nullptr;
    int grid = 0;
    // split path (general shapes)
    double* r = nullptr;         // [n_local][KP] responsibilities of the last E-step
    double* ll_tile = nullptr;   // [n_chunks][chunk / 64] per-tile log-likelihood sums (E kernel -> M kernel)
    int2* feat_e_off = nullptr;  // E-step slots as Z-row offsets
    int grid_e = 0, grid_m = 0;
    KernelTimer timer;
};

using EmSplitKernelFn = void (*)(EmSplitArgs);

// Direct-difference kernels (em_direct.cuh): per-GPU buffers.  The image and kappa are small and always present; the
// responsibilities, the super-chunk partials and the tables are allocated when the path is first taken.
struct EmDirectGpu {
    double* img = nullptr;        // [k][IMG] component images
    double* kappa = nullptr;      // [k] delta^T P delta of the current parameters
    double* r = nullptr;          // [n_local][KPr]
    double* ll_tile = nullptr;    // [ceil(n_local / 64)]
    double* partials = nullptr;   // [n_sc][SVd]
    double* vsum = nullptr;       // [8][SVd]
    long long* sc_begin = nullptr;   // [n_sc + 1]
    int2* tile_tab = nullptr;     // [T]
    int n_sc = 0;
    int grid_e = 0, grid_m = 0;
};

struct EmDirect {
    bool capable = false;         // D <= 128
    bool ready = false;           // the large buffers exist
    int DP = 0, NB = 0, KPr = 0, IMG = 0, L = 0, SVd = 0;
    int cb = 1, cg = 1, tiles_per_range = 0, n_ranges = 1;
    size_t smem_e = 0, smem_m = 0;
    int64_t sc_bounds[kVirtualShards + 1] = {};   // global super-chunk boundaries of the virtual shards
    std::vector<EmDirectGpu> gpus;
    ReduceScratch scratch;
};

constexpr int kDirectMaxDim = 128;
// Above this kappa = max_k (mu_k - c)^T P_k (mu_k - c) the step is routed to the direct kernels.  The feature-space kernels
// lose about 5e-17 * kappa to cancellation (measured against the reference: 1e-10 at kappa = 2e6, 2e-8 at 2e8;
// tests/test_gpu_numerical_domain.py), so the threshold keeps them ~1.5e-11 from the reference, two orders inside the
// 1e-9 bar.  It was 3e4 until r02k: kappa also grows when a component starves (its covariance shrinks onto a few
// points), which an ordinary fit does now and then (bench.py's own C3 run reaches 4.4e4 from iteration 19 on, one
// component at a weight of 2e-7: profiles/kappa_trace_r02k.jsonl), and the direct kernels are ~7x slower.
constexpr double kKappaDirect = 3.0e5;

constexpr int kLlRing = 4096;
constexpr long long kStagePoints = 1 << 20;

}  // namespace mlb

using namespace mlb;

struct mlb_em {
    mlb_ctx* ctx = nullptr;
    mlb_data* data = nullptr;
    int d = 0, k = 0, DP = 0, KP = 0, NT = 0, NE = 0, NM = 0, SV = 0;
    std::vector<int2> feat_m, feat_e;
    std::vector<EmGpu> gpus;
    int cur = 0;
    bool have_params = false, have_step = false;
    int last_path = 0;
    int64_t direct_steps = 0;    // steps that took the direct kernels so far (mlb_em_direct_steps)
    int64_t launches = 0;
    int64_t steps_done = 0;
    EmKernelFn fn_step = nullptr, fn_mstep = nullptr, fn_emit = nullptr;
    int path = 1;                // feature-space kernels of this shape: 1 fused E+M (D <= 16, K <= 32), 2 split E / M; 0: none (D > 64 or K > 256)
    EmDirect dr;                 // direct-difference kernels
    int forced_path = 0;         // mlb_em_force_path: 0 automatic, 3 always direct
    int route = 1;               // the path the NEXT step takes with the current parameters: `path`, or 3 (direct)
    double kappa_max = 0.0;      // max_k (mu_k - c)^T P_k (mu_k - c) of the current parameters
    bool r_direct_valid = false; // the direct R buffer holds the responsibilities of the last step
    double* kappa_host = nullptr;   // pinned: kappa of the current parameters on its way to the routing decision
    EmSplitKernelFn fn_split_e = nullptr, fn_split_m = nullptr;
    size_t smem_split_e = 0, smem_split_m = 0;
    size_t smem_fused = 0;       // dynamic shared memory of the fused kernels (em_small_kernel for D <= 8, em_kernel for D = 16)
    int MW = 4;                  // split M kernel: feature tiles per warp
    // One EM step as a CUDA graph per theta-slot parity (single-GPU contexts): replayed instead of re-launching the
    // 6-8 small operations of a step, which is what bounds small problems (BASELINE config 1: N = 10k).
    cudaGraphExec_t step_graph[2] = {nullptr, nullptr};
    int64_t launches_per_step = 0;
    int plain_steps = 0;         // steps launched the ordinary way since creation (the first two size the scratch buffers)
    ReduceScratch reduce_scratch;   // owned here: the captured step graph has its address baked in

    double* means(int g) const { return gpus[g].params; }
    double* covs(int g) const { return gpus[g].params + d * k; }
    double* weights(int g) const { return covs(g) + static_cast<size_t>(k) * d * d; }
    double* inv_covs(int g) const { return weights(g) + k; }
    double* sqrt_dets(int g) const { return inv_covs(g) + static_cast<size_t>(k) * d * d; }
    size_t params_len() const { return static_cast<size_t>(d) * k + 2 * static_cast<size_t>(k) * d * d + 2 * k; }
};

namespace mlb {

static int pad_to(int v, const int* options, int n)
{
    for (int i = 0; i < n; ++i)
        if (v <= options[i]) return options[i];
    return 0;
}

static EmArgs base_args(const mlb_em* em, int g)
{
    const DataShard& sh = em->data->shards[g];
    const EmGpu& eg = em->gpus[g];
    EmArgs a{};
    a.x = sh.x;
    a.n_local = sh.n();
    a.d = em->d;
    a.k = em->k;
    a.shift = sh.shift;
    a.theta = eg.theta[em->cur];
    a.feat_m = eg.feat_m;
    a.partials = eg.partials;
    a.chunk = em->data->lay.chunk;
    a.n_chunks = static_cast<int>(sh.n_chunks());
    a.counter = eg.counter;
    return a;
}

static int launch_em(mlb_em* em, EmKernelFn fn, const EmArgs& a, int g, int grid)
{
    Gpu& gpu = em->ctx->gpus[g];
    MLB_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(unsigned), gpu.stream));
    if (a.n_chunks > 0) {
        const bool timed = fn == em->fn_step;
        if (timed) MLB_TRY(em->gpus[g].timer.begin(gpu.stream));
        fn<<<std::min(grid, a.n_chunks), em->DP <= 8 ? kSmallThreads : kEmThreads, em->smem_fused, gpu.stream>>>(a);
        MLB_CUDA(cudaGetLastError());
        if (timed) MLB_TRY(em->gpus[g].timer.end(gpu.stream));
        ++em->launches;
    }
    return MLB_OK;
}

static EmSplitArgs split_args(const mlb_em* em, int g, const double* theta)
{
    const DataShard& sh = em->data->shards[g];
    const EmGpu& eg = em->gpus[g];
    EmSplitArgs a{};
    a.x = sh.x;
    a.n_local = sh.n();
    a.d = em->d; a.k = em->k; a.DP = em->DP; a.KP = em->KP;
    a.shift = sh.shift;
    a.theta = theta;
    a.feat_e = eg.feat_e_off;
    a.feat_m = eg.feat_m;
    a.ne = em->NE; a.nm = em->NM;
    a.r = eg.r;
    a.partials = eg.partials;
    a.ll_tile = eg.ll_tile;
    a.sv = em->SV;
    a.chunk = em->data->lay.chunk;
    a.n_chunks = static_cast<int>(sh.n_chunks());
    a.counter = eg.counter;
    return a;
}

// Split path: E kernel (skipped when the responsibilities were supplied by the caller) then M kernel.
static int launch_split(mlb_em* em, int g, const double* theta, bool run_e, bool timed)
{
    Gpu& gpu = em->ctx->gpus[g];
    EmGpu& eg = em->gpus[g];
    const EmSplitArgs a = split_args(em, g, theta);
    if (a.n_chunks == 0) return MLB_OK;
    if (timed) MLB_TRY(eg.timer.begin(gpu.stream));
    if (run_e) {
        MLB_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(unsigned), gpu.stream));
        const long long e_items = static_cast<long long>(a.n_chunks) * (a.chunk / kSpTile);
        em->fn_split_e<<<static_cast<unsigned>(std::min<long long>(eg.grid_e, e_items)), kSpThreads, em->smem_split_e, gpu.stream>>>(a);
        MLB_CUDA(cudaGetLastError());
        ++em->launches;
    }
    const int ngroups = em->KP / (em->NT * 8), nslabs = (em->NM + 4 * em->MW - 1) / (4 * em->MW);
    const long long nitems = static_cast<long long>(a.n_chunks) * nslabs * ngroups;
    MLB_REQUIRE(nitems < (1ll << 31), "EM split path: too many work items");
    MLB_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(unsigned), gpu.stream));
    em->fn_split_m<<<static_cast<unsigned>(std::min<long long>(eg.grid_m, nitems)), kSpThreads, em->smem_split_m, gpu.stream>>>(a);
    MLB_CUDA(cudaGetLastError());
    ++em->launches;
    if (timed) MLB_TRY(eg.timer.end(gpu.stream));
    return MLB_OK;
}

// One pass over the local points with the E-step image `theta`: statistics into the chunk partials.
static int launch_pass(mlb_em* em, int g, const double* theta, bool timed)
{
    if (em->path == 2) return launch_split(em, g, theta, true, timed);
    EmArgs a = base_args(em, g);
    a.theta = theta;
    return launch_em(em, em->fn_step, a, g, em->gpus[g].grid);
}

// stats: 0 = parameters as they are (set_params), 1 = feature-path statistics, 2 = direct-path statistics
static EmFinalizeArgs finalize_args(const mlb_em* em, int g, int stats, int theta_slot, bool want_ll)
{
    const EmGpu& eg = em->gpus[g];
    EmFinalizeArgs f{};
    f.vsum = stats == 1 ? eg.vsum : nullptr;
    f.shift = em->data->shards[g].shift;
    f.d = em->d; f.k = em->k; f.DP = em->DP; f.KP = em->KP; f.SV = em->SV;
    f.n_total = em->data->lay.n_total;
    f.feat_m = eg.feat_m; f.feat_e = eg.feat_e;
    f.nm8 = em->NM * 8; f.ne = em->NE;
    f.means = em->means(g); f.covs = em->covs(g); f.weights = em->weights(g);
    f.inv_covs = em->inv_covs(g); f.sqrt_dets = em->sqrt_dets(g);
    f.theta_out = em->path ? eg.theta[theta_slot] : nullptr;
    if (em->dr.capable) {
        const EmDirectGpu& dg = em->dr.gpus[g];
        f.DPd = em->dr.DP; f.dSV = em->dr.SVd;
        f.dstats = stats == 2 ? dg.vsum : nullptr;
        f.dimg_out = dg.img;
        f.kappa_out = dg.kappa;
    }
    f.ll_ring = want_ll ? eg.ll : nullptr;
    f.ll_counter = eg.ll_counter;
    f.ll_ring_len = kLlRing;
    return f;
}

static size_t finalize_smem(const mlb_em* em, bool* p_in_smem)
{
    const size_t d = static_cast<size_t>(em->d);
    const size_t with_p = sizeof(double) * (2 * d * d + 3 * d), without = sizeof(double) * (d * d + 3 * d);
    const bool fits = with_p <= 200 * 1024;
    if (p_in_smem) *p_in_smem = fits;
    return fits ? with_p : without;
}

static int launch_finalize(mlb_em* em, int g, int stats, int theta_slot, bool want_ll)
{
    EmFinalizeArgs f = finalize_args(em, g, stats, theta_slot, want_ll);
    bool p_in_smem = true;
    const size_t smem = finalize_smem(em, &p_in_smem);
    f.p_in_smem = p_in_smem ? 1 : 0;
    em_finalize_kernel<<<em->path ? em->KP : em->k, 128, smem, em->ctx->gpus[g].stream>>>(f);
    MLB_CUDA(cudaGetLastError());
    ++em->launches;
    return MLB_OK;
}

// ---------------------------------------------------------------- direct path: buffers and launches

using EmDirectKernelFn = void (*)(EmDirectArgs);
static EmDirectKernelFn direct_e_kernel_for(int NB)
{
    return NB == 1 ? em_direct_e_kernel<1> : NB == 2 ? em_direct_e_kernel<2> : em_direct_e_kernel<0>;
}

// Super-chunks: every virtual shard's chunks are cut into at most kDrSuperPerVshard contiguous runs (a function of N only).
static void direct_layout(mlb_em* em, int vshard, std::vector<int64_t>& point_bounds)
{
    const Layout& lay = em->data->lay;
    const int64_t lo = lay.vshard_chunk[vshard], hi = lay.vshard_chunk[vshard + 1];
    const int64_t n = std::min<int64_t>(hi - lo, kDrSuperPerVshard);
    for (int64_t j = 0; j <= n; ++j) {
        if (n == 0) break;
        const int64_t chunk_idx = lo + (hi - lo) * j / n;
        point_bounds.push_back(std::min<int64_t>(chunk_idx * lay.chunk, lay.n_total));
    }
}

static int direct_prepare(mlb_em* em)
{
    EmDirect& dr = em->dr;
    if (dr.ready) return MLB_OK;
    mlb_ctx* ctx = em->ctx;
    const int vpg = ctx->vshards_per_gpu();
    std::vector<int2> tiles;
    for (int mt = 0; mt <= dr.NB; ++mt)
        for (int nt = mt; nt <= dr.NB; ++nt) tiles.push_back(make_int2(mt, nt));
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        EmDirectGpu& dg = dr.gpus[g];
        const DataShard& sh = em->data->shards[g];
        std::vector<long long> begins;
        for (int j = 0; j < vpg; ++j) {
            std::vector<int64_t> pb;
            direct_layout(em, gpu.rank * vpg + j, pb);
            // consecutive shards share a boundary: keep the first entry only for the first non-empty shard
            for (size_t i = begins.empty() ? 0 : 1; i < pb.size(); ++i) begins.push_back(static_cast<long long>(pb[i] - sh.begin));
        }
        if (begins.empty()) begins.push_back(0);
        dg.n_sc = static_cast<int>(begins.size()) - 1;
        const int64_t n = std::max<int64_t>(1, sh.n());
        MLB_CUDA(cudaMallocFromPoolAsync(&dg.r, sizeof(double) * n * dr.KPr, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dg.ll_tile, sizeof(double) * ((n + kDrTile - 1) / kDrTile), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dg.partials, sizeof(double) * std::max(1, dg.n_sc) * static_cast<size_t>(dr.SVd), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dg.vsum, sizeof(double) * kVirtualShards * static_cast<size_t>(dr.SVd), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(dg.vsum, 0, sizeof(double) * kVirtualShards * static_cast<size_t>(dr.SVd), gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dg.sc_begin, sizeof(long long) * begins.size(), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemcpyAsync(dg.sc_begin, begins.data(), sizeof(long long) * begins.size(), cudaMemcpyHostToDevice, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dg.tile_tab, sizeof(int2) * tiles.size(), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemcpyAsync(dg.tile_tab, tiles.data(), sizeof(int2) * tiles.size(), cudaMemcpyHostToDevice, gpu.stream));
        const auto e_kernel = direct_e_kernel_for(dr.NB);
        MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(e_kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(dr.smem_e)));
        MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(em_direct_m_kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(dr.smem_m)));
        int per_e = 0, per_m = 0, sms = 0;
        MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_e, reinterpret_cast<const void*>(e_kernel), kDrThreads, dr.smem_e));
        MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_m, reinterpret_cast<const void*>(em_direct_m_kernel), kDrThreads, dr.smem_m));
        MLB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, gpu.device));
        MLB_REQUIRE(per_e >= 1 && per_m >= 1, "EM direct kernels do not fit on an SM (D=%d, K=%d)", em->d, em->k);
        dg.grid_e = per_e * sms;
        dg.grid_m = per_m * sms;
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));   // `begins` and `tiles` are locals
        return MLB_OK;
    }));
    dr.ready = true;
    return MLB_OK;
}

static EmDirectArgs direct_args(const mlb_em* em, int g)
{
    const EmDirect& dr = em->dr;
    const EmDirectGpu& dg = dr.gpus[g];
    const DataShard& sh = em->data->shards[g];
    EmDirectArgs a{};
    a.x = sh.x; a.n_local = sh.n();
    a.d = em->d; a.k = em->k; a.DP = dr.DP; a.KPr = dr.KPr;
    a.shift = sh.shift;
    a.img = dg.img;
    a.r = dg.r; a.ll_tile = dg.ll_tile;
    a.counter = em->gpus[g].counter;
    a.cb = dr.cb;
    a.sc_begin = dg.sc_begin; a.n_sc = dg.n_sc;
    a.partials = dg.partials; a.svd = dr.SVd;
    a.cg = dr.cg; a.tiles_per_range = dr.tiles_per_range; a.n_ranges = dr.n_ranges;
    a.tile_tab = dg.tile_tab;
    return a;
}

static int launch_direct_e(mlb_em* em, int g, const EmDirectArgs& a)
{
    Gpu& gpu = em->ctx->gpus[g];
    const long long ntiles = (a.n_local + kDrTile - 1) / kDrTile;
    if (ntiles == 0) return MLB_OK;
    MLB_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(unsigned), gpu.stream));
    direct_e_kernel_for(em->dr.NB)<<<static_cast<unsigned>(std::min<long long>(em->dr.gpus[g].grid_e, ntiles)), kDrThreads, em->dr.smem_e, gpu.stream>>>(a);
    MLB_CUDA(cudaGetLastError());
    ++em->launches;
    return MLB_OK;
}

// The M kernel over the super-chunks (the E tiles' log-likelihood sums folded in when with_ll), then nothing else: the
// caller reduces, exchanges and refreshes.
static int launch_direct_m(mlb_em* em, int g, const EmDirectArgs& a, bool with_ll)
{
    Gpu& gpu = em->ctx->gpus[g];
    if (a.n_sc == 0) return MLB_OK;
    if (with_ll) {
        em_direct_ll_kernel<<<a.n_sc, 32, 0, gpu.stream>>>(a);
        MLB_CUDA(cudaGetLastError());
        ++em->launches;
    } else {
        // no E-step behind these statistics: the log-likelihood slots must still be defined
        for (int sc = 0; sc < a.n_sc; ++sc)
            MLB_CUDA(cudaMemsetAsync(a.partials + static_cast<size_t>(sc) * a.svd + static_cast<size_t>(em->k) * em->dr.L, 0, sizeof(double) * 8, gpu.stream));
    }
    const int ngroups = (a.k + a.cg - 1) / a.cg;
    const long long nitems = static_cast<long long>(a.n_sc) * ngroups * a.n_ranges;
    MLB_REQUIRE(nitems < (1ll << 31), "EM direct path: too many work items");
    MLB_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(unsigned), gpu.stream));
    em_direct_m_kernel<<<static_cast<unsigned>(std::min<long long>(em->dr.gpus[g].grid_m, nitems)), kDrThreads, em->dr.smem_m, gpu.stream>>>(a);
    MLB_CUDA(cudaGetLastError());
    ++em->launches;
    return MLB_OK;
}

static int direct_reduce(mlb_em* em)
{
    std::vector<double*> partials, vsum;
    for (EmDirectGpu& dg : em->dr.gpus) { partials.push_back(dg.partials); vsum.push_back(dg.vsum); }
    MLB_TRY(reduce_and_exchange_units(em->data, partials, vsum, em->dr.SVd, em->dr.scratch, em->dr.sc_bounds));
    em->launches += static_cast<int64_t>(em->ctx->gpus.size());
    return MLB_OK;
}

// One iteration on the direct kernels: E, M, reduction + exchange, parameter refresh into the other theta slot.
static int enqueue_step_direct(mlb_em* em)
{
    MLB_TRY(direct_prepare(em));
    mlb_ctx* ctx = em->ctx;
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        const EmDirectArgs a = direct_args(em, g);
        MLB_TRY(em->gpus[g].timer.begin(gpu.stream));
        MLB_TRY(launch_direct_e(em, g, a));
        MLB_TRY(launch_direct_m(em, g, a, true));
        MLB_TRY(em->gpus[g].timer.end(gpu.stream));
        return MLB_OK;
    }));
    MLB_TRY(direct_reduce(em));
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu&) -> int { return launch_finalize(em, g, 2, em->cur ^ 1, true); }));
    em->r_direct_valid = true;
    return MLB_OK;
}

// Chooses the path of the next step from kappa of the parameters just refreshed.  enqueue: the copy of kappa into the
// object's pinned buffer, ordered behind the refresh; finish: after the stream has been synchronised.
static int route_enqueue(mlb_em* em)
{
    if (!em->dr.capable) return MLB_OK;
    Gpu& gpu = em->ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    if (!em->kappa_host) MLB_CUDA(cudaMallocHost(&em->kappa_host, sizeof(double) * em->k));
    MLB_CUDA(cudaMemcpyAsync(em->kappa_host, em->dr.gpus[0].kappa, sizeof(double) * em->k, cudaMemcpyDeviceToHost, gpu.stream));
    return MLB_OK;
}

static void route_finish(mlb_em* em)
{
    em->kappa_max = 0.0;
    if (em->dr.capable && em->kappa_host)
        for (int i = 0; i < em->k; ++i) {
            const double v = em->kappa_host[i];
            if (v != v) em->kappa_max = std::numeric_limits<double>::infinity();   // NaN: a component has collapsed
            else if (v > em->kappa_max) em->kappa_max = v;
        }
    const bool direct = em->path == 0 || em->forced_path == 3 || (em->dr.capable && em->kappa_max > kKappaDirect);
    em->route = direct ? 3 : em->path;
}

static int update_route(mlb_em* em)
{
    MLB_TRY(route_enqueue(em));
    MLB_CUDA(cudaStreamSynchronize(em->ctx->gpus[0].stream));
    route_finish(em);
    return MLB_OK;
}

// E+M over all local points, statistics reduced and exchanged, parameters refreshed into the other theta slot.
static int enqueue_step_plain(mlb_em* em)
{
    mlb_ctx* ctx = em->ctx;
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu&) -> int {
        return launch_pass(em, g, em->gpus[g].theta[em->cur], true);
    }));
    std::vector<double*> partials, vsum;
    for (EmGpu& eg : em->gpus) { partials.push_back(eg.partials); vsum.push_back(eg.vsum); }
    MLB_TRY(reduce_and_exchange(em->data, partials, vsum, em->SV, em->reduce_scratch));
    em->launches += static_cast<int64_t>(ctx->gpus.size());
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu&) -> int {
        return launch_finalize(em, g, 1, em->cur ^ 1, true);
    }));
    em->r_direct_valid = false;
    return MLB_OK;
}

static int enqueue_step(mlb_em* em)
{
    mlb_ctx* ctx = em->ctx;
    if (em->route == 3) {
        MLB_TRY(enqueue_step_direct(em));
        em->cur ^= 1;
        em->last_path = 3;
        ++em->direct_steps;
        return MLB_OK;
    }
    em->last_path = em->path;
    // Graph replay: one local GPU, no collective in the step, no per-launch event timing, and the scratch buffers
    // already sized by two ordinary steps (nothing may allocate while a stream is being captured).
    const bool graphable = ctx->gpus.size() == 1 && ctx->world == 1 && !em->gpus[0].timer.enabled && em->plain_steps >= 2;
    if (!graphable) {
        MLB_TRY(enqueue_step_plain(em));
        ++em->plain_steps;
        em->cur ^= 1;
        return MLB_OK;
    }
    Gpu& gpu = ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    cudaGraphExec_t& exec = em->step_graph[em->cur];
    if (!exec) {
        const int64_t launches_before = em->launches;
        cudaGraph_t graph = nullptr;
        MLB_CUDA(cudaStreamBeginCapture(gpu.stream, cudaStreamCaptureModeThreadLocal));
        const int rc = enqueue_step_plain(em);
        const cudaError_t end = cudaStreamEndCapture(gpu.stream, &graph);
        if (rc != MLB_OK) {
            if (graph) cudaGraphDestroy(graph);
            return rc;
        }
        MLB_CUDA(end);
        em->launches_per_step = em->launches - launches_before;
        em->launches = launches_before;   // nothing ran yet: the capture only recorded the work
        const cudaError_t inst = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        MLB_CUDA(inst);
    }
    MLB_CUDA(cudaGraphLaunch(exec, gpu.stream));
    em->launches += em->launches_per_step;
    em->r_direct_valid = false;
    em->cur ^= 1;
    return MLB_OK;
}

// Start of a direct M-step that has no parameters behind it: every component's image says "mean = shift" (delta = 0,
// which is all the M kernel reads) and the means themselves are set to the shift.
__global__ void em_direct_origin_kernel(double* img, long long img_len, double* means, const double* shift, int d, int k)
{
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < img_len) img[i] = 0.0;
    if (i < static_cast<long long>(d) * k) means[i] = shift[i % d];
}

// maximisation_step on the direct kernels from the responsibilities in the direct R buffer.  from_origin: there are no
// parameters yet, so a first pass about the shift finds the means and a second pass about those means gives the
// covariances without cancellation (the reference makes the same two passes, EM.cpp:229 then :246-248); otherwise one
// pass about the current means.
static int direct_mstep_from_r(mlb_em* em, bool from_origin)
{
    mlb_ctx* ctx = em->ctx;
    for (int pass = 0; pass < (from_origin ? 2 : 1); ++pass) {
        MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
            if (pass == 0 && from_origin) {
                const long long len = static_cast<long long>(em->k) * em->dr.IMG;
                const long long total = std::max<long long>(len, static_cast<long long>(em->d) * em->k);
                em_direct_origin_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, gpu.stream>>>(em->dr.gpus[g].img, len, em->means(g), em->data->shards[g].shift, em->d, em->k);
                MLB_CUDA(cudaGetLastError());
                ++em->launches;
            }
            return launch_direct_m(em, g, direct_args(em, g), false);
        }));
        MLB_TRY(direct_reduce(em));
        MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu&) -> int { return launch_finalize(em, g, 2, em->cur, false); }));
    }
    return MLB_OK;
}

static int direct_import_r(mlb_em* em, std::vector<double*>& dev)
{
    return for_each_gpu(em->ctx, [&](int g, Gpu& gpu) -> int {
        const int64_t n = em->data->shards[g].n();
        if (n == 0) return MLB_OK;
        const long long total = static_cast<long long>(n) * em->dr.KPr;
        em_split_import_r_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, gpu.stream>>>(dev[g], n, n, em->k, em->dr.KPr, em->dr.gpus[g].r);
        MLB_CUDA(cudaGetLastError());
        ++em->launches;
        return MLB_OK;
    });
}

// maximisation_step from responsibilities already on the devices: dev[g] is column-major, local rows of GPU g, leading
// dimension max(1, n_local).  Frees the buffers.
static int mstep_from_device(mlb_em* em, std::vector<double*>& dev, int rc)
{
    mlb_ctx* ctx = em->ctx;
    auto body = [&]() -> int {
        const bool direct_only = em->path == 0 || em->forced_path == 3;
        if (!direct_only) {
            MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu&) -> int {
                const int64_t n = em->data->shards[g].n();
                if (em->path == 2) {
                    if (n == 0) return MLB_OK;
                    const long long total = static_cast<long long>(n) * em->KP;
                    em_split_import_r_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, ctx->gpus[g].stream>>>(dev[g], n, n, em->k, em->KP, em->gpus[g].r);
                    MLB_CUDA(cudaGetLastError());
                    ++em->launches;
                    return launch_split(em, g, em->gpus[g].theta[em->cur], false, false);
                }
                EmArgs a = base_args(em, g);
                a.r_in = dev[g];
                a.r_ld = std::max<int64_t>(1, n);  // device copy: local rows only
                return launch_em(em, em->fn_mstep, a, g, em->gpus[g].grid);
            }));
            std::vector<double*> partials, vsum;
            for (EmGpu& eg : em->gpus) { partials.push_back(eg.partials); vsum.push_back(eg.vsum); }
            MLB_TRY(reduce_and_exchange(em->data, partials, vsum, em->SV, em->reduce_scratch));
            em->launches += static_cast<int64_t>(ctx->gpus.size());
            MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu&) -> int { return launch_finalize(em, g, 1, em->cur, false); }));
            MLB_TRY(update_route(em));
            if (em->route != 3) return MLB_OK;
            // The components sit too far from the centre of the data for moments about the shift: once more about the
            // means just found.
        }
        MLB_TRY(direct_prepare(em));
        MLB_TRY(direct_import_r(em, dev));
        MLB_TRY(direct_mstep_from_r(em, direct_only));
        return update_route(em);
    };
    if (rc == MLB_OK) rc = body();
    // on every path: a pinned source of staged_h2d is still being read by the DMA engine until the stream is idle
    const int rc_sync = mlb_ctx_synchronize(ctx);
    if (rc == MLB_OK) rc = rc_sync;
    for (size_t g = 0; g < dev.size(); ++g)
        if (dev[g]) { cudaSetDevice(ctx->gpus[g].device); cudaFreeAsync(dev[g], ctx->gpus[g].stream); }
    if (rc == MLB_OK) { em->have_params = true; em->have_step = false; }
    return rc;
}

// calculate_sample_covariance (EM.cpp:265-272) on the direct kernels: the M kernel for ONE component with unit
// responsibilities about the shift (a private all-zero image: delta = 0), current parameters untouched.
static int direct_sample_covariance(mlb_em* em, double* cov_out)
{
    MLB_TRY(direct_prepare(em));
    mlb_ctx* ctx = em->ctx;
    EmDirect& dr = em->dr;
    const int d = em->d;
    std::vector<double*> tmp(ctx->gpus.size(), nullptr);
    int rc = for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        MLB_CUDA(cudaMallocFromPoolAsync(&tmp[g], sizeof(double) * dr.IMG, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(tmp[g], 0, sizeof(double) * dr.IMG, gpu.stream));
        EmDirectArgs a = direct_args(em, g);
        a.img = tmp[g];
        a.k = 1;
        a.unit_r = 1;
        return launch_direct_m(em, g, a, false);
    });
    if (rc == MLB_OK) rc = direct_reduce(em);
    std::vector<double> host(static_cast<size_t>(kVirtualShards) * dr.L);
    if (rc == MLB_OK) {
        Gpu& gpu0 = ctx->gpus[0];
        MLB_CUDA(cudaSetDevice(gpu0.device));
        MLB_CUDA(cudaMemcpy2DAsync(host.data(), sizeof(double) * dr.L, dr.gpus[0].vsum, sizeof(double) * dr.SVd, sizeof(double) * dr.L, kVirtualShards,
                                   cudaMemcpyDeviceToHost, gpu0.stream));
    }
    const int rc_sync = mlb_ctx_synchronize(ctx);
    for (size_t g = 0; g < tmp.size(); ++g)
        if (tmp[g]) { cudaSetDevice(ctx->gpus[g].device); cudaFreeAsync(tmp[g], ctx->gpus[g].stream); }
    MLB_TRY(rc);
    MLB_TRY(rc_sync);
    em->r_direct_valid = false;
    const int NBa = dr.NB + 1;
    auto stat = [&](int mt, int nt, int row, int col) { return tree8(host.data() + dr_tile_index(NBa, mt, nt) * 64 + row * 8 + col, dr.L); };
    const double count = stat(dr.NB, dr.NB, 0, 0);
    std::vector<double> m1(d);
    for (int a = 0; a < d; ++a) m1[a] = stat(a / 8, dr.NB, a % 8, 0);
    for (int a = 0; a < d; ++a)
        for (int b = a; b < d; ++b) {
            const double m2 = stat(a / 8, b / 8, a % 8, b % 8);
            const double cv = (m2 - m1[a] * m1[b] / count) / (count - 1.0);
            cov_out[a + static_cast<size_t>(b) * d] = cv;
            cov_out[b + static_cast<size_t>(a) * d] = cv;
        }
    return MLB_OK;
}

// One-hot responsibilities (Clustering.cpp:76,87) from labels: r[i + k * ld] = (labels[i] == k).
__global__ void em_onehot_kernel(const unsigned* __restrict__ labels, long long n, int k, double* __restrict__ r)
{
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned label = labels[i];
    for (int kk = 0; kk < k; ++kk) r[i + static_cast<long long>(kk) * n] = label == static_cast<unsigned>(kk) ? 1.0 : 0.0;
}

}  // namespace mlb

extern "C" {

int mlb_selftest_exp(const double* x, int64_t n, double* out)
{
    MLB_REQUIRE(x && out && n >= 0, "mlb_selftest_exp: bad argument");
    if (n == 0) return MLB_OK;
    MLB_CUDA(cudaSetDevice(0));
    double *dx = nullptr, *dy = nullptr;
    MLB_CUDA(cudaMalloc(&dx, sizeof(double) * n));
    MLB_CUDA(cudaMalloc(&dy, sizeof(double) * n));
    MLB_CUDA(cudaMemcpy(dx, x, sizeof(double) * n, cudaMemcpyHostToDevice));
    selftest_exp_kernel<<<static_cast<unsigned>((n + 127) / 128), 128>>>(dx, n, dy);
    MLB_CUDA(cudaGetLastError());
    MLB_CUDA(cudaMemcpy(out, dy, sizeof(double) * n, cudaMemcpyDeviceToHost));
    MLB_CUDA(cudaFree(dx));
    MLB_CUDA(cudaFree(dy));
    return MLB_OK;
}

int mlb_em_create(mlb_ctx* ctx, mlb_data* data, int k, mlb_em** out)
{
    MLB_ENTER(ctx);
    MLB_REQUIRE(ctx && data && out, "mlb_em_create: null argument");
    MLB_REQUIRE(data->ctx == ctx, "mlb_em_create: data belongs to another context");
    MLB_REQUIRE(k >= 1, "mlb_em_create: number of components must be positive");
    MLB_REQUIRE(data->d <= kDirectMaxDim, "mlb_em_create: D=%d not supported by this build (D <= %d)", data->d, kDirectMaxDim);
    static const int dps[] = {4, 8, 16}, kps[] = {8, 16, 32};
    const bool fused = data->d <= 16 && k <= 32;
    const bool split = !fused && data->d <= 64 && k <= 256;
    int DP = 0, KP = 0, NT = 0;
    if (fused) {
        DP = pad_to(data->d, dps, 3);
        KP = pad_to(k, kps, 3);
        NT = KP / 8;
    } else if (split) {
        // split path: D padded to a multiple of 4, components in groups of 16 (K <= 16), 32 (K <= 32) or 64
        DP = (data->d + 3) / 4 * 4;
        const int KG = k > 32 ? 64 : (k > 16 ? 32 : 16);
        KP = (k + KG - 1) / KG * KG;
        NT = KG / 8;
    }
    auto* em = new mlb_em;
    em->ctx = ctx; em->data = data; em->d = data->d; em->k = k;
    em->path = fused ? 1 : split ? 2 : 0;   // 0: only the direct kernels take this shape (D > 64 or K > 256)
    em->route = em->path ? em->path : 3;
    if (const char* env = std::getenv("MLB200_EM_PATH"))   // developer override: "direct" forces the direct kernels
        if (std::strcmp(env, "direct") == 0) em->forced_path = 3;
    if (em->path) {
        em->DP = DP; em->KP = KP; em->NT = NT; em->NE = em_ne(DP); em->NM = em_nm(DP); em->SV = em_sv(DP, KP);
    }
    if (fused) {
        em->fn_step = em_kernel_for<0>(DP, KP);
        em->fn_mstep = em_kernel_for<1>(DP, KP);
        em->fn_emit = em_kernel_for<2>(DP, KP);
        em->smem_fused = DP <= 8 ? em_small_smem_bytes(DP, KP) : em_smem_bytes(DP, KP);
    } else if (split) {
        em->fn_split_e = NT == 8 ? em_split_e_kernel<8> : NT == 4 ? em_split_e_kernel<4> : em_split_e_kernel<2>;
        // feature tiles per warp of the M kernel: the choice that wastes the fewest tile slots (ties: the larger)
        int best_waste = 1 << 30;
        for (int mw = 3; mw <= 5; ++mw) {
            const int slabs = (em->NM + 4 * mw - 1) / (4 * mw), waste = slabs * 4 * mw - em->NM;
            if (waste <= best_waste) { best_waste = waste; em->MW = mw; }
        }
        if (NT == 8) em->fn_split_m = em->MW == 3 ? em_split_m_kernel<8, 3> : em->MW == 4 ? em_split_m_kernel<8, 4> : em_split_m_kernel<8, 5>;
        else if (NT == 4) em->fn_split_m = em->MW == 3 ? em_split_m_kernel<4, 3> : em->MW == 4 ? em_split_m_kernel<4, 4> : em_split_m_kernel<4, 5>;
        else em->fn_split_m = em->MW == 3 ? em_split_m_kernel<2, 3> : em->MW == 4 ? em_split_m_kernel<2, 4> : em_split_m_kernel<2, 5>;
        em->smem_split_e = em_split_e_smem(NT, DP, KP);
        em->smem_split_m = em_split_m_smem(NT, DP);
    }
    if (em->path) {
        // E-step slots, in the order the kernel enumerates them (see em_ne above); (a, b) with a <= b.
        em->feat_e.assign(static_cast<size_t>(em->NE) * 4, make_int2(-1, -1));
        const int DQ = DP / 4, J0 = em_ne_offdiag(DP);
        auto put = [&](int j, int c, int a, int b) { em->feat_e[static_cast<size_t>(j) * 4 + c] = make_int2(std::min(a, b), std::max(a, b)); };
        for (int a = 0; a < DP - 4; ++a)
            for (int m = a / 4 + 1; m < DQ; ++m)
                for (int c = 0; c < 4; ++c) put(em_estep_offdiag(DP, a, m), c, a, 4 * m + c);
        for (int m = 0; m < DQ; ++m)
            for (int c = 0; c < 4; ++c) {
                put(J0 + m, c, 4 * m + c, 4 * m + c);
                put(J0 + DQ + m, c, 4 * m + c, 4 * m + ((c + 1) & 3));
            }
        for (int h = 0; h < (DQ + 1) / 2; ++h)
            for (int c = 0; c < 4; ++c) {
                const int mx = 2 * h + (c >> 1);
                if (mx < DQ) put(J0 + 2 * DQ + h, c, 4 * mx + c, 4 * mx + ((c + 2) & 3));
            }
        for (int m = 0; m < DQ; ++m)
            for (int c = 0; c < 4; ++c) em->feat_e[static_cast<size_t>(em->NE - DQ + m) * 4 + c] = make_int2(4 * m + c, DP);
        // M-step features as offsets into a Z row: [0,DP) coordinates, DP the constant 1, DP+1 a zero.
        em->feat_m.assign(static_cast<size_t>(em->NM) * 8, make_int2(DP + 1, DP + 1));
        size_t f = 0;
        em->feat_m[f++] = make_int2(DP, DP);
        for (int a = 0; a < DP; ++a) em->feat_m[f++] = make_int2(a, DP);
        for (int a = 0; a < DP; ++a)
            for (int b = a; b < DP; ++b) em->feat_m[f++] = make_int2(a, b);
    }
    if (fused && DP <= 8) {
        // em_small_kernel: the statistics rows are the E-step slots themselves, then the count row (em_small.cuh)
        for (size_t f = 0; f < em->feat_m.size(); ++f) {
            int2 ab = make_int2(DP + 1, DP + 1);
            if (f < em->feat_e.size() && em->feat_e[f].x >= 0) ab = em->feat_e[f];
            if (static_cast<int>(f) == em_small_count_slot(DP)) ab = make_int2(DP, DP);
            em->feat_m[f] = ab;
        }
    }
    {
        // direct kernels: shape constants (the large buffers are allocated when the path is first taken)
        EmDirect& dr = em->dr;
        dr.capable = true;
        dr.DP = (em->d + 7) / 8 * 8;
        dr.NB = dr.DP / 8;
        dr.KPr = (k + 7) / 8 * 8;
        dr.IMG = dr_img_len(dr.DP);
        dr.L = dr_stat_len(dr.DP);
        const long long svd = static_cast<long long>(k) * dr.L + 8;
        if (svd >= (1ll << 31)) { delete em; set_error("mlb_em_create: D=%d, K=%d: statistics vector too long", data->d, k); return MLB_EINVAL; }
        dr.SVd = static_cast<int>(svd);
        dr.cb = static_cast<int>(std::max<size_t>(1, std::min<size_t>(std::min(16, k), (12 * 1024) / (sizeof(double) * dr.IMG))));
        const int T = dr_tiles(dr.NB);
        if (T <= 4 * kDrSlots) {
            const int by_smem = static_cast<int>((96 * 1024) / (sizeof(double) * 2 * kDrSub * (dr.DP + 12))) - 1;
            dr.cg = std::max(1, std::min({16, k, 4 * kDrSlots / T, by_smem}));
            dr.tiles_per_range = T;
            dr.n_ranges = 1;
        } else {
            dr.cg = 1;
            dr.tiles_per_range = 4 * kDrSlots;
            dr.n_ranges = (T + 4 * kDrSlots - 1) / (4 * kDrSlots);
        }
        dr.smem_e = em_direct_e_smem(dr.DP, dr.cb);
        dr.smem_m = em_direct_m_smem(dr.DP, dr.cg, em->d);
        dr.sc_bounds[0] = 0;
        for (int v = 0; v < kVirtualShards; ++v)
            dr.sc_bounds[v + 1] = dr.sc_bounds[v] + std::min<int64_t>(data->lay.vshard_chunk[v + 1] - data->lay.vshard_chunk[v], kDrSuperPerVshard);
        dr.gpus.resize(ctx->gpus.size());
    }
    em->gpus.resize(ctx->gpus.size());
    int rc = for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        EmGpu& eg = em->gpus[g];
        EmDirectGpu& dg = em->dr.gpus[g];
        const DataShard& sh = data->shards[g];
        MLB_CUDA(cudaMallocFromPoolAsync(&eg.params, sizeof(double) * em->params_len(), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&eg.ll, sizeof(double) * kLlRing, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&eg.ll_counter, sizeof(unsigned long long), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(eg.ll_counter, 0, sizeof(unsigned long long), gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&eg.counter, sizeof(unsigned), gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dg.img, sizeof(double) * static_cast<size_t>(k) * em->dr.IMG, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dg.kappa, sizeof(double) * k, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMemsetAsync(dg.kappa, 0, sizeof(double) * k, gpu.stream));
        {
            const size_t fin_smem = finalize_smem(em, nullptr);
            if (fin_smem > 48 * 1024)
                MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(em_finalize_kernel), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(fin_smem)));
        }
        int sms = 0;
        MLB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, gpu.device));
        if (em->path) {
            const size_t theta_len = static_cast<size_t>(em_theta_len(DP, KP));
            MLB_CUDA(cudaMallocFromPoolAsync(&eg.theta[0], sizeof(double) * theta_len, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&eg.theta[1], sizeof(double) * theta_len, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&eg.partials, sizeof(double) * std::max<int64_t>(1, sh.n_chunks()) * em->SV, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&eg.vsum, sizeof(double) * kVirtualShards * em->SV, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&eg.feat_m, sizeof(int2) * em->feat_m.size(), gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&eg.feat_e, sizeof(int2) * em->feat_e.size(), gpu.pool, gpu.stream));
            MLB_CUDA(cudaMemsetAsync(eg.vsum, 0, sizeof(double) * kVirtualShards * em->SV, gpu.stream));
            MLB_CUDA(cudaMemcpyAsync(eg.feat_m, em->feat_m.data(), sizeof(int2) * em->feat_m.size(), cudaMemcpyHostToDevice, gpu.stream));
            MLB_CUDA(cudaMemcpyAsync(eg.feat_e, em->feat_e.data(), sizeof(int2) * em->feat_e.size(), cudaMemcpyHostToDevice, gpu.stream));
        }
        if (em->path == 1) {
            const size_t smem = em->smem_fused;
            for (EmKernelFn fn : {em->fn_step, em->fn_mstep, em->fn_emit})
                MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
            int per_sm = 0;
            MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void*>(em->fn_step), em->DP <= 8 ? kSmallThreads : kEmThreads, smem));
            MLB_REQUIRE(per_sm >= 1, "mlb_em_create: EM kernel does not fit on an SM");
            eg.grid = per_sm * sms;
        } else if (em->path == 2) {
            std::vector<int2> off(em->feat_e.size());
            for (size_t i = 0; i < off.size(); ++i) off[i] = em->feat_e[i].x < 0 ? make_int2(DP + 1, DP + 1) : em->feat_e[i];
            MLB_CUDA(cudaMallocFromPoolAsync(&eg.feat_e_off, sizeof(int2) * off.size(), gpu.pool, gpu.stream));
            MLB_CUDA(cudaMemcpyAsync(eg.feat_e_off, off.data(), sizeof(int2) * off.size(), cudaMemcpyHostToDevice, gpu.stream));
            MLB_CUDA(cudaStreamSynchronize(gpu.stream));   // `off` is a local
            MLB_CUDA(cudaMallocFromPoolAsync(&eg.r, sizeof(double) * std::max<int64_t>(1, sh.n()) * KP, gpu.pool, gpu.stream));
            {
                const size_t n_tiles = static_cast<size_t>(std::max<int64_t>(1, sh.n_chunks())) * (data->lay.chunk / kSpTile);
                MLB_CUDA(cudaMallocFromPoolAsync(&eg.ll_tile, sizeof(double) * n_tiles, gpu.pool, gpu.stream));
                MLB_CUDA(cudaMemsetAsync(eg.ll_tile, 0, sizeof(double) * n_tiles, gpu.stream));
            }
            MLB_CUDA(cudaMemsetAsync(eg.partials, 0, sizeof(double) * std::max<int64_t>(1, sh.n_chunks()) * em->SV, gpu.stream));
            MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(em->fn_split_e), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(em->smem_split_e)));
            MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(em->fn_split_m), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(em->smem_split_m)));
            int per_e = 0, per_m = 0;
            MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_e, reinterpret_cast<const void*>(em->fn_split_e), kSpThreads, em->smem_split_e));
            MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_m, reinterpret_cast<const void*>(em->fn_split_m), kSpThreads, em->smem_split_m));
            MLB_REQUIRE(per_e >= 1 && per_m >= 1, "mlb_em_create: EM kernels do not fit on an SM (D=%d, K=%d)", em->d, em->k);
            eg.grid_e = per_e * sms;
            eg.grid_m = per_m * sms;
        }
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        return MLB_OK;
    });
    if (rc != MLB_OK) { mlb_em_destroy(em); return rc; }
    *out = em;
    return MLB_OK;
}

int mlb_em_destroy(mlb_em* em)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    if (!em) return MLB_OK;
    for (cudaGraphExec_t& ge : em->step_graph)
        if (ge) { cudaGraphExecDestroy(ge); ge = nullptr; }
    for (size_t g = 0; g < em->gpus.size(); ++g) {
        cudaSetDevice(em->ctx->gpus[g].device);
        cudaStreamSynchronize(em->ctx->gpus[g].stream);
        EmGpu& eg = em->gpus[g];
        eg.timer.destroy();
        for (void* ptr : {static_cast<void*>(eg.theta[0]), static_cast<void*>(eg.theta[1]), static_cast<void*>(eg.params),
                          static_cast<void*>(eg.partials), static_cast<void*>(eg.vsum), static_cast<void*>(eg.ll), static_cast<void*>(eg.ll_counter),
                          static_cast<void*>(eg.feat_m), static_cast<void*>(eg.feat_e), static_cast<void*>(eg.counter),
                          static_cast<void*>(eg.stage), static_cast<void*>(eg.stage_labels), static_cast<void*>(eg.r), static_cast<void*>(eg.ll_tile),
                          static_cast<void*>(eg.feat_e_off)})
            if (ptr) cudaFreeAsync(ptr, em->ctx->gpus[g].stream);
        if (g < em->dr.gpus.size()) {
            EmDirectGpu& dg = em->dr.gpus[g];
            for (void* ptr : {static_cast<void*>(dg.img), static_cast<void*>(dg.kappa), static_cast<void*>(dg.r), static_cast<void*>(dg.ll_tile),
                              static_cast<void*>(dg.partials), static_cast<void*>(dg.vsum), static_cast<void*>(dg.sc_begin), static_cast<void*>(dg.tile_tab)})
                if (ptr) cudaFreeAsync(ptr, em->ctx->gpus[g].stream);
        }
    }
    em->reduce_scratch.release(em->ctx);
    em->dr.scratch.release(em->ctx);
    if (em->kappa_host) cudaFreeHost(em->kappa_host);
    delete em;
    return MLB_OK;
}

int mlb_em_set_params(mlb_em* em, const double* means, const double* covariances, const double* weights)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em && means && covariances && weights, "mlb_em_set_params: null argument");
    const size_t dk = static_cast<size_t>(em->d) * em->k, kdd = static_cast<size_t>(em->k) * em->d * em->d;
    MLB_TRY(for_each_gpu(em->ctx, [&](int g, Gpu& gpu) -> int {
        MLB_CUDA(cudaMemcpyAsync(em->means(g), means, sizeof(double) * dk, cudaMemcpyHostToDevice, gpu.stream));
        MLB_CUDA(cudaMemcpyAsync(em->covs(g), covariances, sizeof(double) * kdd, cudaMemcpyHostToDevice, gpu.stream));
        MLB_CUDA(cudaMemcpyAsync(em->weights(g), weights, sizeof(double) * em->k, cudaMemcpyHostToDevice, gpu.stream));
        MLB_TRY(launch_finalize(em, g, 0, em->cur, false));
        MLB_CUDA(cudaStreamSynchronize(gpu.stream));  // the host buffers may go away
        return MLB_OK;
    }));
    MLB_TRY(update_route(em));
    em->have_params = true;
    em->have_step = false;
    return MLB_OK;
}

int mlb_em_run_steps(mlb_em* em, int steps, double* log_likelihoods)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em && steps >= 0, "mlb_em_run_steps: bad argument");
    MLB_REQUIRE(steps <= kLlRing, "mlb_em_run_steps: at most %d steps per call", kLlRing);
    if (!em->have_params) { set_error("mlb_em_run_steps: parameters not set"); return MLB_ESTATE; }
    const int64_t first = em->steps_done;
    Gpu& gpu0 = em->ctx->gpus[0];
    for (int s = 0; s < steps; ++s) {
        MLB_TRY(enqueue_step(em));
        ++em->steps_done;
        // The path of the next step depends on the parameters this one produced: kappa comes back with every step (one
        // small copy; the last step's rides on the synchronisation the call ends with anyway).
        MLB_TRY(route_enqueue(em));
        if (s + 1 < steps) {
            MLB_CUDA(cudaStreamSynchronize(gpu0.stream));
            route_finish(em);
        }
    }
    if (steps > 0) em->have_step = true;
    if (log_likelihoods) {
        MLB_CUDA(cudaSetDevice(gpu0.device));
        for (int s = 0; s < steps; ++s)
            MLB_CUDA(cudaMemcpyAsync(log_likelihoods + s, em->gpus[0].ll + (first + s) % kLlRing, sizeof(double), cudaMemcpyDeviceToHost, gpu0.stream));
    }
    MLB_TRY(mlb_ctx_synchronize(em->ctx));
    if (steps > 0) route_finish(em);
    return MLB_OK;
}

int mlb_em_step(mlb_em* em, double* log_likelihood)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em && log_likelihood, "mlb_em_step: null argument");
    return mlb_em_run_steps(em, 1, log_likelihood);
}

int mlb_em_force_path(mlb_em* em, int path)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em, "mlb_em_force_path: null argument");
    MLB_REQUIRE(path == 0 || path == 3, "mlb_em_force_path: path must be 0 (automatic) or 3 (direct-difference kernels)");
    em->forced_path = path;
    if (em->have_params) MLB_TRY(update_route(em));
    else em->route = (path == 3 || em->path == 0) ? 3 : em->path;
    return MLB_OK;
}

int mlb_em_conditioning(mlb_em* em, double* kappa_max, int* next_path)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em, "mlb_em_conditioning: null argument");
    if (kappa_max) *kappa_max = em->kappa_max;
    if (next_path) *next_path = em->route;
    return MLB_OK;
}

int mlb_em_get_params(mlb_em* em, double* means, double* covariances, double* weights)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em, "mlb_em_get_params: null argument");
    if (!em->have_params) { set_error("mlb_em_get_params: parameters not set"); return MLB_ESTATE; }
    Gpu& gpu = em->ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    if (means) MLB_CUDA(cudaMemcpyAsync(means, em->means(0), sizeof(double) * em->d * em->k, cudaMemcpyDeviceToHost, gpu.stream));
    if (covariances) MLB_CUDA(cudaMemcpyAsync(covariances, em->covs(0), sizeof(double) * em->k * em->d * em->d, cudaMemcpyDeviceToHost, gpu.stream));
    if (weights) MLB_CUDA(cudaMemcpyAsync(weights, em->weights(0), sizeof(double) * em->k, cudaMemcpyDeviceToHost, gpu.stream));
    MLB_CUDA(cudaStreamSynchronize(gpu.stream));
    return MLB_OK;
}

int mlb_em_get_precisions(mlb_em* em, double* inverse_covariances, double* sqrt_determinants)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em, "mlb_em_get_precisions: null argument");
    if (!em->have_params) { set_error("mlb_em_get_precisions: parameters not set"); return MLB_ESTATE; }
    Gpu& gpu = em->ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu.device));
    if (inverse_covariances)
        MLB_CUDA(cudaMemcpyAsync(inverse_covariances, em->inv_covs(0), sizeof(double) * em->k * em->d * em->d, cudaMemcpyDeviceToHost, gpu.stream));
    if (sqrt_determinants) MLB_CUDA(cudaMemcpyAsync(sqrt_determinants, em->sqrt_dets(0), sizeof(double) * em->k, cudaMemcpyDeviceToHost, gpu.stream));
    MLB_CUDA(cudaStreamSynchronize(gpu.stream));
    return MLB_OK;
}

int mlb_em_sample_covariance(mlb_em* em, double* cov_out)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em && cov_out, "mlb_em_sample_covariance: null argument");
    if (em->path == 0 || em->forced_path == 3) return direct_sample_covariance(em, cov_out);
    // A one-component M-step with unit responsibilities: theta = 0 for component 0, -inf constants elsewhere.
    // Uses the spare theta slot and leaves the current parameters untouched.  On the fused path the pass runs the
    // 8-component instantiation of the step kernel (a quarter of the tensor-pipe work of a K = 32 step); the chunk
    // partials, the reduction and the exchange are the usual ones with the shorter statistics vector.
    const int d = em->d, DP = em->DP;
    const bool narrow = em->path == 1 && em->KP > 8;
    const int KP = narrow ? 8 : em->KP, SV = narrow ? em_sv(DP, 8) : em->SV;
    std::vector<double> theta(em_theta_len(DP, KP), 0.0);
    for (int kk = 1; kk < KP; ++kk) theta[static_cast<size_t>(em->NE) * (KP / 8) * 32 + kk] = -std::numeric_limits<double>::infinity();
    MLB_TRY(for_each_gpu(em->ctx, [&](int g, Gpu& gpu) -> int {
        MLB_CUDA(cudaMemcpyAsync(em->gpus[g].theta[em->cur ^ 1], theta.data(), sizeof(double) * theta.size(), cudaMemcpyHostToDevice, gpu.stream));
        if (!narrow) return launch_pass(em, g, em->gpus[g].theta[em->cur ^ 1], false);
        const EmKernelFn fn = em_kernel_for<0>(DP, 8);
        const size_t smem = DP <= 8 ? em_small_smem_bytes(DP, 8) : em_smem_bytes(DP, 8);
        MLB_CUDA(cudaFuncSetAttribute(reinterpret_cast<const void*>(fn), cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
        int per_sm = 0, sms = 0;
        MLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, reinterpret_cast<const void*>(fn), em->DP <= 8 ? kSmallThreads : kEmThreads, smem));
        MLB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, gpu.device));
        MLB_REQUIRE(per_sm >= 1, "mlb_em_sample_covariance: kernel does not fit on an SM");
        EmArgs a = base_args(em, g);
        a.theta = em->gpus[g].theta[em->cur ^ 1];
        a.k = 1;
        MLB_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(unsigned), gpu.stream));
        if (a.n_chunks > 0) {
            fn<<<std::min(per_sm * sms, a.n_chunks), em->DP <= 8 ? kSmallThreads : kEmThreads, smem, gpu.stream>>>(a);
            MLB_CUDA(cudaGetLastError());
            ++em->launches;
        }
        return MLB_OK;
    }));
    if (em->path == 2) em->have_step = false;   // the pass overwrote the stored responsibilities
    std::vector<double*> partials, vsum;
    for (EmGpu& eg : em->gpus) { partials.push_back(eg.partials); vsum.push_back(eg.vsum); }
    MLB_TRY(reduce_and_exchange(em->data, partials, vsum, SV, em->reduce_scratch));
    em->launches += static_cast<int64_t>(em->ctx->gpus.size());
    std::vector<double> host(static_cast<size_t>(kVirtualShards) * SV);
    Gpu& gpu0 = em->ctx->gpus[0];
    MLB_CUDA(cudaSetDevice(gpu0.device));
    MLB_CUDA(cudaMemcpyAsync(host.data(), em->gpus[0].vsum, sizeof(double) * host.size(), cudaMemcpyDeviceToHost, gpu0.stream));
    MLB_TRY(mlb_ctx_synchronize(em->ctx));
    double count = 0;
    std::vector<double> m1(d, 0.0), m2(static_cast<size_t>(d) * d, 0.0);
    for (size_t f = 0; f < em->feat_m.size(); ++f) {
        const int2 ab = em->feat_m[f];
        const double val = tree8(host.data() + f * KP, SV);
        if (ab.x == DP && ab.y == DP) count = val;
        else if (ab.y == DP && ab.x < d) m1[ab.x] = val;
        else if (ab.x < d && ab.y < d) { m2[ab.x + static_cast<size_t>(ab.y) * d] = val; m2[ab.y + static_cast<size_t>(ab.x) * d] = val; }
    }
    // unbiased covariance (EM.cpp:265-272): (sum z z^T - N dbar dbar^T) / (N - 1), z = x - c, dbar = mean(z) ~ 0
    for (int a = 0; a < d; ++a)
        for (int b = 0; b < d; ++b)
            cov_out[a + static_cast<size_t>(b) * d] = (m2[a + static_cast<size_t>(b) * d] - m1[a] * m1[b] / count) / (count - 1.0);
    return MLB_OK;
}

int mlb_em_mstep_from_responsibilities(mlb_em* em, const double* resp, int64_t ld)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em && resp, "mlb_em_mstep_from_responsibilities: null argument");
    mlb_ctx* ctx = em->ctx;
    const int64_t host_begin = ctx->rank_mode ? em->data->shards[0].begin : 0;
    std::vector<double*> dev(ctx->gpus.size(), nullptr);
    const int rc = for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        const DataShard& sh = em->data->shards[g];
        const int64_t n = std::max<int64_t>(1, sh.n());
        MLB_CUDA(cudaMallocFromPoolAsync(&dev[g], sizeof(double) * n * em->k, gpu.pool, gpu.stream));
        if (sh.n() > 0)
            MLB_TRY(staged_h2d(gpu, dev[g], resp + (sh.begin - host_begin), static_cast<size_t>(em->k), sizeof(double) * sh.n(), sizeof(double) * ld));
        return MLB_OK;
    });
    return mstep_from_device(em, dev, rc);
}

int mlb_em_mstep_from_labels(mlb_em* em, const unsigned int* labels)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em && labels, "mlb_em_mstep_from_labels: null argument");
    mlb_ctx* ctx = em->ctx;
    const int64_t host_begin = ctx->rank_mode ? em->data->shards[0].begin : 0;
    {
        // a label outside [0, K) would silently drop its point from every component
        int64_t n_held = 0;
        for (const DataShard& sh : em->data->shards) n_held += sh.n();
        for (int64_t i = 0; i < n_held; ++i)
            MLB_REQUIRE(labels[i] < static_cast<unsigned>(em->k), "mlb_em_mstep_from_labels: label %u of point %lld out of range", labels[i], static_cast<long long>(i + host_begin));
    }
    std::vector<double*> dev(ctx->gpus.size(), nullptr);
    std::vector<unsigned*> dev_labels(ctx->gpus.size(), nullptr);
    const int rc = for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        const DataShard& sh = em->data->shards[g];
        const int64_t n = std::max<int64_t>(1, sh.n());
        MLB_CUDA(cudaMallocFromPoolAsync(&dev[g], sizeof(double) * n * em->k, gpu.pool, gpu.stream));
        MLB_CUDA(cudaMallocFromPoolAsync(&dev_labels[g], sizeof(unsigned) * n, gpu.pool, gpu.stream));
        if (sh.n() > 0) {
            MLB_TRY(staged_h2d(gpu, dev_labels[g], labels + (sh.begin - host_begin), 1, sizeof(unsigned) * sh.n(), sizeof(unsigned) * sh.n()));
            em_onehot_kernel<<<static_cast<unsigned>((sh.n() + 255) / 256), 256, 0, gpu.stream>>>(dev_labels[g], sh.n(), em->k, dev[g]);
            MLB_CUDA(cudaGetLastError());
            ++em->launches;
        }
        return MLB_OK;
    });
    for (size_t g = 0; g < dev_labels.size(); ++g)
        if (dev_labels[g]) { cudaSetDevice(ctx->gpus[g].device); cudaFreeAsync(dev_labels[g], ctx->gpus[g].stream); }
    return mstep_from_device(em, dev, rc);
}

int mlb_em_emit_range(mlb_em* em, int64_t begin, int64_t count, double* resp_out, int64_t ld, unsigned int* labels_out)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em, "mlb_em_emit_range: null argument");
    MLB_REQUIRE(begin >= 0 && count >= 0 && begin + count <= em->data->lay.n_total, "mlb_em_emit_range: range out of bounds");
    if (!em->have_step) { set_error("mlb_em_emit: no step has been run"); return MLB_ESTATE; }
    if (em->last_path == 3 && !em->r_direct_valid) { set_error("mlb_em_emit: the responsibilities of the last step have been overwritten"); return MLB_ESTATE; }
    if ((!resp_out && !labels_out) || count == 0) return MLB_OK;
    MLB_REQUIRE(!resp_out || ld >= count, "mlb_em_emit_range: leading dimension smaller than the row count");
    mlb_ctx* ctx = em->ctx;
    int64_t covered = 0;
    for (const DataShard& sh : em->data->shards) covered += std::max<int64_t>(0, std::min(begin + count, sh.end) - std::max(begin, sh.begin));
    MLB_REQUIRE(covered == count, "mlb_em_emit_range: range is not held by this context");
    // Stage by stage: kStagePoints points per GPU at a time through a device buffer.
    MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
        EmGpu& eg = em->gpus[g];
        if (resp_out && !eg.stage) MLB_CUDA(cudaMallocFromPoolAsync(&eg.stage, sizeof(double) * kStagePoints * em->k, gpu.pool, gpu.stream));
        if (labels_out && !eg.stage_labels) MLB_CUDA(cudaMallocFromPoolAsync(&eg.stage_labels, sizeof(unsigned) * kStagePoints, gpu.pool, gpu.stream));
        return MLB_OK;
    }));
    for (int64_t off = 0;; off += kStagePoints) {
        bool any = false;
        MLB_TRY(for_each_gpu(ctx, [&](int g, Gpu& gpu) -> int {
            const DataShard& sh = em->data->shards[g];
            const int64_t lo = std::max(begin, sh.begin) + off, hi = std::min(begin + count, sh.end);
            const int64_t n = std::min<int64_t>(kStagePoints, hi - lo);
            if (n <= 0) return MLB_OK;
            any = true;
            EmGpu& eg = em->gpus[g];
            const int64_t row = lo - begin;
            if (em->last_path == 3) {
                // direct kernels: the responsibilities of the last E-step are resident in the direct R buffer
                EmSplitArgs a{};
                a.k = em->k; a.KP = em->dr.KPr; a.r = em->dr.gpus[g].r;
                a.range_begin = lo - sh.begin;
                a.range_count = n;
                a.r_out = resp_out ? eg.stage : nullptr;
                a.r_out_ld = kStagePoints;
                a.labels_out = labels_out ? eg.stage_labels : nullptr;
                em_split_emit_kernel<<<static_cast<unsigned>((n + 31) / 32), 256, 0, gpu.stream>>>(a);
                MLB_CUDA(cudaGetLastError());
                ++em->launches;
            } else if (em->path == 2) {
                // the responsibilities of the last E-step are resident: transpose them out, argmax for the labels
                EmSplitArgs a = split_args(em, g, nullptr);
                a.range_begin = lo - sh.begin;
                a.range_count = n;
                a.r_out = resp_out ? eg.stage : nullptr;
                a.r_out_ld = kStagePoints;
                a.labels_out = labels_out ? eg.stage_labels : nullptr;
                em_split_emit_kernel<<<static_cast<unsigned>((n + 31) / 32), 256, 0, gpu.stream>>>(a);
                MLB_CUDA(cudaGetLastError());
                ++em->launches;
            } else {
            EmArgs a = base_args(em, g);
            a.theta = eg.theta[em->cur ^ 1];  // theta_t of the last step
            a.chunk = kTile;
            a.n_chunks = static_cast<int>((n + kTile - 1) / kTile);
            a.range_begin = lo - sh.begin;
            a.range_count = n;
            a.r_out = resp_out ? eg.stage : nullptr;
            a.r_out_ld = kStagePoints;
            a.labels_out = labels_out ? eg.stage_labels : nullptr;
            MLB_TRY(launch_em(em, em->fn_emit, a, g, 8 * kSmCount));
            }
            if (resp_out)
                MLB_TRY(staged_d2h_2d(gpu, resp_out + row, sizeof(double) * ld, eg.stage, sizeof(double) * kStagePoints, static_cast<size_t>(em->k), sizeof(double) * n));
            if (labels_out) MLB_TRY(staged_d2h(gpu, labels_out + row, eg.stage_labels, sizeof(unsigned) * n));
            return MLB_OK;
        }));
        MLB_TRY(mlb_ctx_synchronize(ctx));
        if (!any) break;
    }
    return MLB_OK;
}

int mlb_em_emit(mlb_em* em, double* resp_out, int64_t ld, unsigned int* labels_out)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em, "mlb_em_emit: null argument");
    const std::vector<DataShard>& shards = em->data->shards;
    return mlb_em_emit_range(em, shards.front().begin, shards.back().end - shards.front().begin, resp_out, ld, labels_out);
}

int mlb_em_predict(mlb_em* em, const double* x, int64_t m, int64_t ld_x, double* resp_out, int64_t ld_out, unsigned int* labels_out)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em && x, "mlb_em_predict: null argument");
    MLB_REQUIRE(m >= 0 && ld_x >= em->d, "mlb_em_predict: bad shape (m=%lld, ld_x=%lld, D=%d)", static_cast<long long>(m), static_cast<long long>(ld_x), em->d);
    MLB_REQUIRE(!resp_out || ld_out >= m, "mlb_em_predict: leading dimension smaller than the row count");
    if (!em->have_params) { set_error("mlb_em_predict: parameters not set"); return MLB_ESTATE; }
    if (m == 0 || (!resp_out && !labels_out)) return MLB_OK;
    mlb_ctx* ctx = em->ctx;
    Gpu& gpu = ctx->gpus[0];
    EmGpu& eg = em->gpus[0];
    const int d = em->d;
    MLB_CUDA(cudaSetDevice(gpu.device));
    if (resp_out && !eg.stage) MLB_CUDA(cudaMallocFromPoolAsync(&eg.stage, sizeof(double) * kStagePoints * em->k, gpu.pool, gpu.stream));
    if (labels_out && !eg.stage_labels) MLB_CUDA(cudaMallocFromPoolAsync(&eg.stage_labels, sizeof(unsigned) * kStagePoints, gpu.pool, gpu.stream));
    const int64_t cap = std::min<int64_t>(m, kStagePoints);
    double *xd = nullptr, *r_tmp = nullptr, *ll_tmp = nullptr;
    MLB_CUDA(cudaMallocFromPoolAsync(&xd, sizeof(double) * cap * d, gpu.pool, gpu.stream));
    int rc = MLB_OK;
    const bool direct = em->route == 3;
    auto body = [&]() -> int {
        if (direct) {
            MLB_TRY(direct_prepare(em));
            MLB_CUDA(cudaMallocFromPoolAsync(&r_tmp, sizeof(double) * cap * em->dr.KPr, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&ll_tmp, sizeof(double) * ((cap + kDrTile - 1) / kDrTile), gpu.pool, gpu.stream));
        } else if (em->path == 2) {
            MLB_CUDA(cudaMallocFromPoolAsync(&r_tmp, sizeof(double) * cap * em->KP, gpu.pool, gpu.stream));
            MLB_CUDA(cudaMallocFromPoolAsync(&ll_tmp, sizeof(double) * ((cap + 127) / 128) * 2, gpu.pool, gpu.stream));
        }
        for (int64_t off = 0; off < m; off += kStagePoints) {
            const int64_t n = std::min<int64_t>(kStagePoints, m - off);
            const double* src = x + off * ld_x;
            MLB_TRY(staged_h2d(gpu, xd, src, static_cast<size_t>(n), sizeof(double) * d, sizeof(double) * ld_x));
            if (direct) {
                // direct E kernel on the staged points with the current images, then the transposing emit kernel
                EmDirectArgs a = direct_args(em, 0);
                a.x = xd;
                a.n_local = n;
                a.r = r_tmp;
                a.ll_tile = ll_tmp;
                MLB_TRY(launch_direct_e(em, 0, a));
                EmSplitArgs e{};
                e.k = em->k; e.KP = em->dr.KPr; e.r = r_tmp;
                e.range_begin = 0;
                e.range_count = n;
                e.r_out = resp_out ? eg.stage : nullptr;
                e.r_out_ld = kStagePoints;
                e.labels_out = labels_out ? eg.stage_labels : nullptr;
                em_split_emit_kernel<<<static_cast<unsigned>((n + 31) / 32), 256, 0, gpu.stream>>>(e);
                MLB_CUDA(cudaGetLastError());
                ++em->launches;
            } else if (em->path == 2) {
                // E kernel on the staged points (responsibilities into r_tmp), then the transposing emit kernel
                EmSplitArgs a = split_args(em, 0, eg.theta[em->cur]);
                a.x = xd;
                a.n_local = n;
                a.chunk = 128;
                a.n_chunks = static_cast<int>((n + 127) / 128);
                a.r = r_tmp;
                a.ll_tile = ll_tmp;
                MLB_CUDA(cudaMemsetAsync(a.counter, 0, sizeof(unsigned), gpu.stream));
                const long long e_items = static_cast<long long>(a.n_chunks) * (a.chunk / kSpTile);
                em->fn_split_e<<<static_cast<unsigned>(std::min<long long>(eg.grid_e, e_items)), kSpThreads, em->smem_split_e, gpu.stream>>>(a);
                MLB_CUDA(cudaGetLastError());
                a.range_begin = 0;
                a.range_count = n;
                a.r_out = resp_out ? eg.stage : nullptr;
                a.r_out_ld = kStagePoints;
                a.labels_out = labels_out ? eg.stage_labels : nullptr;
                em_split_emit_kernel<<<static_cast<unsigned>((n + 31) / 32), 256, 0, gpu.stream>>>(a);
                MLB_CUDA(cudaGetLastError());
                em->launches += 2;
            } else {
                EmArgs a = base_args(em, 0);
                a.x = xd;
                a.n_local = n;
                a.theta = eg.theta[em->cur];   // the current parameters (EM.cpp:176-188 uses the post-fit ones)
                a.chunk = kTile;
                a.n_chunks = static_cast<int>((n + kTile - 1) / kTile);
                a.range_begin = 0;
                a.range_count = n;
                a.r_out = resp_out ? eg.stage : nullptr;
                a.r_out_ld = kStagePoints;
                a.labels_out = labels_out ? eg.stage_labels : nullptr;
                MLB_TRY(launch_em(em, em->fn_emit, a, 0, 8 * kSmCount));
            }
            if (resp_out)
                MLB_TRY(staged_d2h_2d(gpu, resp_out + off, sizeof(double) * ld_out, eg.stage, sizeof(double) * kStagePoints, static_cast<size_t>(em->k), sizeof(double) * n));
            if (labels_out) MLB_TRY(staged_d2h(gpu, labels_out + off, eg.stage_labels, sizeof(unsigned) * n));
            MLB_CUDA(cudaStreamSynchronize(gpu.stream));
        }
        return MLB_OK;
    };
    rc = body();
    for (double* ptr : {xd, r_tmp, ll_tmp})
        if (ptr) cudaFreeAsync(ptr, gpu.stream);
    return rc;
}

int mlb_em_set_kernel_timing(mlb_em* em, int enabled)
{
    MLB_REQUIRE(em, "mlb_em_set_kernel_timing: null argument");
    for (EmGpu& eg : em->gpus) {
        eg.timer.enabled = enabled != 0;
        eg.timer.reset();
    }
    return MLB_OK;
}

int mlb_em_kernel_time_ms(mlb_em* em, double* total_ms, int64_t* launches)
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em, "mlb_em_kernel_time_ms: null argument");
    MLB_CUDA(cudaSetDevice(em->ctx->gpus[0].device));
    return em->gpus[0].timer.total(total_ms, launches);
}

int mlb_em_last_path(const mlb_em* em, int* path)
{
    MLB_REQUIRE(em && path, "mlb_em_last_path: null argument");
    *path = em->last_path;
    return MLB_OK;
}

int mlb_em_direct_steps(const mlb_em* em, int64_t* steps)
{
    MLB_REQUIRE(em && steps, "mlb_em_direct_steps: null argument");
    *steps = em->direct_steps;
    return MLB_OK;
}

int mlb_em_launch_count(const mlb_em* em, int64_t* launches)
{
    MLB_REQUIRE(em && launches, "mlb_em_launch_count: null argument");
    *launches = em->launches;
    return MLB_OK;
}

int mlb_em_kernel_config(const mlb_em* em, int out[8])
{
    MLB_ENTER(em ? em->ctx : nullptr);
    MLB_REQUIRE(em && out, "mlb_em_kernel_config: null argument");
    out[0] = em->path;
    out[1] = em->DP;
    out[2] = em->KP;
    out[3] = em->NT;
    out[4] = em->path == 2 ? em->MW : 0;
    out[5] = em->dr.DP;
    out[6] = em->dr.NB;
    out[7] = em->data->lay.chunk;
    return MLB_OK;
}

}  // extern "C"
