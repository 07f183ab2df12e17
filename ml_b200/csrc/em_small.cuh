// Fused E+M kernel for small dimensions (D <= 8; BASELINE configs C1 and C2), included by em.cu inside namespace mlb.
//
// Same mathematics as em_kernel (feature-space products on the FP64 tensor pipe), different choreography.  With D <= 8
// the whole statistics matrix S[F x K] fits one warp's registers (F <= 48, K <= 32: 48 doubles per lane), so every warp
// runs the complete E -> M chain on its own 16-point sub-tiles and nothing is handed between warps:
//   - no block barrier per tile (only __syncwarp), so the FP64 pipe always has the DMMAs of some warp to run while
//     another warp is in its log-sum-exp;
//   - the E-step's feature products z_a z_b ARE the M-step's features: the E-step stores them once into a per-warp
//     table Phi[point][slot] as it computes them, and the M-step reads its A fragments from it: no second round of
//     multiplies (48 DMUL per 16 points at D = 8) and one shared-memory load per operand instead of two;
//   - M-step rows are in E-step slot order (+ the count row), so the chunk partial has the usual [row][KP] layout and
//     the reduction / exchange / finalize code is shared (the row -> (a, b) table is just different).
// At the end of a chunk the four warps' accumulators are added in the fixed order ((w0 + w1) + w2) + w3.
#pragma once

constexpr int kSmallSub = 16;   // points per warp sub-tile
// Warps per CTA.  Every warp is self-contained (own sub-tiles, own feature table, own accumulators), so the number is free;
// what it sets is how many warps share the SM's registers: 4 warps x 4 CTAs at 128 registers (round 1), or 6 x 3 at 112.
constexpr int kSmallWarps = 4;
constexpr int kSmallThreads = kSmallWarps * 32;
// At most 6 accumulator tiles (K <= 8, or D <= 4 with K <= 16): 96 registers suffice without spilling and a fifth
// resident CTA per SM is worth 4-6 % (measured per 10M points: D = 8, K = 8: 0.832 -> 0.787 ms; D = 4, K = 8:
// 0.464 -> 0.441 ms).  With 12 tiles (C2: D = 8, K = 16) the same bound spills and costs 11 % (1.337 -> 1.488 ms).

// Slot of the constant-1 feature (weighted count): the first dead E-step slot if the packing has one (DQ odd), else a
// new slot after the last E-step slot.
__host__ __device__ constexpr int em_small_count_slot(int DP) { return (DP / 4) % 2 == 1 ? (em_ne(DP) - DP / 4 - 1) * 4 + 2 : em_ne(DP) * 4; }
__host__ __device__ constexpr int em_small_nm(int DP) { return (((DP / 4) % 2 == 1 ? em_ne(DP) * 4 : em_ne(DP) * 4 + 1) + 7) / 8; }

constexpr size_t em_small_smem_bytes(int DP, int KP)
{
    return sizeof(double) * (em_theta_len(DP, KP) + kSmallWarps * kSmallSub * (em_small_nm(DP) * 8 + 4) + kSmallWarps * kSmallSub * (KP + 4) + 8 + DP + kExpTableSize);
}

template <int DP, int KP, int MODE>
__global__ void __launch_bounds__(kSmallThreads, MODE >= 2 ? 4 : ((em_small_nm(DP) * (KP / 8) <= 6) ? 5 : (em_small_nm(DP) * (KP / 8) <= 12) ? 4 : 3)) em_small_kernel(const EmArgs p)
{
    constexpr int NT = KP / 8, DQ = DP / 4, NE = em_ne(DP), NM = em_small_nm(DP);
    constexpr int RS = KP + 4, PS = NM * 8 + 4;
    constexpr int LIN = (NE - DQ) * 4;   // the linear slots of a feature row hold z itself: the point tile lives there
    constexpr int SV = em_sv(DP, KP);
    constexpr int XR = (kSmallSub * DP + 31) / 32;
    constexpr int CS = em_small_count_slot(DP);
    static_assert(NM == em_nm(DP), "the small-shape row count must match the shared partial layout");

    extern __shared__ __align__(16) double sm[];
    double* thE = sm;
    double* cE = thE + NE * NT * 32;
    double* Phi = cE + KP;                        // [warps][16][PS] feature rows (products | z | count); reused as the chunk-end reduction buffer
    double* Rw = Phi + kSmallWarps * kSmallSub * PS;        // [warps][16][RS]
    double* wl = Rw + kSmallWarps * kSmallSub * RS;
    double* sh = wl + 8;
    double* etab = sh + DP;
    __shared__ int s_next;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, c = lane & 3;
    const int d = p.d;

    if (MODE != 1)
        for (int i = tid; i < em_theta_len(DP, KP); i += kSmallThreads) sm[i] = p.theta[i];
    for (int i = tid; i < kSmallWarps * kSmallSub * PS; i += kSmallThreads) Phi[i] = 0.0;
    for (int i = tid; i < kSmallWarps * kSmallSub * RS; i += kSmallThreads) Rw[i] = 0.0;
    if (tid < DP) sh[tid] = tid < d ? p.shift[tid] : 0.0;
    load_exp_table(etab);

    double* F = Phi + warp * kSmallSub * PS;
    double* R = Rw + warp * kSmallSub * RS;

    const long long work_begin = MODE >= 2 ? p.range_begin : 0;
    const long long work_end = MODE >= 2 ? p.range_begin + p.range_count : p.n_local;

    double xr[XR];
    auto load_sub = [&](long long point0, int nvalid) {
        const double* xg = p.x + point0 * d;
        const int nel = nvalid * d;
#pragma unroll
        for (int r = 0; r < XR; ++r) {
            const int e = lane + 32 * r;
            xr[r] = e < nel ? xg[e] : 0.0;
        }
    };
    auto store_sub = [&](int nvalid) {
        const int nel = nvalid * d;
#pragma unroll
        for (int r = 0; r < XR; ++r) {
            const int e = lane + 32 * r;
            if (e < kSmallSub * d) {
                const int pt = (d == DP) ? e / DP : FastDiv(d).div(e);
                const int dm = e - pt * d;
                F[pt * PS + LIN + dm] = e < nel ? xr[r] - sh[dm] : 0.0;
            }
        }
        if (lane < kSmallSub) F[lane * PS + CS] = lane < nvalid ? 1.0 : 0.0;   // the count feature
    };

    for (;;) {
        __syncthreads();
        if (tid == 0) s_next = static_cast<int>(atomicAdd(p.counter, 1u));
        __syncthreads();
        const int chunk = s_next;
        if (chunk >= p.n_chunks) break;
        const long long p_begin = work_begin + static_cast<long long>(chunk) * p.chunk;
        const long long p_end = min64(p_begin + p.chunk, work_end);
        const int nsubs = static_cast<int>((p_end - p_begin + kSmallSub - 1) / kSmallSub);

        double sacc[NM][NT][2];
        if (MODE < 2) {
#pragma unroll
            for (int i = 0; i < NM; ++i)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) sacc[i][nt][0] = sacc[i][nt][1] = 0.0;
        }
        double ll_acc = 0.0, ll_prod = 1.0;
        int nlogged = 0;

        // warp w takes the sub-tiles w, w + warps, w + 2 warps, ... of the chunk
        if (warp < nsubs) load_sub(p_begin + static_cast<long long>(warp) * kSmallSub, static_cast<int>(min64(kSmallSub, p_end - p_begin - static_cast<long long>(warp) * kSmallSub)));
        for (int t = warp; t < nsubs; t += kSmallWarps) {
            const long long tile0 = p_begin + static_cast<long long>(t) * kSmallSub;
            const int nvalid = static_cast<int>(min64(kSmallSub, p_end - tile0));
            __syncwarp();
            store_sub(nvalid);
            if (t + kSmallWarps < nsubs) load_sub(tile0 + kSmallWarps * kSmallSub, static_cast<int>(min64(kSmallSub, p_end - tile0 - kSmallWarps * kSmallSub)));
            __syncwarp();

            const double* z0 = F + g * PS + LIN;
            const double* z1 = z0 + 8 * PS;
            double* f0 = F + g * PS + c;
            double* f1 = f0 + 8 * PS;
            double zc0[DQ], zc1[DQ];
#pragma unroll
            for (int m = 0; m < DQ; ++m) {
                zc0[m] = z0[4 * m + c];
                zc1[m] = z1[4 * m + c];
            }
            double acc[2][NT][2];
            if (MODE != 1) {
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const double2 cc = *reinterpret_cast<const double2*>(cE + 8 * nt + 2 * c);
                    acc[0][nt][0] = acc[1][nt][0] = cc.x;
                    acc[0][nt][1] = acc[1][nt][1] = cc.y;
                }
            }
            // One E-step slot group: the products go to the feature table and (unless the responsibilities are given) into Q.
            auto estep = [&](int j, double a0, double a1, bool keep) {
                if (MODE < 2 && keep) {
                    f0[4 * j] = a0;
                    f1[4 * j] = a1;
                }
                if (MODE != 1) {
                    double bf[NT];
                    load_theta_frag<NT>(thE, j, lane, bf);
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        dmma(acc[0][nt], a0, bf[nt]);
                        dmma(acc[1][nt], a1, bf[nt]);
                    }
                }
            };
#pragma unroll
            for (int a = 0; a < DP - 4; ++a) {
                const double za0 = z0[a], za1 = z1[a];
#pragma unroll
                for (int m = a / 4 + 1; m < DQ; ++m) estep(em_estep_offdiag(DP, a, m), za0 * zc0[m], za1 * zc1[m], true);
            }
            constexpr int J0 = em_ne_offdiag(DP);
#pragma unroll
            for (int m = 0; m < DQ; ++m) estep(J0 + m, zc0[m] * zc0[m], zc1[m] * zc1[m], true);
#pragma unroll
            for (int m = 0; m < DQ; ++m) {
                const int o = 4 * m + ((c + 1) & 3);
                estep(J0 + DQ + m, zc0[m] * z0[o], zc1[m] * z1[o], true);
            }
#pragma unroll
            for (int h = 0; h < (DQ + 1) / 2; ++h) {
                const int mx = 2 * h + (c >> 1);
                const int o = 4 * mx + c, o2 = 4 * mx + ((c + 2) & 3);
                const bool live = mx < DQ;                     // dead lanes: slot 2 of them holds the count feature
                const double u0 = live ? z0[o] * z0[o2] : 0.0, u1 = live ? z1[o] * z1[o2] : 0.0;
                estep(J0 + 2 * DQ + h, u0, u1, live);
            }
#pragma unroll
            for (int m = 0; m < DQ; ++m) estep(NE - DQ + m, zc0[m], zc1[m], false);   // already in the row

            if (MODE == 1) {
                // responsibilities given by the caller (maximise_first, EM.cpp:120-125)
                for (int idx = lane; idx < kSmallSub * p.k; idx += 32) {
                    const int pt = idx % kSmallSub, kk = idx / kSmallSub;
                    R[pt * RS + kk] = pt < nvalid ? p.r_in[tile0 + pt + kk * p.r_ld] : 0.0;
                }
            } else {
                // ---------------- log-sum-exp over the 4 lanes that share a point
                double mxs[2], sums[2];
#pragma unroll
                for (int mt = 0; mt < 2; ++mt) {
                    int mkey = lse_key(acc[mt][0][0]);
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) mkey = max(mkey, max(lse_key(acc[mt][nt][0]), lse_key(acc[mt][nt][1])));
                    mkey = max(mkey, __shfl_xor_sync(0xffffffffu, mkey, 1));
                    mkey = max(mkey, __shfl_xor_sync(0xffffffffu, mkey, 2));
                    const double mx = lse_shift_of_key(mkey);   // within 2^-20 of the largest term (fastmath.cuh)
                    double sum = 0.0;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        acc[mt][nt][0] = exp_nonpositive(acc[mt][nt][0] - mx, etab);
                        acc[mt][nt][1] = exp_nonpositive(acc[mt][nt][1] - mx, etab);
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
                    const int pl = mt * 8 + g;
                    const double inv = invs[mt];
                    if (c == 0 && pl < nvalid) {
                        ll_acc += mxs[mt];
                        ll_prod *= sums[mt];
                    }
                    if (MODE == 0) {
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt)
                            *reinterpret_cast<double2*>(R + pl * RS + 8 * nt + 2 * c) = make_double2(acc[mt][nt][0] * inv, acc[mt][nt][1] * inv);
                    } else if (MODE == 3) {
                        if (c == 0 && pl < nvalid) p.r_out[(tile0 - p.range_begin) + pl] = (mxs[mt] + log(sums[mt])) - 0.5 * d * kLog2Pi;
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
                if (++nlogged == kLogBatch) {
                    ll_acc += log(ll_prod);
                    ll_prod = 1.0;
                    nlogged = 0;
                }
            }
            if (MODE < 2) {
                __syncwarp();
                // ---------------- M-step: S += Phi^T . R over the warp's 16 points, all rows and components in registers
#pragma unroll
                for (int s = 0; s < kSmallSub / 4; ++s) {
                    const double* fp = F + (4 * s + c) * PS + g;
                    const double* rp = R + (4 * s + c) * RS + g;
                    double bf[NT];
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) bf[nt] = rp[8 * nt];
#pragma unroll
                    for (int i = 0; i < NM; ++i) {
                        const double af = fp[8 * i];
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) dmma(sacc[i][nt], af, bf[nt]);
                    }
                }
            }
        }

        if (MODE < 2) {
            ll_acc += log(ll_prod);
            // ---------------- chunk partial: the warps' statistics added in the fixed order ((w0 + w1) + w2) + w3 ...
            double* red = Phi;   // NM * 8 * KP doubles; every warp is past its last read of the feature table
            for (int w = 0; w < kSmallWarps; ++w) {
                __syncthreads();
                if (warp == w) {
#pragma unroll
                    for (int i = 0; i < NM; ++i)
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            double2* cell = reinterpret_cast<double2*>(red + (i * 8 + g) * KP + nt * 8 + 2 * c);
                            double2 v = make_double2(sacc[i][nt][0], sacc[i][nt][1]);
                            if (w > 0) {
                                const double2 o = *cell;
                                v.x = o.x + v.x;
                                v.y = o.y + v.y;
                            }
                            *cell = v;
                        }
                }
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) ll_acc += __shfl_xor_sync(0xffffffffu, ll_acc, off);
            if (lane == 0) wl[warp] = ll_acc;
            __syncthreads();
            double* out = p.partials + static_cast<long long>(chunk) * SV;
            for (int i = tid; i < NM * 8 * KP; i += kSmallThreads) out[i] = red[i];
            if (tid == 0) {
                double ll = (wl[0] + wl[1]) + (wl[2] + wl[3]);
                for (int w = 4; w < kSmallWarps; ++w) ll += wl[w];
                out[NM * 8 * KP] = ll;
            }
            if (tid >= 1 && tid < 8) out[NM * 8 * KP + tid] = 0.0;
            __syncthreads();
            // the feature table must be clean again (dead slots and padding rows are read as zeros by the M-step)
            for (int i = tid; i < NM * 8 * KP && i < kSmallWarps * kSmallSub * PS; i += kSmallThreads) Phi[i] = 0.0;
        }
    }
}
