// Pitch-corrector path kernels (sm_100a): YIN period detection, pitch-mark
// chain + note snapping, LPC residual + PSOLA, all-pole resynthesis + OLA.
// Reference behaviour: Source/PitchProcess.cpp:166-342 (scheduling, filters),
// :350-448 (YIN), :455-658 (marks), :665-870 (PSOLA); Source/Notes.cpp:79-110.
// SURVEY.md App. A.4 / App. B describe the semantics that are restated here.
#include <algorithm>

#include <cuda_pipeline.h>

#include "vp_common.cuh"

// ===========================================================================
// YIN (PitchProcess.cpp:350-448). One CTA per (frame, stream).
//   d[k]  = sum_{i<L} (x[q+i] - x[q+i+k])^2,  q = p - tauMax,  k < tauMax
//   d'[k] = d[k] * k / sum_{j<=k} d[j]
// Direct (a-b)^2 form: all terms positive, so FP32 accumulation keeps ~1e-6
// relative accuracy even in deep minima -- as long as the squares stay normal
// floats. Below 2^-126 rounding is absolute (gradual underflow: up to 2^-150
// per FFMA, squares under 2^-149 vanish), so d[k] also carries an error of up
// to L 2^-150 that no relative margin covers (a frame of samples near 2^-75
// has d[k] ~ 2^-140 and is decided on noise). Thread tile: R consecutive lags
// x one i-range, sliding window of R samples in registers (2 LDS per 2R FP32
// ops; odd R -> conflict-free window loads). CMND prefix sum, threshold search
// and descent run on warp 0 in FP64. A frame whose deciding comparisons are
// within yinEps (relative) or within the bound that the absolute error of d
// puts on d' is queued for the FP64 re-check kernel, which runs the same code
// with T = double (products of floats are normal doubles: no underflow term).
// ===========================================================================
#define YF_RECHECK 1u
#define YF_NEAR 2u
#define YF_UB 4u
#define YF_DONE64 8u

// Exclusive prefix over the lanes of a warp from the inclusive one: the previous lane's inclusive sum. (Not inclusive minus
// own: where a lane's own lags are loud and the lags before them tiny -- a frame that ends where loud audio begins -- the
// subtraction cancels and leaves rounding noise of the loud sum where the tiny prefix should be.)
__device__ __forceinline__ double yin_lane_exclusive(double incl, int lane) {
    const double prev = __shfl_up_sync(0xffffffffu, incl, 1);
    return lane == 0 ? 0.0 : prev;
}

template <int R, typename T, bool MASK>
__device__ __forceinline__ void yin_round(const float* __restrict__ xs, int nb, int nEnd, int k0, T* W, T* acc) {
#pragma unroll
    for (int u = 0; u < R; ++u) {
        const int n = nb + u;
        if (u > 0) W[(u + R - 1) % R] = (T)xs[n + k0 + R - 1];
        const T a = (T)xs[n];
        const T msk = (!MASK || n < nEnd) ? (T)1 : (T)0;
#pragma unroll
        for (int j = 0; j < R; ++j) {
            T d = a - W[(u + j) % R];
            if (MASK) d *= msk;
            acc[j] = fma(d, d, acc[j]);
        }
    }
    W[(R - 1) % R] = (T)xs[nb + R + k0 + R - 1];
}

template <int R, typename T>
__global__ void __launch_bounds__(512) k_yin(VPGeom g, const float* __restrict__ voice, const uint8_t* __restrict__ gate,
                                             int* __restrict__ period, uint32_t* __restrict__ yflags,
                                             int* __restrict__ list, int* __restrict__ listCount, int maxList, int LT,
                                             int IG, int xsLen, bool fromList) {
    extern __shared__ double smd[];
    const int tauMax = g.tauMax, L = g.L;
    const int lagPad = LT * R;
    double* dp = smd;                                 // [lagPad] d then d'
    float* xs = (float*)(smd + lagPad);               // [xsLen]
    T* part = (T*)(xs + ((xsLen + 3) & ~3));          // [IG][lagPad]

    for (int item = blockIdx.x;; item += gridDim.x) {
        long long fidx;
        if (fromList) {
            int cnt = *listCount;
            if (cnt > maxList) cnt = maxList;
            if (item >= cnt) return;
            fidx = list[item];
        } else {
            if (item >= g.nFramesP) return;
            fidx = (long long)blockIdx.y * g.nFramesP + item;
        }
        const int s = (int)(fidx / g.nFramesP), f = (int)(fidx - (long long)s * g.nFramesP);
        const long long p = (long long)f * g.hopP + g.offP;
        const int b = (int)(p / g.B);
        if (gate[(size_t)s * g.nBlocks + b] & VP_GATE_VOICE) {  // gated: yin() is not run (PitchProcess.cpp:208-214)
            if (threadIdx.x == 0) { period[fidx] = 0; yflags[fidx] = 0; }
            if (!fromList) return;
            continue;
        }
        const VPRow v = vp_row(voice, g.histV, s, g);
        const long long q = p - tauMax;
        __syncthreads();
        int nzLoc = 0;
        for (int j = threadIdx.x; j < xsLen; j += blockDim.x) {
            const float x = (j < L + tauMax) ? vp_x(v, q + j, g) : 0.0f;
            xs[j] = x;
            nzLoc |= x != 0.0f;
        }
        const bool nonzero = __syncthreads_or(nzLoc) != 0;  // an all-zero frame is exact: d = 0, no error term
        {
            const int lt = threadIdx.x % LT, ig = threadIdx.x / LT;
            const int iLen = ((L + IG - 1) / IG + R - 1) / R * R;  // multiple of R
            const int i0 = ig * iLen;
            int iEnd = i0 + iLen;
            if (iEnd > L) iEnd = L;
            const int k0 = lt * R;
            T W[R], acc[R];
#pragma unroll
            for (int j = 0; j < R; ++j) { acc[j] = (T)0; W[j] = (i0 < L) ? (T)xs[i0 + k0 + j] : (T)0; }
            int nb = i0;
            for (; nb + R <= iEnd; nb += R) yin_round<R, T, false>(xs, nb, iEnd, k0, W, acc);
            if (nb < iEnd) yin_round<R, T, true>(xs, nb, iEnd, k0, W, acc);
#pragma unroll
            for (int j = 0; j < R; ++j) part[ig * lagPad + k0 + j] = acc[j];
        }
        __syncthreads();
        for (int k = threadIdx.x; k < lagPad; k += blockDim.x) {
            double d = 0.0;
            for (int ig = 0; ig < IG; ++ig) d += (double)part[ig * lagPad + k];
            dp[k] = d;
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            const int lane = threadIdx.x;
            const bool is64 = sizeof(T) == 8;
            const int per = (tauMax + 31) / 32;
            const int kA = lane * per, kB = min(kA + per, tauMax);
            // FP32: absolute error bound of each d[k] from gradual underflow (L FFMAs, 2^-150 each, 25 % head room; the
            // subtraction is exact where it underflows), and ep[k] = the resulting bound on d'[k] (part[] is free now)
            const double eAbs = (!is64 && nonzero) ? (double)L * 0x1p-150 * 1.25 : 0.0;
            double* ep = reinterpret_cast<double*>(part);
            bool unsafe = false;
            // cumulative mean normalisation (PitchProcess.cpp:396-402); d'[0] = 1 and the sum starts at k = 1
            double loc = 0.0;
            for (int k = max(kA, 1); k < kB; ++k) loc += dp[k];
            double incl = loc;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const double t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            double run = yin_lane_exclusive(incl, lane);
            const double total = __shfl_sync(0xffffffffu, incl, 31);
            for (int k = max(kA, 1); k < kB; ++k) {
                run += dp[k];
                const double dn = dp[k] * ((double)k / run);
                if (eAbs > 0.0) {
                    const double runE = eAbs * k;
                    if (run > 2.0 * runE) ep[k] = (eAbs * ((double)k / run) + fabs(dn) * (runE / run)) * 1.01;
                    else { ep[k] = 1e300; if (k >= g.tauMin) unsafe = true; }  // the sum itself is not resolved
                }
                dp[k] = dn;
            }
            if (lane == 0) dp[0] = 1.0;
            __syncwarp();
            // first tau >= tauMin with d'[tau] < yinTol (PitchProcess.cpp:429-433)
            const double tol = 0.25;
            int first = 0x7fffffff;
            for (int k = max(kA, g.tauMin); k < kB; ++k)
                if (dp[k] < tol) { first = k; break; }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
            int per_ = 0;
            unsigned fl = 0;
            double margin = 1e300;
            if (first != 0x7fffffff && total > 0.0) {
                // descent while d'[tau+1] < d'[tau]  (PitchProcess.cpp:435-440)
                if (first + 1 >= tauMax) fl |= YF_UB;  // U3: reads yinTemp[tauMax]
                int stop = 0x7fffffff;
                for (int k = max(kA, first); k < kB; ++k)
                    if (k + 1 >= tauMax || !(dp[k + 1] < dp[k])) { stop = k; break; }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) stop = min(stop, __shfl_xor_sync(0xffffffffu, stop, o));
                per_ = stop;
                for (int k = max(kA, g.tauMin); k < kB; ++k) {
                    if (k <= first) {
                        margin = fmin(margin, fabs(dp[k] - tol) / tol);
                        if (eAbs > 0.0 && !(fabs(dp[k] - tol) > ep[k])) unsafe = true;
                    }
                    if (k >= first && k <= stop && k + 1 < tauMax) {
                        margin = fmin(margin, fabs(dp[k + 1] - dp[k]) / fmax(fabs(dp[k]), 1e-300));
                        if (eAbs > 0.0 && !(fabs(dp[k + 1] - dp[k]) > ep[k] + ep[k + 1])) unsafe = true;
                    }
                }
            } else if (total > 0.0) {
                for (int k = max(kA, g.tauMin); k < kB; ++k) {
                    margin = fmin(margin, fabs(dp[k] - tol) / tol);
                    if (eAbs > 0.0 && !(fabs(dp[k] - tol) > ep[k])) unsafe = true;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) margin = fmin(margin, __shfl_xor_sync(0xffffffffu, margin, o));
            unsafe = __any_sync(0xffffffffu, unsafe);
            if (lane == 0) {
                if (margin < (is64 ? 1e-12 : g.yinEps) || unsafe) fl |= is64 ? YF_NEAR : YF_RECHECK;
                if (is64) fl |= YF_DONE64;
                period[fidx] = per_;
                yflags[fidx] = fl;
                if (!is64 && (fl & YF_RECHECK)) {
                    const int slot = atomicAdd(listCount, 1);
                    if (slot < maxList) list[slot] = (int)fidx;
                }
            }
        }
        if (!fromList) return;
    }
}

struct YinCfg { int R, LT, IG; };
static YinCfg yin_cfg(int tauMax) {
    YinCfg best = {7, 64, 4};
    int bestWaste = 1 << 30;
    const int Rs[6] = {5, 7, 9, 11, 13, 15};
    for (int i = 0; i < 6; ++i) {
        const int R = Rs[i];
        int LT = ((tauMax + R - 1) / R + 31) / 32 * 32;
        const int waste = LT * R - tauMax;
        if (LT <= 128 && waste <= bestWaste) { bestWaste = waste; best.R = R; best.LT = LT; }
    }
    best.IG = 256 / best.LT;
    if (best.IG < 1) best.IG = 1;
    return best;
}

template <typename T>
static void yin_dispatch(cudaStream_t st, const VPGeom& g, int S, const float* voice, const uint8_t* gate, int* period,
                         uint32_t* yflags, int* list, int* listCount, int maxList, bool fromList) {
    const YinCfg c = yin_cfg(g.tauMax);
    const int lagPad = c.LT * c.R;
    const int xsLen = ((g.L + c.R * 2 + lagPad + c.R + 8) + 3) & ~3;
    const size_t smem = (size_t)lagPad * 8 + (size_t)xsLen * 4 + (size_t)c.IG * lagPad * sizeof(T);
    const int threads = c.LT * c.IG;
    dim3 grid = fromList ? dim3(148 * 4) : dim3(g.nFramesP, S);
#define YIN_CASE(RR)                                                                                               \
    case RR:                                                                                                       \
        cudaFuncSetAttribute(k_yin<RR, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);               \
        VP_LAUNCH(k_yin<RR, T><<<grid, threads, smem, st>>>(g, voice, gate, period, yflags, list, listCount, maxList, c.LT, \
                                                  c.IG, xsLen, fromList));                                          \
        break;
    switch (c.R) {
        YIN_CASE(5) YIN_CASE(7) YIN_CASE(9) YIN_CASE(11) YIN_CASE(13) YIN_CASE(15)
    }
#undef YIN_CASE
}

void vp_launch_yin(cudaStream_t st, const VPGeom& g, int S, const float* voice, const uint8_t* gate, int* period,
                   uint32_t* yflags, int* recheckList, int* recheckCount, int maxList) {
    yin_dispatch<float>(st, g, S, voice, gate, period, yflags, recheckList, recheckCount, maxList, false);
}
void vp_launch_yin_recheck(cudaStream_t st, const VPGeom& g, int S, const float* voice, const uint8_t* gate, int* period,
                           uint32_t* yflags, const int* recheckList, const int* recheckCount, int maxList) {
    yin_dispatch<double>(st, g, S, voice, gate, period, yflags, const_cast<int*>(recheckList),
                         const_cast<int*>(recheckCount), maxList, true);
}

// ===========================================================================
// YIN, correlation form (default path). d[k] = A + B(k) - 2 C(k) with
//   A = sum_{i<L} x[q+i]^2,  B(k) = sum_{i<L} x[q+k+i]^2,  C(k) = sum_{i<L} x[q+i] x[q+k+i]
// -- one FFMA per (i, k) pair instead of FADD + FFMA, and because hop = 3c and
// L = 4c (PluginProcessor.cpp:168-170) C(k) splits into four chunk partials
//   Pm(k) = sum_{j in chunk m} x[j] x[j+k],  chunk m = [m c - tauMax, (m+1) c - tauMax)
// of which frame f uses m = 3f .. 3f+3 and shares the last with frame f+1:
// 0.75 L tauMax FFMAs per frame instead of 2 L tauMax lane-ops.
//   k_yin_corr   : FP32, warp <-> chunk, lane <-> 15 consecutive lags (odd stride: conflict-free
//                  window loads; the a[n] load is a broadcast), 15-deep register window.
//   k_yin_decide : one warp per frame, FP64: energies by running sums, CMND, threshold search and
//                  descent, each deciding comparison checked against a rigorous bound on the FP32
//                  accumulation error of C(k),
//                    |err d[k]| <= yin_corr_beta(c) (A + B(k)) + yin_corr_abs(c)   (0 where A + B(k) = 0):
//                  a relative part for the roundings of normal floats and an absolute one for gradual
//                  underflow (products and sums below 2^-126 round to multiples of 2^-149, products
//                  below 2^-150 vanish: without it a frame of samples near 2^-70 is decided on noise,
//                  with d[k] far outside the relative part). A frame with any comparison inside its
//                  bound goes to the FP64 direct-form kernel above.
// ===========================================================================
#define YC_R 15
#define YC_LAGS (32 * YC_R)  // lags per warp pass
#define YC_CH 8              // chunks (= warps) per CTA

#ifndef YC_PAIR_A
#define YC_PAIR_A 1       // 64-bit loads of the broadcast sample in k_yin_corr (0: one 32-bit load per step)
#endif
#define YC_SUB (4 * YC_R)    // first-level accumulation length (two-level FP32 summation: tighter error bound)

// Persistent CTAs: each loops over tiles (one stream x YC_CH chunks) with the samples of the NEXT tile arriving through
// cp.async (zero-filled outside the call's input) into the second of two shared buffers while the current one is
// being correlated -- the staging latency never reaches the FFMA loop.
__global__ void __launch_bounds__(32 * YC_CH, 4) k_yin_corr(VPGeom g, const float* __restrict__ voice, float* __restrict__ P,
                                                             double* __restrict__ Ech, int nChunks, int lagPad,
                                                             int tilesPerStream, long long nTiles, int spanPad, int lagBegin,
                                                             int lagEnd, const int* __restrict__ tileList,
                                                             const int* __restrict__ tileCount, int pairLags) {
    extern __shared__ float xsAll[];  // 2 x [spanPad]; spanPad = 2 sub-spans of subPad floats
    const int c = g.c, tauMax = g.tauMax;
    // A tile = 2 groups of YC_CH consecutive chunks. Warp w works on chunk w of BOTH groups at once: its lower half-warp on
    // group 0, its upper half-warp on group 1, 16 lanes x YC_R lags = YC_LAGS / 2 lags per pass. A pass costs what half of a
    // 32-lane pass over one chunk would, so the lag range can be cut in two phases at no loss. Each group is staged as its
    // own sub-span (its chunks + the lag tail); group 1's starts 16 banks after group 0's so that the two half-warps' window
    // loads (lane stride YC_R floats, odd) never meet in a bank.
    // pairLags (one pass over all lags: single-phase calls, streaming blocks): a tile is ONE group of YC_CH chunks and the
    // two half-warps of a warp split the lag range of the same chunk instead (lags k and k + YC_LAGS / 2 are 16 banks apart).
    const int sub = YC_CH * c + lagPad + 16;
    const int subPad = spanPad >> 1;
    const int tileChunks = pairLags ? YC_CH : 2 * YC_CH;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // with a tile list (second lag phase) the persistent loop runs over the listed tiles only
    const long long nWork = tileList ? (long long)*tileCount : nTiles;
    auto tileOf = [&](long long i) -> long long { return tileList ? (long long)tileList[i] : i; };
    auto issue = [&](long long tile, float* dst) {
        const int s = (int)((unsigned)tile / (unsigned)tilesPerStream);  // tile < 2^31 (checked by the launcher)
        const int m0 = (int)((unsigned)tile - (unsigned)s * (unsigned)tilesPerStream) * tileChunks;
        const VPRow v = vp_row(voice, g.histV, s, g);
        for (int grp = 0; grp < (pairLags ? 1 : 2); ++grp) {
            const long long t0 = (long long)(m0 + grp * YC_CH) * c + g.offP - tauMax - g.lat;  // (call-local) input index of the sub-span's first sample
            float* d = dst + grp * subPad;
            if (t0 >= 0 && t0 + sub <= g.n) {  // common case: the sub-span lies inside this call's input
                const float* src = v.x + t0;
                for (int j = threadIdx.x; j < sub; j += blockDim.x) __pipeline_memcpy_async(d + j, src + j, 4);
            } else {
                for (int j = threadIdx.x; j < sub; j += blockDim.x) {
                    const long long t = t0 + j;
                    const bool ok = t >= -(long long)g.H && t < g.n;
                    const float* src = (t >= 0) ? v.x + (ok ? t : 0) : v.h + (ok ? g.H + t : 0);  // this call's samples / carried history
                    __pipeline_memcpy_async(d + j, src, 4, ok ? 0 : 4);
                }
            }
        }
        __pipeline_commit();
    };
    long long wi = blockIdx.x;
    if (wi >= nWork) return;
    int cur = 0;
    issue(tileOf(wi), xsAll);
    const int half = lane >> 4, lg = lane & 15;
    const bool pairA = YC_PAIR_A && (c & 1) == 0 && (subPad & 1) == 0 && (spanPad & 1) == 0;  // every warp's chunk starts on an even float
    for (; wi < nWork; wi += gridDim.x) {
        const long long tile = tileOf(wi);
        const long long next = wi + gridDim.x;
        float* xs = xsAll + (size_t)cur * spanPad;
        if (next < nWork) { issue(tileOf(next), xsAll + (size_t)(cur ^ 1) * spanPad); __pipeline_wait_prior(1); }
        else __pipeline_wait_prior(0);
        __syncthreads();
        const int s = (int)((unsigned)tile / (unsigned)tilesPerStream);
        const int m = (int)((unsigned)tile - (unsigned)s * (unsigned)tilesPerStream) * tileChunks + (pairLags ? 0 : half * YC_CH) + warp;  // this half-warp's chunk
        const bool live = m < nChunks;
        {
            const float* xa = xs + (pairLags ? 0 : half * subPad) + warp * c;
            float* out = P + ((size_t)s * nChunks + (live ? m : 0)) * (size_t)lagPad;
            if (lagBegin == 0) {  // chunk energy sum_j x[j]^2 in FP64 (exact products): A and B(k) of the decision kernel build on it
                double e2 = 0.0;
                for (int n = lg; n < c; n += 16) { const double x = (double)xa[n]; e2 = fma(x, x, e2); }
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) e2 += __shfl_xor_sync(0xffffffffu, e2, o);
                if (lg == 0 && live && !(pairLags && half)) Ech[(size_t)s * nChunks + m] = e2;
            }
            const int kStep = pairLags ? YC_LAGS : YC_LAGS / 2;
            for (int k0 = lagBegin + (pairLags ? half * (YC_LAGS / 2) : 0) + lg * YC_R; k0 < lagEnd; k0 += kStep) {
                const float* xw = xa + k0;
                float acc[YC_R], acc2[YC_R], W[YC_R];
#pragma unroll
                for (int r = 0; r < YC_R; ++r) { acc[r] = 0.0f; acc2[r] = 0.0f; W[r] = xw[r]; }
                int n = 0;
                while (n + YC_R <= c) {
                    const int nSub = min(n + YC_SUB, c);
                    // a shared-memory load holds the scheduler for ~3 issue cycles next to FFMAs (tools/ubench_yin.cu: 22.6
                    // cycles per 15 FFMA + 2 LDS step, 19.9 with the broadcast sample fetched for two steps at once): rounds
                    // of 2 YC_R steps with 64-bit `a` loads while the chunk length keeps them aligned (n stays even: a single
                    // YC_R round can only close the last, partial group), same order of additions as single rounds
                    if (pairA) {
                        for (; n + 2 * YC_R <= nSub; n += 2 * YC_R) {
#pragma unroll
                            for (int u = 0; u < 2 * YC_R; u += 2) {
                                const float2 a2 = *reinterpret_cast<const float2*>(xa + n + u);
#pragma unroll
                                for (int r = 0; r < YC_R; ++r) acc[r] = fmaf(a2.x, W[(u + r) % YC_R], acc[r]);
                                W[u % YC_R] = xw[n + u + YC_R];
#pragma unroll
                                for (int r = 0; r < YC_R; ++r) acc[r] = fmaf(a2.y, W[(u + 1 + r) % YC_R], acc[r]);
                                W[(u + 1) % YC_R] = xw[n + u + 1 + YC_R];
                            }
                        }
                    }
                    for (; n + YC_R <= nSub; n += YC_R) {
#pragma unroll
                        for (int u = 0; u < YC_R; ++u) {
                            const float a = xa[n + u];
#pragma unroll
                            for (int r = 0; r < YC_R; ++r) acc[r] = fmaf(a, W[(u + r) % YC_R], acc[r]);
                            W[u % YC_R] = xw[n + u + YC_R];
                        }
                    }
#pragma unroll
                    for (int r = 0; r < YC_R; ++r) { acc2[r] += acc[r]; acc[r] = 0.0f; }
                }
#pragma unroll
                for (int u = 0; u < YC_R; ++u) {  // tail: fewer than YC_R samples left
                    if (n + u >= c) break;        // warp-uniform
                    const float a = xa[n + u];
#pragma unroll
                    for (int r = 0; r < YC_R; ++r) acc[r] = fmaf(a, W[(u + r) % YC_R], acc[r]);
                    W[u % YC_R] = xw[n + u + YC_R];
                }
                if (live) {
#pragma unroll
                    for (int r = 0; r < YC_R; ++r) out[k0 + r] = acc2[r] + acc[r];
                }
            }
        }
        __syncthreads();  // everyone is done with this buffer before the tile after next lands in it
        cur ^= 1;
    }
}

// relative bound on |err d[k]| / (A + B(k)): first level <= YC_SUB terms, second level c / YC_SUB + 2 adds, 25 % head room
__host__ __device__ inline double yin_corr_beta(int c) {
    return (double)(YC_SUB + c / YC_SUB + 4) * 5.9604644775390625e-08 * 1.25;
}
// absolute bound on |err d[k]| from gradual underflow: an FP32 rounding into the subnormal range is off by up to 2^-150
// whatever the size of its result. C(k) = 4 chunk partials of c FFMAs + c / YC_SUB + 2 adds (k_yin_corr); x 2 for the 2 C
// in d, 25 % head room. (A and B(k) are double sums of exact products: no underflow.)
__host__ __device__ inline double yin_corr_abs(int c) {
    return 2.0 * 4.0 * (double)(c + c / YC_SUB + 2) * 0x1p-150 * 1.25;
}

#define YD_WARPS 4

__global__ void __launch_bounds__(32 * YD_WARPS) k_yin_decide(VPGeom g, const float* __restrict__ voice,
                                                              const uint8_t* __restrict__ gate, const float* __restrict__ P,
                                                              const double* __restrict__ Ech, int nChunks, int lagPad, int tauPad, int S,
                                                              int* __restrict__ period, uint32_t* __restrict__ yflags,
                                                              int* __restrict__ list, int* __restrict__ listCount, int maxList) {
    extern __shared__ double smd[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long fidx = (long long)blockIdx.x * YD_WARPS + warp;
    if (fidx >= (long long)S * g.nFramesP) return;
    double* dp = smd + (size_t)warp * 2 * tauPad;  // d then d'
    double* er = dp + tauPad;                      // absolute error bound of d'[k]
    float* xlo = (float*)(smd + (size_t)YD_WARPS * 2 * tauPad) + (size_t)warp * 2 * tauPad;  // x[q + i], i < tauMax
    float* xhi = xlo + tauPad;                                                               // x[q + L + i]
    const int tauMax = g.tauMax, L = g.L, c = g.c;
    const int s = (int)(fidx / g.nFramesP), f = (int)(fidx - (long long)s * g.nFramesP);
    const long long p = (long long)f * g.hopP + g.offP;
    const int b = (int)(p / g.B);
    if (gate[(size_t)s * g.nBlocks + b] & VP_GATE_VOICE) {  // gated: yin() is not run (PitchProcess.cpp:208-214)
        if (lane == 0) { period[fidx] = 0; yflags[fidx] = 0; }
        return;
    }
    const VPRow v = vp_row(voice, g.histV, s, g);
    const long long q = p - tauMax;
    // ---- A = sum x[q+i]^2 (exact products in double), edge samples for the running B(k)
    double A = 0.0;
    for (int i = lane; i < L; i += 32) {
        const float x = vp_x(v, q + i, g);
        A = fma((double)x, (double)x, A);
        if (i < tauMax) xlo[i] = x;
    }
    for (int i = lane; i < tauMax; i += 32) xhi[i] = vp_x(v, q + L + i, g);
    A = vp_warp_sum(A);
    // ---- C(k) = four chunk partials
    const float* P0 = P + ((size_t)s * nChunks + (size_t)3 * f) * (size_t)lagPad;
    for (int k = lane; k < tauMax; k += 32) {
        const double cc = ((double)P0[k] + (double)P0[(size_t)lagPad + k]) + ((double)P0[(size_t)2 * lagPad + k] + (double)P0[(size_t)3 * lagPad + k]);
        dp[k] = cc;
    }
    __syncwarp();
    // ---- lane owns consecutive lags [kA, kB): B(k) = A + sum_{i<k} (xhi[i]^2 - xlo[i]^2)
    const int per = (tauMax + 31) / 32;
    const int kA = lane * per, kB = min(kA + per, tauMax);
    double locDelta = 0.0;
    for (int k = kA; k < kB; ++k) { const double h = xhi[k], l = xlo[k]; locDelta += h * h - l * l; }
    double inc = locDelta;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const double t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    double run = yin_lane_exclusive(inc, lane);  // sum of deltas before kA
    const double beta = yin_corr_beta(c), eAbs = yin_corr_abs(c);
    double locD = 0.0, locE = 0.0;
    for (int k = kA; k < kB; ++k) {
        const double Bk = A + run;
        const double h = xhi[k], l = xlo[k];
        run += h * h - l * l;
        const double d = (k == 0) ? 0.0 : (A + Bk) - 2.0 * dp[k];
        const double e = (A + Bk > 0.0) ? fma(beta, A + Bk, eAbs) : 0.0;  // A + B(k) = 0: all samples 0, C(k) exact
        dp[k] = d;
        er[k] = e;
        if (k >= 1) { locD += d; locE += e; }
    }
    double incD = locD, incE = locE;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, incD, o), t2 = __shfl_up_sync(0xffffffffu, incE, o);
        if (lane >= o) { incD += t; incE += t2; }
    }
    double runD = yin_lane_exclusive(incD, lane), runE = yin_lane_exclusive(incE, lane);
    const double total = __shfl_sync(0xffffffffu, incD, 31);
    const double energy = __shfl_sync(0xffffffffu, incE, 31);
    bool shaky = false;  // cumulative sum not resolved against its own error bound
    for (int k = max(kA, 1); k < kB; ++k) {
        runD += dp[k];
        runE += er[k];
        const double d = dp[k], e = er[k];
        const double dn = d * ((double)k / runD);  // cumulative mean normalisation (PitchProcess.cpp:396-402)
        double en;
        if (runD > 2.0 * runE) en = e * ((double)k / runD) + fabs(dn) * (runE / runD) * 1.01;
        else { en = 1e300; if (runE > 0.0 && k >= g.tauMin) shaky = true; }
        dp[k] = dn;
        er[k] = en;
    }
    if (lane == 0) { dp[0] = 1.0; er[0] = 0.0; }
    __syncwarp();
    // ---- first tau >= tauMin with d'[tau] < yinTol, then the descent (PitchProcess.cpp:429-440)
    const double tol = 0.25;
    int first = 0x7fffffff;
    for (int k = max(kA, g.tauMin); k < kB; ++k)
        if (dp[k] < tol) { first = k; break; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
    int per_ = 0;
    unsigned fl = 0;
    bool unsafe = false;
    const bool have = (first != 0x7fffffff) && total > 0.0;
    if (energy > 0.0) {  // all-zero input is exact: d = 0, d' = NaN, unvoiced
        const int kLast = have ? first : tauMax - 1;
        for (int k = max(kA, g.tauMin); k < kB && k <= kLast; ++k)
            if (!(fabs(dp[k] - tol) > er[k])) unsafe = true;
        if (shaky) unsafe = true;
    }
    if (have) {
        if (first + 1 >= tauMax) fl |= YF_UB;  // U3: reads yinTemp[tauMax]
        int stop = 0x7fffffff;
        for (int k = max(kA, first); k < kB; ++k)
            if (k + 1 >= tauMax || !(dp[k + 1] < dp[k])) { stop = k; break; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) stop = min(stop, __shfl_xor_sync(0xffffffffu, stop, o));
        per_ = stop;
        for (int k = max(kA, first); k < kB && k <= stop; ++k)
            if (k + 1 < tauMax && !(fabs(dp[k + 1] - dp[k]) > er[k] + er[k + 1])) unsafe = true;
    }
    unsafe = __any_sync(0xffffffffu, unsafe);
    if (lane == 0) {
        if (unsafe) fl |= YF_RECHECK;
        period[fidx] = per_;
        yflags[fidx] = fl;
        if (unsafe) {
            const int slot = atomicAdd(listCount, 1);
            if (slot < maxList) list[slot] = (int)fidx;
        }
    }
}

#ifndef YD9_CTAS
#define YD9_CTAS 3  // resident CTAs per SM the phase-1 kernel (PER = 9) is compiled for (80 registers, 24 warps: 37.6 -> 33.2 ms; 4: 33.8)
#endif
// Register-resident decision kernel for tauMax <= 32 * PER: lane owns lags [lane PER, (lane + 1) PER), no shared memory.
template <int PER>
__global__ void __launch_bounds__(256, (PER <= 9) ? YD9_CTAS : 2) k_yin_decide_reg(VPGeom g, const float* __restrict__ voice, const uint8_t* __restrict__ gate,
                                                        const float* __restrict__ P, const double* __restrict__ Ech, int nChunks,
                                                        int lagPad, int S, int* __restrict__ period, uint32_t* __restrict__ yflags,
                                                        int* __restrict__ list, int* __restrict__ listCount, int maxList,
                                                        int kLimit, int phase, int* __restrict__ pendList, int* __restrict__ pendCount,
                                                        int* __restrict__ tileFlag, int* __restrict__ tileList,
                                                        int* __restrict__ tileCount, int tilesPerStream, int rs) {
    // rs = row stride of the warp's shared rows in floats (>= 32 PER, multiple of 4): lagPad, or less when only the lags
    // below kLimit are staged (phase 1) -- the kernel waits on its staging copies, so resident warps are what it needs
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    // phase 2 runs over the list of frames phase 1 left pending (persistent warps); phases 0 / 1 over every frame
    const long long nItems = (phase == 2) ? (long long)*pendCount : (long long)S * g.nFramesP;
    for (long long wi = (long long)blockIdx.x * wpb + warp; wi < nItems; wi += (long long)gridDim.x * wpb) {
    const long long fidx = (phase == 2) ? (long long)pendList[wi] : wi;
    const int tauMax = g.tauMax, L = g.L;
    const int s = (int)(fidx / g.nFramesP), f = (int)(fidx - (long long)s * g.nFramesP);
    const long long p = (long long)f * g.hopP + g.offP;
    const int b = (int)(p / g.B);
    // Two lag phases (phase 1: lags below kLimit only, phase 2: all lags, for the frames phase 1 could not finish; phase 0:
    // one pass over all lags). The decision reads d'(tau) only up to the end of the descent after the first dip below the
    // threshold, and d' at a lag depends on smaller lags only: whenever that point lies below kLimit the result of phase 1
    // is the result of the full computation, and the upper lags of the frame's chunks are never correlated.
    if (phase != 2 && (gate[(size_t)s * g.nBlocks + b] & VP_GATE_VOICE)) {
        if (lane == 0) { period[fidx] = 0; yflags[fidx] = 0; }
        continue;
    }
    const int kEnd = (phase == 1) ? min(kLimit, tauMax) : tauMax;  // lags [0, kEnd) are available
    const bool partial = kEnd < tauMax;
    const VPRow v = vp_row(voice, g.histV, s, g);
    const long long q = p - tauMax;
    const double* Ec = Ech + (size_t)s * nChunks + (size_t)3 * f;
    const double A = (Ec[0] + Ec[1]) + (Ec[2] + Ec[3]);
    const int kA = lane * PER;
    const long long tq = q - g.lat;                                     // input index of x[q]
    const bool inside = tq >= 0 && tq + L + tauMax <= g.n;              // common case: no history, no end of input
    // A lane owns PER consecutive lags, so direct global reads touch ~15 cache lines per load instruction and the kernel
    // was bound by L1 wavefronts. The frame's inputs -- 4 chunk rows of P, the tauMax samples entering and leaving the
    // window -- are copied global -> shared asynchronously with lanes on consecutive addresses instead (16-byte
    // copies for the aligned P rows), and each lane then reads its own lags from shared memory (stride PER floats, PER
    // odd: conflict-free).
    extern __shared__ float ydsm[];
    float* sb = ydsm + (size_t)warp * 6 * rs;  // rows 0..3: P chunks 3f..3f+3; row 4: x[q + L + k]; row 5: x[q + k]
    {
        const float4* src = reinterpret_cast<const float4*>(P + ((size_t)s * nChunks + (size_t)3 * f) * (size_t)lagPad);
        float4* dst = reinterpret_cast<float4*>(sb);
        if (!partial) {
            for (int j = lane; j < lagPad; j += 32) __pipeline_memcpy_async(dst + j, src + j, 16);  // 4 rows x lagPad / 4 (rs == lagPad)
        } else {
            const int q4 = (kEnd + 3) >> 2, r4 = lagPad >> 2, d4 = rs >> 2;  // 16-byte pieces per row that hold lags < kEnd
            for (int j = lane; j < 4 * q4; j += 32) {  // (the division is cheaper than it looks: two forms without it measured 37 ms against 31)
                const int row = j / q4, col = j - row * q4;
                __pipeline_memcpy_async(dst + row * d4 + col, src + row * r4 + col, 16);
            }
        }
        float* sh = sb + 4 * rs;
        float* sl = sb + 5 * rs;
        if (inside) {
            const float* ph = v.x + tq + L;
            const float* pl = v.x + tq;
            for (int k = lane; k < kEnd; k += 32) {
                __pipeline_memcpy_async(sh + k, ph + k, 4);
                __pipeline_memcpy_async(sl + k, pl + k, 4);
            }
        } else {
            for (int k = lane; k < kEnd; k += 32) { sh[k] = vp_x(v, q + L + k, g); sl[k] = vp_x(v, q + k, g); }
        }
        __pipeline_commit();
        __pipeline_wait_prior(0);
        __syncwarp();
    }
    const float* P0 = sb + kA;
    double dn[PER], en[PER];
    double locDelta = 0.0;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const int k = kA + j;
        double dl = 0.0;
        if (k < kEnd) {
            const double h = (double)sb[4 * rs + k], l = (double)sb[5 * rs + k];
            dl = h * h - l * l;
        }
        en[j] = dl;  // delta for now
        locDelta += dl;
        dn[j] = ((double)P0[j] + (double)P0[rs + j]) + ((double)P0[2 * rs + j] + (double)P0[3 * rs + j]);
    }
    double inc = locDelta;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const double t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
    double run = yin_lane_exclusive(inc, lane);  // sum of deltas before kA
    const double beta = yin_corr_beta(g.c), eAbs = yin_corr_abs(g.c);
    double locD = 0.0, locE = 0.0;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const int k = kA + j;
        const double Bk = A + run;
        run += en[j];
        double d = (A + Bk) - 2.0 * dn[j], e = (A + Bk > 0.0) ? fma(beta, A + Bk, eAbs) : 0.0;  // 0: all samples 0, C(k) exact
        if (k == 0 || k >= kEnd) { d = 0.0; e = 0.0; }
        dn[j] = d;
        en[j] = e;
        locD += d;
        locE += e;
    }
    double incD = locD, incE = locE;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, incD, o), t2 = __shfl_up_sync(0xffffffffu, incE, o);
        if (lane >= o) { incD += t; incE += t2; }
    }
    double runD = yin_lane_exclusive(incD, lane), runE = yin_lane_exclusive(incE, lane);
    const double total = __shfl_sync(0xffffffffu, incD, 31);
    const double energy = __shfl_sync(0xffffffffu, incE, 31);
    bool shaky = false;
#pragma unroll
    for (int j = 0; j < PER; ++j) {
        const int k = kA + j;
        runD += dn[j];
        runE += en[j];
        const double d = dn[j], e = en[j];
        // one reciprocal instead of three divisions per lag (the divisions were ~45 % of this kernel's instructions);
        // its 1-ulp rounding is covered by the 1.01 slack of the bound (and the decision itself is re-done in the
        // reference's own arithmetic whenever |x - tol| <= ex)
        const double kr = (double)k * __drcp_rn(runD);
        double x = d * kr, ex;
        if (runD > 2.0 * runE) ex = (e * kr + fabs(x) * (runE * __drcp_rn(runD))) * 1.01;
        else { ex = 1e300; if (runE > 0.0 && k >= g.tauMin && k < kEnd) shaky = true; }
        if (k == 0) { x = 1.0; ex = 0.0; }
        dn[j] = x;
        en[j] = ex;
    }
    // value at k + 1 of this lane's last lag lives in the next lane
    const double dnNext = __shfl_down_sync(0xffffffffu, dn[0], 1), enNext = __shfl_down_sync(0xffffffffu, en[0], 1);
    const double tol = 0.25;
    int first = 0x7fffffff;
#pragma unroll
    for (int j = PER - 1; j >= 0; --j) {
        const int k = kA + j;
        if (k >= g.tauMin && k < kEnd && dn[j] < tol) first = k;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
    int per_ = 0;
    unsigned fl = 0;
    bool unsafe = false;
    const bool have = (first != 0x7fffffff) && total > 0.0;
    bool complete = !partial;  // phase 1: the decision is final only if it ends below kEnd
    if (energy > 0.0) {
        const int kLast = have ? first : kEnd - 1;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int k = kA + j;
            if (k >= g.tauMin && k <= kLast && k < kEnd && !(fabs(dn[j] - tol) > en[j])) unsafe = true;
        }
        if (shaky) unsafe = true;
    }
    if (have) {
        if (first + 1 >= tauMax) fl |= YF_UB;
        int stop = 0x7fffffff;
#pragma unroll
        for (int j = PER - 1; j >= 0; --j) {
            const int k = kA + j;
            const double nx = (j == PER - 1) ? dnNext : dn[(j + 1) % PER];
            // (phase 1: d'(k + 1) must be one of the available lags)
            if (k >= first && k < kEnd && (partial ? (k + 1 < kEnd && !(nx < dn[j])) : (k + 1 >= tauMax || !(nx < dn[j])))) stop = k;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) stop = min(stop, __shfl_xor_sync(0xffffffffu, stop, o));
        per_ = stop;
        if (partial) complete = (stop != 0x7fffffff) && energy > 0.0;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int k = kA + j;
            const double nx = (j == PER - 1) ? dnNext : dn[(j + 1) % PER];
            const double ne = (j == PER - 1) ? enNext : en[(j + 1) % PER];
            if (k >= first && k <= stop && k + 1 < kEnd && !(fabs(nx - dn[j]) > en[j] + ne)) unsafe = true;
        }
    }
    if (!complete) {  // uniform across the warp: hand the frame to phase 2 and ask for the upper lags of its chunks' tiles
        if (lane == 0) {
            pendList[atomicAdd(pendCount, 1)] = (int)fidx;
            const int tl = 2 * YC_CH;
            const int t0 = (3 * f) / tl, t1 = (3 * f + 3) / tl;
            for (int t = t0; t <= t1; ++t) {
                const int ti = s * tilesPerStream + t;
                if (atomicExch(tileFlag + ti, 1) == 0) tileList[atomicAdd(tileCount, 1)] = ti;
            }
        }
        continue;
    }
    unsafe = __any_sync(0xffffffffu, unsafe);
    if (lane == 0) {
        if (unsafe) fl |= YF_RECHECK;
        period[fidx] = per_;
        yflags[fidx] = fl;
        if (unsafe) {
            const int slot = atomicAdd(listCount, 1);
            if (slot < maxList) list[slot] = (int)fidx;
        }
    }
    __syncwarp();  // the warp's shared rows are free for its next frame
    }
}

int vp_yin_corr_lagpad(const VPGeom& g) { return (g.tauMax + YC_LAGS - 1) / YC_LAGS * YC_LAGS; }
int vp_yin_corr_chunks(const VPGeom& g) { return 3 * g.nFramesP + 1; }
int vp_yin_corr_tiles(const VPGeom& g) { return (vp_yin_corr_chunks(g) + 2 * YC_CH - 1) / (2 * YC_CH); }  // per stream; tile = 2 x YC_CH chunks

// lags [lagBegin, lagEnd) (multiples of YC_LAGS / 2) of every tile, or -- tileList != nullptr -- of the *tileCount listed tiles
void vp_launch_yin_corr(cudaStream_t st, const VPGeom& g, int S, const float* voice, float* P, double* Ech, int lagBegin,
                        int lagEnd, const int* tileList, const int* tileCount) {
    const int lagPad = vp_yin_corr_lagpad(g), nChunks = vp_yin_corr_chunks(g);
    // sub-span of one chunk group, rounded to 32 floats, + 16: group 1 starts half the banks after group 0
    const int subPad = ((YC_CH * g.c + lagPad + 16 + 31) & ~31) + 16;
    const int spanPad = 2 * subPad;
    const size_t smem = (size_t)2 * spanPad * sizeof(float);
    if (lagEnd <= 0 || lagEnd > lagPad) lagEnd = lagPad;
    // one pass over every lag of every tile: half-warps split the lags of one chunk (tile = YC_CH chunks); lag phases: half-
    // warps take two chunk groups (tile = 2 YC_CH chunks, what vp_yin_corr_tiles counts)
    const int pairLags = (lagBegin == 0 && lagEnd == lagPad && !tileList) ? 1 : 0;
    const int tilesPerStream = pairLags ? (nChunks + YC_CH - 1) / YC_CH : vp_yin_corr_tiles(g);
    const long long nTiles = (long long)tilesPerStream * S;
    cudaFuncSetAttribute(k_yin_corr, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    int perSM = 4;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_yin_corr, 32 * YC_CH, smem);
    if (perSM < 1) perSM = 1;
    int dev = 0, nSM = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nSM, cudaDevAttrMultiProcessorCount, dev);
    long long grid = (long long)nSM * perSM;
    if (grid > nTiles) grid = nTiles;
    if (nTiles >= (1LL << 31)) return;  // cannot happen: the workspace bounds streams x frames per pass far below this
    VP_LAUNCH(k_yin_corr<<<(unsigned)grid, 32 * YC_CH, smem, st>>>(g, voice, P, Ech, nChunks, lagPad, tilesPerStream, nTiles, spanPad, lagBegin,
                                                         lagEnd, tileList, tileCount, pairLags));
}

// First lag phase of the two-phase YIN (0 = not applicable: one pass over all lags). Applicable when the register-resident
// decision kernel is (tauMax <= 32 x 15, one YC_LAGS pass) and the split leaves lags on both sides.
int vp_yin_phase_split(const VPGeom& g) {
    const int k1 = YC_LAGS / 2;
    return (vp_yin_corr_lagpad(g) == YC_LAGS && g.tauMax > k1 + 8 && g.tauMin + 8 < k1) ? k1 : 0;
}

// phase 0: all lags, every frame. phase 1: lags < kLimit, frames whose decision needs more are marked pending and their
// tiles listed. phase 2: all lags, pending frames only. aux = {pending bytes, tileFlag, tileList, tileCount}.
void vp_launch_yin_decide(cudaStream_t st, const VPGeom& g, int S, const float* voice, const uint8_t* gate, const float* P,
                          const double* Ech, int* period, uint32_t* yflags, int* recheckList, int* recheckCount, int maxList,
                          int kLimit, int phase, int* pendList, int* pendCount, int* tileFlag, int* tileList, int* tileCount) {
    const int lagPad = vp_yin_corr_lagpad(g), nChunks = vp_yin_corr_chunks(g);
    const long long tot = (long long)S * g.nFramesP;
    if (g.tauMax <= 32 * 15) {
        const size_t smemReg = (size_t)8 * 6 * lagPad * sizeof(float);
        const int rs9 = std::min(lagPad, 32 * 9);  // phase 1: 9 lags per lane, rows of 288 floats instead of lagPad
        cudaFuncSetAttribute(k_yin_decide_reg<15>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        if (phase == 1 && kLimit <= 32 * 9) {
            // phase 1 reads lags < kLimit only: 9 lags per lane (odd: conflict-free) instead of 15 -> 0.6 x the instructions
            cudaFuncSetAttribute(k_yin_decide_reg<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            VP_LAUNCH(k_yin_decide_reg<9><<<(unsigned)((tot + 7) / 8), 256, (size_t)8 * 6 * rs9 * sizeof(float), st>>>(
                g, voice, gate, P, Ech, nChunks, lagPad, S, period, yflags, recheckList, recheckCount, maxList, kLimit, phase, pendList,
                pendCount, tileFlag, tileList, tileCount, vp_yin_corr_tiles(g), rs9));
            return;
        }
        long long grid = (tot + 7) / 8;
        if (phase == 2) {  // persistent warps over the pending list (its length is only known on the device)
            int dev = 0, nSM = 148;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&nSM, cudaDevAttrMultiProcessorCount, dev);
            grid = std::min<long long>(grid, (long long)nSM * 8);
        }
        VP_LAUNCH(k_yin_decide_reg<15><<<(unsigned)grid, 256, smemReg, st>>>(g, voice, gate, P, Ech, nChunks, lagPad, S, period, yflags,
                                                             recheckList, recheckCount, maxList, kLimit, phase, pendList, pendCount,
                                                             tileFlag, tileList, tileCount, vp_yin_corr_tiles(g), lagPad));
        return;
    }
    const int tauPad = (g.tauMax + 3) & ~3;
    const size_t smem = (size_t)YD_WARPS * 2 * tauPad * (sizeof(double) + sizeof(float));
    cudaFuncSetAttribute(k_yin_decide, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    VP_LAUNCH(k_yin_decide<<<(unsigned)((tot + YD_WARPS - 1) / YD_WARPS), 32 * YD_WARPS, smem, st>>>(
        g, voice, gate, P, Ech, nChunks, lagPad, tauPad, S, period, yflags, recheckList, recheckCount, maxList));
}

// ===========================================================================
// Pitch-mark chain (PitchProcess.cpp:455-658): sequential over the frames of a
// stream, so one warp per stream. The four mark vectors are modelled as
// storage-slot arrays, one slot per lane: push_back writes slot[size],
// insert(begin) shifts right, clear() keeps the values (the reference reads
// slot[size] at PitchProcess.cpp:818, SURVEY.md App. B U1).
// ===========================================================================
struct ArgMin { float v; int i; };

__device__ __forceinline__ int marks_argmin(const float* __restrict__ fr, int i0, int i1, int lane) {
    // first index of the minimum over [i0, i1) (strict '<', PitchProcess.cpp:752-764); empty range -> i0.
    // fr = the frame's samples staged in shared memory.
    float bv = __int_as_float(0x7f800000);
    int bi = 0x7fffffff;
    for (int i = i0 + lane; i < i1; i += 32) {
        const float x = fr[i];
        if (x < bv) { bv = x; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    return (bi == 0x7fffffff) ? i0 : bi;
}

__global__ void __launch_bounds__(128) k_marks(VPGeom g, VPTables tb, const float* __restrict__ voice,
                                               const uint8_t* __restrict__ gate, const int* __restrict__ periodArr,
                                               const uint32_t* __restrict__ yflags, vp_pitch_frame* __restrict__ frames,
                                               VPMarkState* __restrict__ carry, int S) {
    // [warps][2][L + 8] floats: the current frame's samples (argExt searches hit shared memory) and the NEXT frame's, which
    // arrive by cp.async while this frame's marks are placed -- the chain is sequential per stream and latency-bound, and
    // half of its time used to be the wait for a frame's samples (ncu: 51 % of the stall samples on the staging lines)
    extern __shared__ __align__(16) float smarks[];
    const int LB = (g.L + 8 + 3) & ~3;
    float* fbuf = smarks + (size_t)(threadIdx.x >> 5) * 2 * LB;
    const int lane = threadIdx.x & 31;
    const int s = (int)((blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5);
    if (s >= S) return;
    const VPRow v = vp_row(voice, g.histV, s, g);
    const uint8_t* gt = gate + (size_t)s * g.nBlocks;
    const int L = g.L, hop = g.hopP, cap = g.anCap;
    const int lut0 = tb.sp[s].key * (g.tauMax + 1);
    // PitchProcess state (PitchProcess.cpp:76-92), carried from the previous call of this stream
    VPMarkState* cs = carry + s;
    int period = cs->period, prevPeriod = cs->prevPeriod, prevVoicedPeriod = cs->prevVoicedPeriod, periodNew = cs->periodNew;
    bool voiced = cs->voiced != 0, prevVoiced = cs->prevVoiced != 0;
    double beta = cs->beta;
    int an = cs->an[lane], pan = 0, st = cs->st[lane], pst = 0;  // this lane's storage slot of each vector
    int nAn = cs->nAn, nPan = 0, nSt = cs->nSt, nPst = 0;
#define SLOT(arr, i) __shfl_sync(0xffffffffu, (arr), (i))
#define AN_PUSH(val)                                   \
    do {                                               \
        if (nAn >= cap) ub = true;                     \
        if (nAn < VP_SLOTS - 1) { if (lane == nAn) an = (val); ++nAn; } \
    } while (0)
#define ST_PUSH(val)                                   \
    do {                                               \
        if (nSt >= cap) ub = true;                     \
        if (nSt < VP_SLOTS - 1) { if (lane == nSt) st = (val); ++nSt; } \
    } while (0)
    // asynchronous copy of frame f's samples into buffer f & 1; returns the offset of the frame's first sample in the buffer
    // (16-byte copies start at the aligned address at or below it). Frames that reach into the carried history or past the
    // call's input are staged synchronously when they are needed (shift -1).
    auto issue = [&](int f) -> int {
        if (f >= g.nFramesP) return 0;
        const long long t0 = (long long)f * hop + g.offP - g.lat;
        int m = -1;
        if (t0 >= 4 && t0 + L + 4 <= g.n) {
            m = (int)((reinterpret_cast<uintptr_t>(v.x + t0) >> 2) & 3);
            const float4* s4 = reinterpret_cast<const float4*>(v.x + t0 - m);
            float4* d4 = reinterpret_cast<float4*>(fbuf + (f & 1) * LB);
            const int n4 = (m + L + 3) >> 2;
            for (int j = lane; j < n4; j += 32) __pipeline_memcpy_async(d4 + j, s4 + j, 16);
        }
        __pipeline_commit();
        return m;
    };
    int shiftNext = issue(0);
    for (int f = 0; f < g.nFramesP; ++f) {
        const long long p = (long long)f * hop + g.offP;
        const int b = (int)(p / g.B);
        const size_t fidx = (size_t)s * g.nFramesP + f;
        __pipeline_wait_prior(0);
        __syncwarp();  // frame f has landed; every lane is done with frame f - 1's buffer
        const int shift = shiftNext;
        float* fsm = fbuf + (f & 1) * LB + (shift > 0 ? shift : 0);
        shiftNext = issue(f + 1);
        vp_pitch_frame* rec = frames + vp_prow(g, s, f);
        unsigned flags = 0;
        bool ub = false;
        int note = -1, nAnOv = 0;
        const uint8_t gb = gt[b];
        // the note LUT row of the stream's key in the block the frame starts in (Notes.cpp:79-110, read per pitch frame); a call
        // without scheduled changes has one key per stream, loaded once: the chain is sequential, a load per frame is on its path
        const int lut = tb.spStride ? vp_sp(tb, b, s).key * (g.tauMax + 1) : lut0;
        if (gb & VP_GATE_NEAR) flags |= VP_PF_NEAR_GATE;
        if (gb & VP_GATE_VOICE) {
            // PitchProcess.cpp:208-214: anMarks.clear(); prevPitch = 0; return (pitch, stMarks stay stale)
            nAn = 0;
            flags |= VP_PF_GATED;
        } else {
            // ---- yin() state roll (PitchProcess.cpp:415-425)
            prevPeriod = period;
            prevVoiced = voiced;
            if (voiced) prevVoicedPeriod = period;
            period = periodArr[fidx];
            voiced = period > 0;
            if (voiced && shift < 0) {  // (only voiced frames search the waveform) edge frame: not prefetched
                __syncwarp();
                vp_stage<12>(fsm, v, p, L, g, lane, 32);
                __syncwarp();
            }
            const uint32_t yf = yflags[fidx];
            if (yf & YF_NEAR) flags |= VP_PF_NEAR_YIN;
            if ((yf & YF_UB) && !g.defined) ub = true;  // U3; defined: the descent simply ends at the last lag
            if (yf & YF_DONE64) flags |= VP_PF_YIN_RECHECKED;
            // ---- pitchMarks() (PitchProcess.cpp:455-567)
            pan = an; nPan = nAn;  // prevAnMarks = anMarks (element copy)
            nAn = 0;               // clear(): slots keep their values
            pan -= hop;
            nAnOv = __popc(__ballot_sync(0xffffffffu, lane < nPan && pan >= 0));
            if (voiced) {
                const int sw_c = (int)floor(0.94 * period);
                const int sw_f = (int)ceil((2.0 - 0.94) * period);
                bool searchLeft = false;
                int t;
                // defined mode: "previous frame voiced" without previous marks (a gated frame cleared them) searches the frame
                // like the first voiced frame after an unvoiced one
                if (prevVoiced && !(g.defined && nPan == 0)) {
                    if (nAnOv == 0) {
                        int lastMark = 0;
                        if (nPan == 0) ub = true;  // U4: prevAnMarks.back() on an empty vector
                        else lastMark = SLOT(pan, nPan - 1);
                        const int mn = min(prevPeriod, period), mx = max(prevPeriod, period);
                        const int l_lim = max(lastMark + min(sw_c, (int)floor(0.94 * mn)), 0);
                        const int r_lim = min(lastMark + max(sw_f, (int)ceil((2 - 0.94) * mx)), L);
                        t = marks_argmin(fsm, l_lim, r_lim, lane);
                    } else {
                        t = SLOT(pan, nPan - nAnOv);
                    }
                } else {
                    searchLeft = true;
                    t = marks_argmin(fsm, 0, L, lane);
                }
                AN_PUSH(t);
                for (;;) {
                    const int bk = SLOT(an, nAn - 1);
                    if (!(bk + sw_c < L)) break;
                    if (bk + sw_f < L) {
                        const int m = marks_argmin(fsm, bk + sw_c, bk + sw_f, lane);
                        AN_PUSH(m);
                    } else {
                        if (bk + period < L) {
                            const int m = marks_argmin(fsm, bk + sw_c, L, lane);
                            AN_PUSH(m);
                        }
                        break;
                    }
                    if (nAn >= VP_SLOTS - 1) break;
                }
                if (searchLeft) {
                    for (;;) {
                        const int fr = SLOT(an, 0);
                        if (!(fr - sw_c > 0)) break;
                        int m;
                        bool last = false;
                        if (fr - sw_f >= 0) m = marks_argmin(fsm, fr - sw_f, fr - sw_c, lane);
                        else if (fr - period >= 0) { m = marks_argmin(fsm, 0, fr - sw_c, lane); last = true; }
                        else break;
                        // insert(begin): slots [0, nAn) move one to the right
                        if (nAn >= cap) ub = true;
                        if (nAn >= VP_SLOTS - 1) break;
                        const int up = __shfl_up_sync(0xffffffffu, an, 1);
                        if (lane >= 1 && lane <= nAn) an = up;
                        if (lane == 0) an = m;
                        ++nAn;
                        if (last) break;
                    }
                }
            } else if (nPan > 0) {
                if (nAnOv > 0) {
                    for (int i = 0; i < nAnOv; ++i) { const int m = SLOT(pan, nPan - nAnOv + i); AN_PUSH(m); }
                } else {
                    const int m = SLOT(pan, nPan - 1) + prevVoicedPeriod;
                    AN_PUSH(m);
                }
                if (prevVoicedPeriod <= 0) ub = true;
                else
                    for (;;) {
                        const int bk = SLOT(an, nAn - 1);
                        if (!(bk + prevVoicedPeriod < L) || nAn >= VP_SLOTS - 1) break;
                        AN_PUSH(bk + prevVoicedPeriod);
                    }
            }
            // ---- placeStMarks() (PitchProcess.cpp:573-658)
            pst = st; nPst = nSt;
            nSt = 0;
            pst -= hop;
            if (nAn > 0) {
                const int nStOv = __popc(__ballot_sync(0xffffffffu, lane < nPst && pst >= 0));
                if (voiced) {
                    beta = tb.lutBeta[lut + period];
                    periodNew = tb.lutPeriodNew[lut + period];
                    note = tb.lutNote[lut + period];
                } else {
                    periodNew = prevVoicedPeriod;
                }
                bool place = true;
                int firstMark = 0;
                if (periodNew <= 0) { ub = true; place = false; }
                else if (voiced) {
                    if (prevVoiced) {
                        if (nStOv > 0) firstMark = SLOT(pst, nPst - nStOv);
                        else if (nPst == 0) { if (!g.defined) ub = true; firstMark = SLOT(an, 0); }
                        else {
                            const int bk = SLOT(pst, nPst - 1);
                            firstMark = (bk + periodNew >= 0) ? bk + periodNew : SLOT(an, 0);
                        }
                    } else firstMark = SLOT(an, 0);
                } else {
                    if (nPst == 0) place = false;
                    else if (nStOv > 0) firstMark = SLOT(pst, nPst - nStOv);
                    else {
                        const int bk = SLOT(pst, nPst - 1);
                        int nn = 1;
                        while (bk + nn * periodNew < 0) nn += 1;
                        firstMark = bk + nn * periodNew;
                    }
                }
                if (place) {
                    ST_PUSH(firstMark);
                    int bk = firstMark;
                    while (bk + periodNew < L && nSt < VP_SLOTS - 1) { bk += periodNew; ST_PUSH(bk); }
                }
            }
            if (voiced) flags |= VP_PF_VOICED;
            if (nAn > 0) flags |= VP_PF_HAS_MARKS;
        }
        if (ub) flags |= VP_PF_UB;
        // ---- record
        const int stale = (nAn < cap) ? SLOT(an, nAn) : 0;
        // last mark of the previous frame that does not overlap this one (PitchProcess.cpp:812), in this frame's coordinates
        const int kPrev = nPan - nAnOv - 1;
        const int prevLast = ((flags & VP_PF_GATED) || kPrev < 0) ? VP_NO_MARK : SLOT(pan, kPrev);
        if (lane < VP_MAX_MARKS) {
            rec->anMarks[lane] = (lane < nAn) ? an : 0;
            rec->stMarks[lane] = (lane < nSt) ? st : 0;
        }
        if (lane == 0) {
            rec->flags = flags;
            rec->period = (flags & VP_PF_GATED) ? period : period;
            rec->periodPsola = voiced ? period : prevVoicedPeriod;
            rec->periodNew = periodNew;
            rec->note = ((flags & VP_PF_VOICED) && nAn > 0) ? note : -1;
            rec->nAn = nAn;
            rec->nSt = nSt;
            rec->anStale = stale;
            rec->nAnOv = nAnOv;
            rec->prevAnLast = prevLast;
            rec->beta = beta;
        }
    }
    __syncwarp();
    cs->an[lane] = an;
    cs->st[lane] = st;
    if (lane == 0) {
        cs->period = period; cs->prevPeriod = prevPeriod; cs->prevVoicedPeriod = prevVoicedPeriod; cs->periodNew = periodNew;
        cs->voiced = voiced ? 1 : 0; cs->prevVoiced = prevVoiced ? 1 : 0;
        cs->nAn = nAn; cs->nSt = nSt;
        cs->beta = beta;
    }
#undef SLOT
#undef AN_PUSH
#undef ST_PUSH
}

void vp_launch_marks(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                     const uint8_t* gate, const int* period, const uint32_t* yflags, vp_pitch_frame* frames,
                     VPMarkState* carry) {
    const int threads = 128;
    const long long tot = (long long)S * 32;
    cudaFuncSetAttribute(k_marks, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);  // 4 frames of L floats: > 48 KB above 132 kHz
    VP_LAUNCH(k_marks<<<(unsigned)((tot + threads - 1) / threads), threads, (size_t)(threads / 32) * 2 * ((g.L + 8 + 3) & ~3) * sizeof(float), st>>>(
        g, tb, voice, gate, period, yflags, frames, carry, S));
}

// ===========================================================================
// Per pitch frame with marks: LPC (rectangular window, PitchProcess.cpp:233),
// residual e = A(z) x (PitchProcess.cpp:235, :258-259, :280-302), PSOLA on the
// residual (PitchProcess.cpp:665-741, :788-870) -> the IIR input outE, with the
// reference's chunk-by-chunk visibility made explicit (SURVEY.md App. A.4 #6):
// a grain handled while chunk n is current only lands on samples i >= n*c, and
// can only see residual samples up to L + n*c.
// One CTA per (frame, stream), FP64.
// ===========================================================================
// Three kernels (no serial section inside a CTA):
//   k_pitch_autocorr : one warp per frame, FP64, lane = (segment of 16, half of the 16-lag group)
//   k_pitch_levinson : one thread per frame, order-15 recursion fully in registers
//   k_pitch_psola    : one 128-thread CTA per frame: residual (register window) then PSOLA, float outE
#define PA_WARPS 4
#define PA_SEGS 16
#define PA_R 8
#ifndef PA_LOADS
#define PA_LOADS 18  // frame loads in flight per lane in k_pitch_autocorr (measured: 8 -> 17.0 ms, 12 -> 15.3, 18 -> 14.9 for the LPC stage)
#endif

// Frame slots of the pitch synthesis kernels: slot index = f + VP_PC; f < 0 are the last frames of earlier calls (their
// records are carried): the reference adds a chunk's samples into the output ring when the chunk is handled, also
// beyond the current block, so such a frame still owns output positions of this call. Returns false for frames that
// are gated, have no marks, or have no processed chunk reaching into [0, n).
__device__ __forceinline__ bool pf_live(const VPGeom& g, const vp_pitch_frame* rec, int f) {
    const unsigned flags = rec->flags;
    if ((flags & VP_PF_GATED) || !(flags & VP_PF_HAS_MARKS)) return false;
    if (f >= 0) return true;
    if (!g.hasPrev) return false;
    const long long p = vp_ppos(g, f);
    const int lim = vp_plim(g, f);  // chunks of a carried frame that are processed at all (silence() cuts the rest)
    for (int n = 0; n < lim; ++n) {
        const long long q = p + (long long)n * g.c;
        if (q < g.n && q + g.c > 0) return true;
    }
    return false;
}

__global__ void __launch_bounds__(32 * PA_WARPS) k_pitch_autocorr(VPGeom g, const float* __restrict__ voice,
                                                                  const vp_pitch_frame* __restrict__ frames,
                                                                  double* __restrict__ rP, int segLen, int xdLen, long long nFramesTot) {
    extern __shared__ double smd[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long fidx = (long long)blockIdx.x * PA_WARPS + warp;  // slot index over [S][nFramesP + VP_PC]
    if (fidx >= nFramesTot) return;
    const int s = (int)(fidx / (g.nFramesP + VP_PC)), f = (int)(fidx - (long long)s * (g.nFramesP + VP_PC)) - VP_PC;
    if (!pf_live(g, frames + fidx, f)) return;
    const int L = g.L, ord = g.ordP;
    double* xd = smd + (size_t)warp * xdLen;  // frame samples as double, zero beyond L (rectangular window, LPC.cpp:44-97)
    const VPRow v = vp_row(voice, g.histV, s, g);
    const long long p = vp_ppos(g, f);
    {   // frame samples -> double. Common case (frame inside this call's input): plain coalesced loads, 8 in flight per lane.
        // No float landing zone in shared memory: the 9.5 KB of xd per warp alone decide how many warps an SM holds.
        const long long t0 = p - g.lat;
        if (t0 >= 0 && t0 + L <= g.n) {
            const float* src = v.x + t0;
            // batches of PA_LOADS predicated loads per lane, all issued before the first conversion, no remainder loop (the
            // kernel waits on these loads more than on anything else: a 1112-sample frame is 3 round trips instead of 4 + 3)
            for (int j0 = lane; j0 < L; j0 += 32 * PA_LOADS) {
                float t[PA_LOADS];
#pragma unroll
                for (int i = 0; i < PA_LOADS; ++i) t[i] = (j0 + 32 * i < L) ? __ldg(src + j0 + 32 * i) : 0.0f;
#pragma unroll
                for (int i = 0; i < PA_LOADS; ++i) if (j0 + 32 * i < L) xd[j0 + 32 * i] = (double)t[i];
            }
        } else {
            for (int j = lane; j < L; j += 32) xd[j] = (double)vp_x(v, p + j, g);
        }
        for (int j = L + lane; j < xdLen; j += 32) xd[j] = 0.0;
    }
    __syncwarp();
    const int seg = lane & (PA_SEGS - 1), half = lane >> 4;
    const int n0 = seg * segLen;
    const int full = segLen / PA_R, rem = segLen - full * PA_R;
    double* r = rP + (size_t)fidx * (size_t)(ord + 1);
    for (int m0 = half * PA_R; m0 <= ord; m0 += 2 * PA_R) {
        double acc[PA_R], W[PA_R];
#pragma unroll
        for (int j = 0; j < PA_R; ++j) { acc[j] = 0.0; W[j] = xd[n0 + m0 + j]; }
        const double* pa = xd + n0;              // a = x[n]
        const double* pw = pa + m0 + PA_R;       // window element entering at step u: x[n + m0 + R]
        for (int rr = 0; rr < full; ++rr, pa += PA_R, pw += PA_R) {  // full rounds: no bounds predicate
#pragma unroll
            for (int u = 0; u < PA_R; ++u) {
                const double a = pa[u];
#pragma unroll
                for (int j = 0; j < PA_R; ++j) acc[j] = fma(a, W[(u + j) % PA_R], acc[j]);
                W[u % PA_R] = pw[u];
            }
        }
        if (rem > 0) {
#pragma unroll
            for (int u = 0; u < PA_R; ++u) {
                if (u >= rem) break;  // warp-uniform
                const double a = pa[u];
#pragma unroll
                for (int j = 0; j < PA_R; ++j) acc[j] = fma(a, W[(u + j) % PA_R], acc[j]);
                W[u % PA_R] = pw[u];
            }
        }
#pragma unroll
        for (int j = 0; j < PA_R; ++j) {
            double t = acc[j];
            t += __shfl_xor_sync(0xffffffffu, t, 1);
            t += __shfl_xor_sync(0xffffffffu, t, 2);
            t += __shfl_xor_sync(0xffffffffu, t, 4);
            t += __shfl_xor_sync(0xffffffffu, t, 8);
            if (seg == 0 && m0 + j <= ord) r[m0 + j] = t;  // raw sum; k_pitch_levinson applies the 1/L of LPC.cpp:93-96
        }
    }
}

// P > 0: every frame has order P; P == 0: order g.ordP, or with g.ordTabP each frame its stream's own order (rows stay
// g.ordP + 1 wide, the taps beyond the frame's order are written as zeros). Both forms run the same FMA sequence and
// vp_div_const is the correctly rounded x / L, so a frame solved here at order 15 has the bits of k_pitch_levinson<15>.
template <int P>
__global__ void __launch_bounds__(128) k_pitch_levinson(VPGeom g, const int16_t* __restrict__ ordTab, const vp_pitch_frame* __restrict__ frames,
                                                        const double* __restrict__ rP, double* __restrict__ aP, long long nFramesTot) {
    const long long fidx = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // slot index over [S][nFramesP + VP_PC]
    if (fidx >= nFramesTot) return;
    const int s = (int)(fidx / (g.nFramesP + VP_PC)), f = (int)(fidx - (long long)s * (g.nFramesP + VP_PC)) - VP_PC;
    if (!pf_live(g, frames + fidx, f)) return;
    constexpr int PM = (P > 0) ? P : VP_ORDER_MAX;
    const int row = (P > 0) ? P : g.ordP;
    const int ord = (P > 0) ? P : (g.ordTabP ? (int)ordTab[s] : g.ordP);
    double r[PM + 1], a[PM + 1];
    const double* rp = rP + (size_t)fidx * (size_t)(row + 1);
    if (P > 0) {
#pragma unroll
        for (int m = 0; m <= PM; ++m) r[m] = vp_div_const(rp[m], (double)g.L, 1.0 / (double)g.L);
    } else {
        for (int m = 0; m <= ord; ++m) r[m] = rp[m] / (double)g.L;
    }
    // Levinson-Durbin (LPC.cpp:107-148)
    a[0] = 1.0;
    if (fabs(r[0]) < 1e-9) {
        if (P > 0) {
#pragma unroll
            for (int i = 1; i <= PM; ++i) a[i] = 0.0;
        } else {
            for (int i = 1; i <= ord; ++i) a[i] = 0.0;
        }
    } else {
        a[1] = r[1] / r[0];
        if (P > 0) {
#pragma unroll
            for (int q = 2; q <= PM; ++q) {
                double rho = 0.0, ra = 0.0;
#pragma unroll
                for (int i = 1; i < q; ++i) { rho = fma(r[q - i], a[i], rho); ra = fma(r[i], a[i], ra); }
                const double k = (r[q] - rho) / (r[0] - ra);
#pragma unroll
                for (int i = 1; 2 * i <= q; ++i) {
                    const double t1 = a[i], t2 = a[q - i];
                    a[i] = fma(-k, t2, t1);
                    if (i != q - i) a[q - i] = fma(-k, t1, t2);
                }
                a[q] = k;
            }
#pragma unroll
            for (int i = 1; i <= PM; ++i) a[i] = -a[i];
        } else {
            for (int q = 2; q <= ord; ++q) {
                double rho = 0.0, ra = 0.0;
                for (int i = 1; i < q; ++i) { rho = fma(r[q - i], a[i], rho); ra = fma(r[i], a[i], ra); }
                const double k = (r[q] - rho) / (r[0] - ra);
                for (int i = 1; 2 * i <= q; ++i) {
                    const double t1 = a[i], t2 = a[q - i];
                    a[i] = fma(-k, t2, t1);
                    if (i != q - i) a[q - i] = fma(-k, t1, t2);
                }
                a[q] = k;
            }
            for (int i = 1; i <= ord; ++i) a[i] = -a[i];
        }
    }
    double* ap = aP + (size_t)fidx * (size_t)(row + 1);
    if (P > 0) {
#pragma unroll
        for (int i = 0; i <= PM; ++i) ap[i] = a[i];
    } else {
        for (int i = 0; i <= ord; ++i) ap[i] = a[i];
        for (int i = ord + 1; i <= row; ++i) ap[i] = 0.0;
    }
}

#define PF_THREADS 128
#define PF_RJ 9  // residual outputs per thread and pass (odd stride: conflict-free window loads)
#define PF_XPAD 32  // zero floats after the staged frame / spare doubles after the residual (>= 2 PF_RJ)

// P > 0: LPC order known at compile time (coefficients and the residual window live in registers); P == 0: any order.
template <int P>
__global__ void __launch_bounds__(PF_THREADS, 7) k_pitch_psola(VPGeom g, VPTables tb, const float* __restrict__ voice,
                                                            vp_pitch_frame* __restrict__ frames,
                                                            const double* __restrict__ aP, float* __restrict__ outE,
                                                            int xLen, int eLen, int eAlloc) {
    extern __shared__ __align__(16) double smd[];
    const int f = (int)blockIdx.x - VP_PC, s = blockIdx.y;  // f = -1: the previous call's last frame
    const size_t fidx = vp_prow(g, s, f);
    vp_pitch_frame* rec = frames + fidx;
    const int L = g.L, c = g.c, ord = (P > 0) ? P : g.ordP, tauMax = g.tauMax;
    const int X0 = tauMax + ord;        // xf[X0 + idx] = voice at frame-relative idx, idx in [-tauMax - ord, L + 3c)
    double* e = smd;  // [eLen + pad] residual, e[j] <-> frame-relative idx j - tauMax (16-byte aligned: the shared-memory window is)
    // (eAlloc <= eLen doubles are allocated: grain samples end at clAn + T + tauMax <= L + 2 tauMax, the 3-chunk look-ahead of
    // the reference's eFrame beyond that is never read)
    float* xfBase = (float*)(e + ((eAlloc + PF_XPAD + 1) & ~1));  // 16-byte aligned; [xLen + pad] floats; dead after the residual -> oE [L] doubles + Hann table
    double* oE = (double*)xfBase;
    __shared__ int sAn[VP_MAX_MARKS + 1], sSt[VP_MAX_MARKS];
    __shared__ __align__(16) double sAr[(P > 0 ? P : 1) + 1];  // the frame's LPC row (P > 0), staged with the samples
    const VPRow v = vp_row(voice, g.histV, s, g);
    const long long p = vp_ppos(g, f);
    const int chunkLim = vp_plim(g, f);
    const int tid = threadIdx.x;

    // ---- frame samples global -> shared without a register round trip. Common case (the whole span lies inside this
    // call's input): 16-byte copies from the 16-byte aligned address at or below the first sample, the frame then starts
    // m floats into the buffer. Otherwise (history before the call / end of the input): 4-byte copies with zero fill.
    // Issued before the frame's record is looked at: the copies, the record and the marks are then ONE round trip to memory
    // instead of three in a row (the ncu source view had 30 % of this kernel's stall samples on those dependent loads); a
    // frame without marks waits for its copies and leaves.
    const long long t0 = p - X0 - g.lat;
    int m = (int)((reinterpret_cast<uintptr_t>(v.x + t0) >> 2) & 3);
    if (t0 - m >= 0 && t0 + xLen + 4 <= g.n) {
        const float4* s4 = reinterpret_cast<const float4*>(v.x + t0 - m);
        float4* d4 = reinterpret_cast<float4*>(xfBase);
        const int n4 = (m + xLen + 3) >> 2;
        for (int j = tid; j < n4; j += PF_THREADS) __pipeline_memcpy_async(d4 + j, s4 + j, 16);
    } else {
        m = 0;
        for (int j = tid; j < xLen; j += PF_THREADS) {
            const long long t = t0 + j;
            const bool ok = t >= -(long long)g.H && t < g.n;
            const float* src = (t >= 0) ? v.x + (ok ? t : 0) : v.h + (ok ? g.H + t : 0);
            __pipeline_memcpy_async(xfBase + j, src, 4, ok ? 0 : 4);
        }
    }
    const float* xf = xfBase + m;  // the PF_XPAD floats after xf[xLen - 1] only feed residual samples nobody reads
    const double* ap = aP + fidx * (size_t)(ord + 1);
    if (P > 0 && tid < (P + 1) / 2) __pipeline_memcpy_async(sAr + 2 * tid, ap + 2 * tid, 16);  // rows of P + 1 = 16 doubles: 16-byte aligned
    __pipeline_commit();
    const unsigned flags = rec->flags;
    const int T = rec->periodPsola, nSt = rec->nSt, nAn = rec->nAn, nAnOv = rec->nAnOv;
    const double beta = rec->beta;
    if (tid < VP_MAX_MARKS) { sAn[tid] = rec->anMarks[tid]; sSt[tid] = rec->stMarks[tid]; }
    if (!pf_live(g, rec, f)) { __pipeline_wait_prior(0); return; }
    __shared__ int sELo, sEHi, sUb;
    if (tid == 0) { sAn[VP_MAX_MARKS] = 0; sELo = eLen; sEHi = 0; sUb = 0; }
    // Hann table of this frame's period (PitchProcess.cpp:878-882): read in place (one table per period, shared by every
    // frame with that period: cache resident) -- a private shared copy would cost a CTA slot per SM
    const double* __restrict__ hs = tb.hann + ((T > 0 && T < tauMax) ? tb.hannOff[T] : 0);
    __syncthreads();  // marks visible; the staging copies are still in flight under the grain table
    // ---- PSOLA (PitchProcess.cpp:665-741, :788-870). Grain table first: thread m prepares synthesis mark m -- the
    // chunk n at which the reference handles it (the first n with stMark - T < (n + 1) c), the look-ahead and residual
    // extent visible at that chunk, the closest complete analysis mark, the output range -- so that the element loop
    // below carries no per-grain scalar work.
    // per synthesis mark: flags, mark, output range [gI0, gI1), e index of grain sample 0, number of grain samples that exist
    // in the residual filtered so far, and the range [gW0, gW1) of grain samples the Hann window applies to (all of them for
    // an inner mark, the second half for the first mark, the first half for the last: PitchProcess.cpp:697-731)
    __shared__ int gSt[VP_MAX_MARKS], gI0[VP_MAX_MARKS], gI1[VP_MAX_MARKS], gFl[VP_MAX_MARKS], gEb[VP_MAX_MARKS], gJl[VP_MAX_MARKS],
        gW0[VP_MAX_MARKS], gW1[VP_MAX_MARKS];
    const bool okT = T > 0 && T < tauMax;
    if (tid < VP_MAX_MARKS) {
        int fl = 0;  // 1 = process, 2 = first mark, 4 = last mark, 8 = UB in the reference
        if (okT && tid < nSt) {
            const int stMark = sSt[tid];
            const int d = stMark - T;
            const int n = (d < c) ? 0 : d / c;
            const long long Pn = p + (long long)n * c;
            if (n < chunkLim && Pn < g.n) {
                const int stale = rec->anStale;
                const int startSample = (int)(((Pn % g.B) + g.B) % g.B);  // Pn < 0: a chunk emitted by an earlier call
                const int lookahead = g.lat + g.B - startSample;  // bufferIdxMax - startSample (PitchProcess.cpp:800)
                const int nc = n * c;
                // getClosestAnMarkIdx (PitchProcess.cpp:788-831)
                int lo = 0, hi = nAn;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (sAn[mid] < stMark) lo = mid + 1; else hi = mid; }
                const int idx = lo;
                int cl;
                if (idx > 0 && idx < nAn) {
                    if (abs(sAn[idx] - stMark) <= abs(sAn[idx - 1] - stMark) && sAn[idx] + T - nc < lookahead) cl = idx;
                    else if (sAn[idx - 1] + T - nc < lookahead) cl = idx - 1;
                    else if (idx - 2 > 0) cl = idx - 2;
                    else cl = -nAnOv - 1;
                } else if (idx == 0) cl = 0;
                else if (g.defined) {
                    // the completeness test is meant for the mark about to be returned: the last one
                    if (sAn[idx - 1] + T - nc < lookahead) cl = idx - 1;
                    else cl = (idx - 2 >= 0) ? idx - 2 : idx - 1;
                } else {
                    if (stale + T - nc < lookahead) cl = idx - 1;  // anMarks[size]: stale storage slot (U1)
                    else if (idx - 2 >= 0) cl = idx - 2;
                    else { cl = 0; fl |= 8; }
                }
                int clAn;
                if (cl >= 0) clAn = sAn[cl];
                else if (g.defined) clAn = (rec->prevAnLast != VP_NO_MARK) ? rec->prevAnLast : sAn[0];  // what :812 means
                else { clAn = 0; fl |= 8; }  // U2: out-of-bounds prevAnMarks read in the reference
                const double dSt = (double)stMark;
                const double x0 = dSt + (double)(-T) / beta;
                const double xEnd = dSt + (double)(T) / beta;
                if (!g.defined && x0 >= 0.0 && x0 == floor(x0)) fl |= 8;  // U5
                gSt[tid] = stMark;
                // output indices i with x0 <= i <= xEnd (interp(), PitchProcess.cpp:850-852), i >= nc (chunk already
                // filtered, App. A.4 #6), i < L: as integer bounds -- i >= x0 <=> i >= ceil(x0), and i < ceil(xEnd)
                // already implies i <= xEnd -- so that the element loop compares integers only
                gI0[tid] = max(max((int)ceil(x0), 0), nc);
                gI1[tid] = min((int)ceil(xEnd), L);
                {
                    const int eValid = L + nc;                  // residual filtered so far
                    const int eBase = clAn - T + tauMax;        // e index of grain sample j = 0
                    gEb[tid] = eBase;
                    gJl[tid] = min(min(eLen, eAlloc) - eBase, eValid - (clAn - T));  // grain samples j < jLim exist in the residual so far
                    const bool first = tid == 0, last = tid == nSt - 1;
                    gW0[tid] = first ? T : 0;
                    gW1[tid] = (!first && last) ? T : 2 * T + 1;
                }
                atomicMin(&sELo, max(clAn - T + tauMax - 1, 0));          // grain samples j = 0 .. 2T (and j - 1)
                atomicMax(&sEHi, min(clAn + T + tauMax + 1, min(eLen, eAlloc)));
                fl |= 1 | (tid == 0 ? 2 : 0) | (tid == nSt - 1 ? 4 : 0);
            }
        }
        if (fl & 8) atomicOr(&sUb, 1);
        gFl[tid] = fl;
    }
    __pipeline_wait_prior(0);
    __syncthreads();
    // ---- residual e[j] = sum_k a[k] x[j - tauMax - k] (PitchProcess.cpp:280-302). The reference filters frame-relative
    // [-samplesToKeep, L + 3c); only the part the grains read is computed: [eLo, eHi) from the grain table.
    const int eLo = sELo, eHi = sEHi;
    if (P > 0) {
        constexpr int PP = (P > 0) ? P : 1;
        double ar[PP + 1];
#pragma unroll
        for (int k = 0; k <= PP; ++k) ar[k] = sAr[k];
        // Scatter form: every input sample is loaded and converted once and feeds the (up to PP + 1) outputs of this
        // thread it belongs to -- PF_RJ accumulators instead of a PF_RJ + PP window in registers, no bounds predicates
        // (xf and e are padded). Inputs run newest to oldest so that each output still sums its taps k = 0 .. PP in order.
        for (int j0 = eLo + tid * PF_RJ; j0 < eHi; j0 += PF_THREADS * PF_RJ) {
            double acc[PF_RJ];
#pragma unroll
            for (int jj = 0; jj < PF_RJ; ++jj) acc[jj] = 0.0;
            const float* xq = xf + j0;  // xq[q] = x at e-index j0 + q - PP
#pragma unroll
            for (int q = PF_RJ + PP - 1; q >= 0; --q) {
                const double x = (double)xq[q];
#pragma unroll
                for (int jj = 0; jj < PF_RJ; ++jj) {
                    const int k = jj + PP - q;
                    if (k >= 0 && k <= PP) acc[jj] = fma(ar[k], x, acc[jj]);
                }
            }
#pragma unroll
            for (int jj = 0; jj < PF_RJ; ++jj) e[j0 + jj] = acc[jj];
        }
    } else {
        for (int j = eLo + tid; j < eHi; j += PF_THREADS) {
            double acc = 0.0;
            for (int k = 0; k <= ord; ++k) acc = fma(ap[k], (double)xf[j + ord - k], acc);
            e[j] = acc;
        }
    }
    __syncthreads();
    // ---- PSOLA proper. The frame's Hann table (PitchProcess.cpp:878-882, one per period) is copied into the dead sample
    // region first (behind the accumulator), so the two window values of a contribution are shared-memory reads -- they were
    // dependent global loads, 21 % of this kernel's stall samples in the round-1 profile. Per synthesis mark everything that
    // does not depend on the output index comes from the grain table; thread <-> output index i is fixed (i mod PF_THREADS)
    // so that successive grains accumulate into oE[i] in mark order without synchronisation.
    bool ub = !okT;
    for (int i = tid; i < L; i += PF_THREADS) oE[i] = 0.0;  // own indices only: no barrier needed for the accumulator
    if (okT) {
        // first half of the table only (T + 1 values, behind the accumulator in the sample region): the window is symmetric,
        // hann[j] and hann[2 T - j] differ by an ulp of the cosine at most (1e-16 of a contribution)
        double* hsm = oE + L;
        for (int j = tid; j <= T; j += PF_THREADS) hsm[j] = __ldg(hs + j);
        __syncthreads();
        const double dT = (double)T;
        for (int m = 0; m < nSt; ++m) {
            if (!(gFl[m] & 1)) continue;
            const int eb = gEb[m], jl = gJl[m], w0 = gW0[m], w1 = gW1[m], startIdx = gI0[m], stopIdx = gI1[m];
            // first own index >= startIdx
            int i = startIdx + ((tid - startIdx) & (PF_THREADS - 1));
            // interp() (PitchProcess.cpp:842-870): lower_bound j over x[j] = stMark + (j - T) / beta, then linear interpolation
            // between grain samples j-1 and j. In grain coordinates tg = T + (i - stMark) beta the bound is j = ceil(tg) and the
            // weight (i - x[j-1]) / (x[j] - x[j-1]) = tg - (j - 1). The interpolant is continuous in tg, so a lower_bound that
            // differs from the reference's when tg is within rounding of an integer changes the value by O(1e-13) only.
            const double dSt = (double)gSt[m];
            for (; i < stopIdx; i += PF_THREADS) {
                const double tg = fma((double)i - dSt, beta, dT);
                int j = (int)ceil(tg);
                j = max(0, min(j, 2 * T));
                const int ej = eb + j;
                double y1 = (ej >= 0 && j < jl) ? e[ej] : 0.0;
                if (j >= w0 && j < w1) y1 *= hsm[min(j, 2 * T - j)];
                double val = y1;
                if (j > 0) {
                    double y0 = (ej >= 1 && j - 1 < jl) ? e[ej - 1] : 0.0;
                    if (j - 1 >= w0 && j - 1 < w1) y0 *= hsm[min(j - 1, 2 * T - j + 1)];
                    val = fma(y1 - y0, tg - (double)(j - 1), y0);
                }
                oE[i] += val;
            }
        }
        if (sUb) ub = true;
    }
    float* dst = outE + fidx * (size_t)L;
    for (int i = tid; i < L; i += PF_THREADS) dst[i] = (float)oE[i];  // own indices again
    if (ub && tid == 0) rec->flags = flags | VP_PF_UB;
}

// Rows of g.ordP + 1: with g.ordTabP the widest order of the call (at least 15 when the rows can hold it), and each frame
// solved at its own. The autocorrelation's lag sums do not depend on how many lags are computed (the segmentation depends on
// L only), and the residual in k_pitch_psola sums taps 0 .. g.ordP in ascending order, where a zero tap leaves the sum as it
// is: both run unchanged on padded rows, and a row of order <= 15 padded to 16 keeps the P = 15 register path.
void vp_launch_pitch_lpc(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                         const vp_pitch_frame* frames, double* rP, double* aP) {
    const long long tot = (long long)S * (g.nFramesP + VP_PC);
    int segLen = (g.L + PA_SEGS - 1) / PA_SEGS;
    if ((segLen & 1) == 0) ++segLen;  // odd -> the 16 segments of a half-warp hit 16 distinct 64-bit banks
    const int groups = (g.ordP + 1 + 2 * PA_R - 1) / (2 * PA_R);
    const int xdLen = (PA_SEGS * segLen + 2 * PA_R * groups + 2 * PA_R + 3) & ~1;
    const size_t smem = (size_t)PA_WARPS * xdLen * sizeof(double);
    cudaFuncSetAttribute(k_pitch_autocorr, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    VP_LAUNCH(k_pitch_autocorr<<<(unsigned)((tot + PA_WARPS - 1) / PA_WARPS), 32 * PA_WARPS, smem, st>>>(g, voice, frames, rP, segLen, xdLen, tot));
    if (g.ordP == 15 && !g.ordTabP) VP_LAUNCH(k_pitch_levinson<15><<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(g, tb.ordP, frames, rP, aP, tot));
    else VP_LAUNCH(k_pitch_levinson<0><<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(g, tb.ordP, frames, rP, aP, tot));
}

void vp_launch_pitch_psola(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                           vp_pitch_frame* frames, const double* aP, float* outE) {
    const int eLen = g.tauMax + g.L + 3 * g.c;
    const int eAlloc = std::min(eLen, g.L + 2 * g.tauMax + 2);
    int xLen = g.tauMax + g.ordP + g.L + 3 * g.c;  // frame-relative [-tauMax - ord, L + 3c)
    xLen = std::max(xLen, 2 * g.L + 2 * (g.tauMax + 1));  // the region is reused as outE [L] doubles + half a Hann table [tauMax] doubles
    xLen = (xLen + 3) & ~3;
    const size_t smem = (size_t)((eAlloc + PF_XPAD + 1) & ~1) * sizeof(double) + (size_t)(xLen + PF_XPAD + 4) * sizeof(float) + 16;
    dim3 grid(g.nFramesP + VP_PC, S);
    if (g.ordP == 15) {
        cudaFuncSetAttribute(k_pitch_psola<15>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        VP_LAUNCH(k_pitch_psola<15><<<grid, PF_THREADS, smem, st>>>(g, tb, voice, frames, aP, outE, xLen, eLen, eAlloc));
    } else {
        cudaFuncSetAttribute(k_pitch_psola<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        VP_LAUNCH(k_pitch_psola<0><<<grid, PF_THREADS, smem, st>>>(g, tb, voice, frames, aP, outE, xLen, eLen, eAlloc));
    }
}

// ===========================================================================
// All-pole resynthesis of the PSOLA'd residual (PitchProcess.cpp:307-322),
// synthesis window and overlap-add (PitchProcess.cpp:328-342). The recursion is
// serial in i and restarts at every frame, so one thread per frame; a warp
// moves 32-sample slabs of its 32 frames through shared memory so that global
// reads of outE and writes of the output are coalesced 128/256-byte rows.
// Chunks 1..2 are private to a frame (plain stores); chunk 0 / chunk 3 overlap
// the neighbouring frame (exactly two contributors -> deterministic float
// atomics on a zeroed buffer).
// ===========================================================================
#define PI_WARPS 2
#define PI_ROW 36  // floats per tile row: 32 samples + 4 spare (16-byte aligned rows, conflict-free 128-bit accesses)

// STREAM_GAIN: each chunk scales by the gainPitch its stream has in the block that handles the chunk (the block its start lies
// in: fillOutputBuffer scales the whole chunk, also the part past the block's end, PitchProcess.cpp:328-342), and a chunk
// that an earlier call handled by the gain it was emitted with (pgIn); else every chunk of the call has the same gain, passed
// as gpCall. Measured on the default workload (same-box A/B against the form that always reads the table): the table form
// took this kernel from 18.9 to 19.8 ms per step, the argument form is at 18.9 again.
// Both forms store the gains of the chunks of the frames the next call carries (pgOut, the last VP_PC of carried ++ new).
// P = 15: transposed direct form II in registers; P = 0: direct form with a circular history at order g.ordP. The two round
// differently, so a call whose streams have different orders (g.ordTabP) runs P = -1: each frame takes the form and the order
// a call at its stream's order alone would run -- the transposed form (its own 16 registers) at 15, else the direct form.
// Frames of different forms share a warp only where a stream boundary falls inside its 32 slots.
template <int P, bool STREAM_GAIN>
__global__ void __launch_bounds__(32 * PI_WARPS, 8) k_pitch_iir(VPGeom g, VPTables tb, const vp_pitch_frame* __restrict__ frames,
                                                             const double* __restrict__ aP, const float* __restrict__ outE,
                                                             float* __restrict__ outP, long long nFramesTot, double gpCall,
                                                             const float* __restrict__ pgIn, float* __restrict__ pgOut) {
    // Rows of 36 floats: 16-byte aligned (128-bit copies in, 128-bit reads / writes by the filter thread: a quarter-warp's 8
    // rows start 4 banks apart), and the 4 spare floats of a tout row carry that frame's output range and position for the
    // row-wise write-out. A shared-memory or shuffle instruction costs the scheduler ~3 cycles next to FP64 work
    // (tools/ubench_mix.cu), so the slab moves count: per sample and lane this form issues 4.5 of them, the round-1 form
    // (4-byte copies, 4 shuffles per output row) 10.
    __shared__ __align__(16) float tin[PI_WARPS][2][32][PI_ROW];
    __shared__ __align__(16) float tout[PI_WARPS][32][PI_ROW];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long f0 = ((long long)blockIdx.x * PI_WARPS + warp) * 32;
    if (f0 >= nFramesTot) return;
    const long long fidx = f0 + lane;
    const int L = g.L, c = g.c;
    const int row = (P > 0) ? P : g.ordP;  // row width - 1
    int order = row;
    bool active = false;
    int s = 0, f = 0, nSteps = 0;
    if (fidx < nFramesTot) {  // slot index over [S][nFramesP + VP_PC]
        s = (int)(fidx / (g.nFramesP + VP_PC));
        f = (int)(fidx - (long long)s * (g.nFramesP + VP_PC)) - VP_PC;
        active = pf_live(g, frames + fidx, f);
        const long long p = vp_ppos(g, f);
        const int lim = vp_plim(g, f);
        for (int n = 0; n < lim; ++n) if (p + (long long)n * c < g.n) nSteps += c;  // chunks handled up to the end of this call
        if (P < 0) order = tb.ordP[s];
    }
    if (!active) nSteps = 0;
    constexpr int PA = (P > 0) ? P : VP_ORDER_MAX;
    double a[PA + 1], h[PA + 1];  // P > 0: h[k] = transposed-form state s_{k+1} (h[PA] stays 0); else circular output history
    constexpr int PT = (P < 0) ? 15 : 0;
    double at[PT + 1], ht[PT + 1];  // P < 0: coefficients and state of a transposed-form frame (ht[PT] stays 0)
    const bool tdf = P < 0 && order == 15;
    for (int k = 0; k <= PA; ++k) { a[k] = 0.0; h[k] = 0.0; }
#pragma unroll
    for (int k = 0; k <= PT; ++k) { at[k] = 0.0; ht[k] = 0.0; }
    if (active) {
        const double* ap = aP + (size_t)fidx * (row + 1);
        if (tdf) {
#pragma unroll
            for (int k = 0; k <= PT; ++k) at[k] = ap[k];
        } else {
            for (int k = 0; k <= order; ++k) a[k] = ap[k];
        }
    }
    // frame-relative output range that lands inside this call (positions before 0 went out with an earlier call, beyond n go
    // out with a later one) and the frame's offset in the output plane relative to the warp's first stream: lane fr's values
    // go into the spare floats of tout row fr
    const long long myP = vp_ppos(g, f);
    const int s0 = (int)(f0 / (g.nFramesP + VP_PC));
    const long long planeBase = (long long)s0 * (long long)g.pstride;
    {
        int4 meta;
        meta.x = (int)max(0LL, -myP);
        meta.y = (int)min((long long)nSteps, (long long)g.n - myP);
        meta.z = (int)((long long)(s - s0) * (long long)g.pstride + myP);  // |.| < 2^31: checked by the launcher
        meta.w = 0;
        if (nSteps == 0 || meta.y < meta.x) { meta.x = 0; meta.y = 0; meta.z = 0; }  // empty range: hi == lo (the write-out tests i - lo < hi - lo unsigned)
        *reinterpret_cast<int4*>(&tout[warp][lane][32]) = meta;
    }
    // gain of each of the frame's chunks (read per emitted chunk, PitchProcess.cpp:336): chunk n starts at myP + n c; one
    // that starts before the call went out with an earlier call (carried frames only), one that starts at or past the call's
    // end is not emitted in it (0)
    float gch[4];
#pragma unroll
    for (int n = 0; n < 4; ++n) {
        const long long q = myP + (long long)n * c;
        float v = 0.0f;
        if (q < 0) v = (f < 0 && fidx < nFramesTot) ? pgIn[(size_t)s * (VP_PC * 4) + (f + VP_PC) * 4 + n] : 0.0f;
        else if (q < g.n) v = STREAM_GAIN ? vp_sp(tb, (int)(q / g.B), s).gainPitchF : (float)gpCall;
        gch[n] = v;
    }
    {
        const float4 g4 = make_float4(gch[0], gch[1], gch[2], gch[3]);
        const int j = f + VP_PC - g.nFramesP;  // slot of this frame among the ones the next call carries
        if (fidx < nFramesTot && j >= 0) *reinterpret_cast<float4*>(pgOut + (size_t)s * (VP_PC * 4) + j * 4) = g4;
        // (kept in the spare floats of the lane's own row of the first input tile, which the copies never write: a slab of 32
        // samples spans at most two chunks, c >= 46, so the filter loop holds two gains and a boundary instead of four)
        if (STREAM_GAIN) *reinterpret_cast<float4*>(&tin[warp][0][lane][32]) = g4;
    }
    const double gp = gpCall;
    const int nSlabs = (L + 31) / 32;
    int maxSteps = nSteps;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) maxSteps = max(maxSteps, __shfl_xor_sync(0xffffffffu, maxSteps, o));
    // slab sl: row fr of the tile <- outE[frame f0+fr][32 sl .. 32 sl + 32) as asynchronous 16-byte copies (rows of outE are
    // L = 4 c floats: aligned; zero fill beyond the frame's steps) into one of two tiles: the next slab is in flight while
    // this one is filtered
    // (the steps of the 8 frames whose rows this lane copies: fetched once, not once per slab -- the wait for these shuffles
    // was 18 % of the kernel's stall samples)
    int stepsOf[8];
#pragma unroll
    for (int it = 0; it < 8; ++it) stepsOf[it] = __shfl_sync(0xffffffffu, nSteps, it * 4 + (lane >> 3));
    auto issue = [&](int sl, int buf) {
        const int i0 = sl * 32;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int idx = it * 32 + lane, fr = idx >> 3, q4 = (idx & 7) * 4;
            const int valid = min(max(stepsOf[it] - (i0 + q4), 0), 4);
            __pipeline_memcpy_async(&tin[warp][buf][fr][q4], outE + (valid ? (size_t)(f0 + fr) * L + i0 + q4 : 0), 16, 16 - 4 * valid);
        }
        __pipeline_commit();
    };
    if (maxSteps > 0) issue(0, 0);
    for (int sl = 0; sl < nSlabs; ++sl) {
        const int i0 = sl * 32, buf = sl & 1;
        if (i0 >= maxSteps) break;
        if (sl + 1 < nSlabs && i0 + 32 < maxSteps) { issue(sl + 1, buf ^ 1); __pipeline_wait_prior(1); }
        else __pipeline_wait_prior(0);
        __syncwarp();
        float gA = 0.0f, gB = 0.0f;  // STREAM_GAIN: gains of the chunk the slab starts in and of the next one, which starts at bnd
        int bnd = 0;
        if (STREAM_GAIN) {
            const int k = min(i0 / c, 3);
            gA = tin[warp][0][lane][32 + k];
            gB = tin[warp][0][lane][32 + min(k + 1, 3)];
            bnd = (k < 3) ? (k + 1) * c : L + 32;
        }
#pragma unroll 2
        for (int q4 = 0; q4 < 32; q4 += 4) {
            const float4 x4 = *reinterpret_cast<const float4*>(&tin[warp][buf][lane][q4]);
            const float xin[4] = {x4.x, x4.y, x4.z, x4.w};
            float yo[4];
            double wv[4] = {0.0, 0.0, 0.0, 0.0};
            if (i0 + q4 < L) {  // L is a multiple of 4: a group of 4 lies inside the synthesis window or beyond it
                const double2 w01 = *reinterpret_cast<const double2*>(tb.stP + i0 + q4);
                const double2 w23 = *reinterpret_cast<const double2*>(tb.stP + i0 + q4 + 2);
                wv[0] = w01.x; wv[1] = w01.y; wv[2] = w23.x; wv[3] = w23.y;
            }
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                const int i = i0 + q4 + jj;
                double acc = (double)xin[jj];
                if (P > 0) {
                    // transposed direct form II: y = x + s_1; s_k <- s_{k+1} - a[k] y  (independent DFMAs, no history shift)
                    acc += h[0];
#pragma unroll
                    for (int k = 0; k < PA; ++k) h[k] = fma(-a[k + 1], acc, h[k + 1]);
                } else if (tdf) {  // (the same DFMAs as P = 15)
                    acc += ht[0];
#pragma unroll
                    for (int k = 0; k < PT; ++k) ht[k] = fma(-at[k + 1], acc, ht[k + 1]);
                } else {
                    for (int k = 1; k <= order && k <= i; ++k) acc = fma(-a[k], h[(i - k) % order], acc);
                    h[i % order] = acc;
                }
                if (STREAM_GAIN) {
                    const float gi = (i < bnd) ? gA : gB;
                    yo[jj] = (float)(acc * wv[jj] * (double)gi);
                } else {
                    yo[jj] = (float)(acc * wv[jj] * gp);
                }
            }
            *reinterpret_cast<float4*>(&tout[warp][lane][q4]) = make_float4(yo[0], yo[1], yo[2], yo[3]);
        }
        __syncwarp();
        {
            const int i = i0 + lane;
            float* const oLane = outP + planeBase + i;         // per slab; a row then only adds its 32-bit plane offset
            const bool shared2 = i < c || i >= 3 * c;          // cross-fade chunks: two frames contribute
#pragma unroll 4
            for (int fr = 0; fr < 32; ++fr) {
                const int4 meta = *reinterpret_cast<const int4*>(&tout[warp][fr][32]);  // {lo, hi, plane offset}: one broadcast load
                if ((unsigned)(i - meta.x) < (unsigned)(meta.y - meta.x)) {             // lo <= i < hi (an empty range has hi = lo = 0)
                    float* o = oLane + meta.z;
                    const float val = tout[warp][fr][lane];
                    if (shared2) atomicAdd(o, val);
                    else *o = val;
                }
            }
        }
        __syncwarp();
    }
}

void vp_launch_pitch_iir(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const vp_pitch_frame* frames,
                         const double* aP, const float* outE, float* outP, const float* gainUniform, const float* pgIn,
                         float* pgOut) {
    const long long tot = (long long)S * (g.nFramesP + VP_PC);
    const unsigned grid = (unsigned)((tot + 32 * PI_WARPS - 1) / (32 * PI_WARPS));
    // a warp's 32 frame slots span at most 32 / (nFramesP + VP_PC) + 1 streams: their plane offsets relative to the first
    // one are kept in 32 bits
    if (((long long)(32 / (g.nFramesP + VP_PC)) + 2) * (long long)g.pstride >= (1LL << 31)) {
        if (g_vpLaunchError == cudaSuccess) g_vpLaunchError = cudaErrorInvalidValue;
        return;
    }
    const double gp = gainUniform ? (double)*gainUniform : 0.0;
    if (g.ordTabP) {
        if (gainUniform) VP_LAUNCH(k_pitch_iir<-1, false><<<grid, 32 * PI_WARPS, 0, st>>>(g, tb, frames, aP, outE, outP, tot, gp, pgIn, pgOut));
        else VP_LAUNCH(k_pitch_iir<-1, true><<<grid, 32 * PI_WARPS, 0, st>>>(g, tb, frames, aP, outE, outP, tot, gp, pgIn, pgOut));
    } else if (g.ordP == 15) {
        if (gainUniform) VP_LAUNCH(k_pitch_iir<15, false><<<grid, 32 * PI_WARPS, 0, st>>>(g, tb, frames, aP, outE, outP, tot, gp, pgIn, pgOut));
        else VP_LAUNCH(k_pitch_iir<15, true><<<grid, 32 * PI_WARPS, 0, st>>>(g, tb, frames, aP, outE, outP, tot, gp, pgIn, pgOut));
    } else {
        if (gainUniform) VP_LAUNCH(k_pitch_iir<0, false><<<grid, 32 * PI_WARPS, 0, st>>>(g, tb, frames, aP, outE, outP, tot, gp, pgIn, pgOut));
        else VP_LAUNCH(k_pitch_iir<0, true><<<grid, 32 * PI_WARPS, 0, st>>>(g, tb, frames, aP, outE, outP, tot, gp, pgIn, pgOut));
    }
}
