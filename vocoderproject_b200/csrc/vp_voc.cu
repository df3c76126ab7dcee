// Vocoder path kernels (sm_100a): ring-RMS gate, windowed autocorrelation,
// Levinson-Durbin + residual energies, all-pole resynthesis + overlap-add.
// Reference behaviour: Source/VocoderProcess.cpp:190-297, Source/LPC.cpp:44-148,
// Source/MyBuffer.cpp:258-261,:299-302 (SURVEY.md App. A.2-A.3).
#include <cuda_pipeline.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "vp_common.cuh"

// ---------------------------------------------------------------------------
// Gate: RMS of the whole ring at every host block (MyBuffer.cpp:258-261).
// The ring at block b holds input times [(b+1)B - inSize, (b+1)B); zeros
// before time 0. One CTA per (block, stream); FP64 accumulation.
// ---------------------------------------------------------------------------
// Two steps so that every sample is read once: per host block the sum of squares of the whole block and of its last
// `rem` samples (inSize = q B + rem); the ring at block b is then blocks b-q+1 .. b plus the tail of block b-q.
__global__ void __launch_bounds__(128) k_gate_partial(VPGeom g, const float* __restrict__ voice,
                                                      const float* __restrict__ synth, double* __restrict__ part, int rem,
                                                      int carry, int partRows) {
    // part rows per stream: `carry` = q + 1 blocks of the previous calls, then this call's blocks
    const int b = blockIdx.x, s = blockIdx.y;
    const float* v = voice + (size_t)s * g.stride + (size_t)b * g.B;
    const float* y = synth + (size_t)s * g.stride + (size_t)b * g.B;
    double sv = 0.0, ss = 0.0, tv = 0.0, ts = 0.0;
    const int tail0 = g.B - rem;
    // 2 x 8 independent loads in flight per thread before the first use (a block of 1024 samples = one batch)
    constexpr int GU = 8;
    for (int t0 = threadIdx.x; t0 < g.B; t0 += blockDim.x * GU) {
        float av[GU], cv[GU];
#pragma unroll
        for (int k = 0; k < GU; ++k) {
            const int t = t0 + k * (int)blockDim.x;
            av[k] = (t < g.B) ? __ldg(v + t) : 0.0f;
            cv[k] = (t < g.B) ? __ldg(y + t) : 0.0f;
        }
#pragma unroll
        for (int k = 0; k < GU; ++k) {
            const int t = t0 + k * (int)blockDim.x;
            const double a = (double)av[k], c = (double)cv[k];
            // the square of a float is exact in double, so fma(a, a, s) rounds exactly what s + a * a rounds: one FP64
            // instruction per sample and signal instead of two, same sums, same order (zeros beyond the block add nothing)
#ifndef GATE_MULADD
            sv = fma(a, a, sv);
            ss = fma(c, c, ss);
            if (t >= tail0) { tv = fma(a, a, tv); ts = fma(c, c, ts); }
#else
            const double a2 = a * a, c2 = c * c;
            sv += a2; ss += c2;
            if (t >= tail0) { tv += a2; ts += c2; }
#endif
        }
    }
    sv = vp_warp_sum(sv); ss = vp_warp_sum(ss); tv = vp_warp_sum(tv); ts = vp_warp_sum(ts);
    __shared__ double red[4][4];
    if ((threadIdx.x & 31) == 0) {
        const int w = threadIdx.x >> 5;
        red[0][w] = sv; red[1][w] = ss; red[2][w] = tv; red[3][w] = ts;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        const int q = threadIdx.x;
        part[((size_t)s * partRows + carry + b) * 4 + q] = (red[q][0] + red[q][1]) + (red[q][2] + red[q][3]);
    }
}

__global__ void __launch_bounds__(128) k_gate_decide(VPGeom g, const double* __restrict__ part, uint8_t* __restrict__ gate,
                                                     int q, long long tot, int carry, int partRows) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= tot) return;
    const int s = (int)(idx / g.nBlocks), b = (int)(idx - (long long)s * g.nBlocks);
    const double* ps = part + ((size_t)s * partRows + carry) * 4;  // row 0 = this call's block 0; rows -carry..-1 carried (zeros before time 0)
    double sv = ps[(ptrdiff_t)(b - q) * 4 + 2], ss = ps[(ptrdiff_t)(b - q) * 4 + 3];  // oldest: tail of block b - q
    for (int j = q - 1; j >= 0; --j) { sv += ps[(ptrdiff_t)(b - j) * 4 + 0]; ss += ps[(ptrdiff_t)(b - j) * 4 + 1]; }
    // juce::Decibels::gainToDecibels(rms) < -60 (VocoderProcess.cpp:199-204, MyBuffer.cpp:258-261, :299-302)
    const double rv = sqrt(sv / (double)g.inSize), rs = sqrt(ss / (double)g.inSize);
    const double dv = rv > 0.0 ? fmax(-100.0, log10(rv) * 20.0) : -100.0;
    const double ds = rs > 0.0 ? fmax(-100.0, log10(rs) * 20.0) : -100.0;
    uint8_t f = 0;
    if (dv < -60.0) f |= VP_GATE_VOICE;
    if (ds < -60.0) f |= VP_GATE_SYNTH;
    if (fabs(dv + 60.0) < 1e-7 || fabs(ds + 60.0) < 1e-7) f |= VP_GATE_NEAR;
    gate[idx] = f;
}

int vp_gate_carry_rows(const VPGeom& g) { return g.inSize / g.B + 1; }

void vp_launch_gate(cudaStream_t st, const VPGeom& g, int S, const float* voice, const float* synth, uint8_t* gate,
                    double* part, int partRows) {
    const int q = g.inSize / g.B, rem = g.inSize - q * g.B;
    const int carry = q + 1;
    dim3 grid(g.nBlocks, S);
    VP_LAUNCH(k_gate_partial<<<grid, 128, 0, st>>>(g, voice, synth, part, rem, carry, partRows));
    const long long tot = (long long)S * g.nBlocks;
    VP_LAUNCH(k_gate_decide<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(g, part, gate, q, tot, carry, partRows));
}

// ---------------------------------------------------------------------------
// Windowed biased autocorrelation (LPC.cpp:44-97), FP64.
// CTA = 4 consecutive frames of one stream. Warp w owns one group of R lags of
// either signal; lane = segment (8 n-segments) + 8 * frame. Each thread keeps
// R accumulators and an R-deep sliding window of the windowed signal in
// registers: 2 shared loads per R DFMAs. Segment length == 2 (mod 4) and a
// frame stride == 1 (mod 16) make the 64-bit shared loads conflict-free.
// ---------------------------------------------------------------------------
#define AC_R 14
#define AC_FRAMES 4
#define AC_SEGS 8

template <int R>
__device__ __forceinline__ void ac_task(const double* __restrict__ xw, int n0, int segLen, int m0, double* acc) {
    double W[R];
#pragma unroll
    for (int j = 0; j < R; ++j) { acc[j] = 0.0; W[j] = xw[n0 + m0 + j]; }
    // full rounds of R samples: no bounds predicate, every shared-memory access is base + immediate
    const double* p = xw + n0;            // a = x[n]
    const double* pw = p + m0 + R - 1;    // newest window element x[n + m0 + R - 1]
    const int full = segLen / R;
    for (int r = 0; r < full; ++r, p += R, pw += R) {
#pragma unroll
        for (int u = 0; u < R; ++u) {
            if (u > 0) W[(u + R - 1) % R] = pw[u];
            const double a = p[u];
#pragma unroll
            for (int j = 0; j < R; ++j) acc[j] = fma(a, W[(u + j) % R], acc[j]);
        }
        W[(R - 1) % R] = pw[R];  // element for u = 0 of the next round
    }
    const int rem = segLen - full * R;
    if (rem > 0) {  // last, partial round: `rem` steps (a 10 ms frame is 4 full rounds + 6 steps per segment; running the
                    // round out with a = 0 would be 11 % of the kernel's DFMAs). The window reads stay inside the zero padding.
#pragma unroll
        for (int u = 0; u < R; ++u) {
            if (u >= rem) break;  // warp-uniform
            if (u > 0) W[(u + R - 1) % R] = pw[u];
            const double a = p[u];
#pragma unroll
            for (int j = 0; j < R; ++j) acc[j] = fma(a, W[(u + j) % R], acc[j]);
        }
    }
}

__global__ void __launch_bounds__(32 * 12) k_voc_autocorr(VPGeom g, VPTables tb, const float* __restrict__ voice,
                                                          const float* __restrict__ synth, double* __restrict__ rV,
                                                          double* __restrict__ rS, int segLen, int FS, int Gv) {
    extern __shared__ double sm[];
    double* xw = sm;                   // [AC_FRAMES][FS] voice * window
    double* sw = sm + AC_FRAMES * FS;  // [AC_FRAMES][FS] synth ch0 * window
    const int s = blockIdx.y;
    const int k0 = blockIdx.x * AC_FRAMES;
    const VPRow v = vp_row(voice, g.histV, s, g), y = vp_row(synth, g.histS, s, g);
    for (int i = threadIdx.x; i < AC_FRAMES * FS; i += blockDim.x) {
        const int f = i / FS, j = i - f * FS;
        const int k = k0 + f;
        double a = 0.0, c = 0.0;
        if (j < g.wlenV && k < g.nFramesV) {
            const long long u = (long long)k * g.hopV + g.offV + j;
            const double w = tb.wV[j];
            a = (double)vp_x(v, u, g) * w;
            c = (double)vp_x(y, u, g) * w;
        }
        xw[i] = a;
        sw[i] = c;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int seg = lane & (AC_SEGS - 1), f = lane >> 3;
    const bool isVoice = warp < Gv;
    const int grp = isVoice ? warp : warp - Gv;
    const double* sig = (isVoice ? xw : sw) + f * FS;
    const int order = isVoice ? g.ordV : g.ordS;
    double acc[AC_R];
    ac_task<AC_R>(sig, seg * segLen, segLen, grp * AC_R, acc);
#pragma unroll
    for (int j = 0; j < AC_R; ++j) {
        double a = acc[j];
        a += __shfl_xor_sync(0xffffffffu, a, 1);
        a += __shfl_xor_sync(0xffffffffu, a, 2);
        a += __shfl_xor_sync(0xffffffffu, a, 4);
        acc[j] = a;
    }
    const int k = k0 + f;
    if (seg == 0 && k < g.nFramesV) {
        double* r = (isVoice ? rV : rS) + ((size_t)s * g.nFramesV + k) * (size_t)vp_rowlen(order);
#pragma unroll
        for (int j = 0; j < AC_R; ++j) {
            const int m = grp * AC_R + j;
            if (m <= order) r[m] = acc[j];  // raw sum; the Levinson kernel applies the 1/wlen of LPC.cpp:93-96
        }
    }
    // the frame's last `order` windowed samples, appended to its row
    for (int i = threadIdx.x; i < AC_FRAMES * (g.ordV + g.ordS); i += blockDim.x) {
        const int ff = i / (g.ordV + g.ordS), t = i - ff * (g.ordV + g.ordS);
        const int kk = k0 + ff;
        if (kk >= g.nFramesV) continue;
        const bool tv = t < g.ordV;
        const int ord = tv ? g.ordV : g.ordS, tt = tv ? t : t - g.ordV;
        const int j = g.wlenV - ord + tt;
        double* r = (tv ? rV : rS) + ((size_t)s * g.nFramesV + kk) * (size_t)vp_rowlen(ord);
        r[ord + 1 + tt] = (j >= 0) ? (tv ? xw : sw)[ff * FS + j] : 0.0;
    }
}

// The same task with 128-bit shared loads: two `a` samples per load at even steps, two window elements per load at odd
// steps (tools/ubench_mix.cu: a shared load next to DFMAs holds the scheduler ~3 cycles whatever its width, so 14 loads per
// round of 14 steps instead of 28). Needs xw 16-byte aligned and n0, m0, segLen even; the additions are the same, in the same
// order. A 128-bit load is served per quarter-warp (the 8 segments of one lag group): segment stride = 4 (mod 8) words puts
// the 8 lanes on 8 disjoint groups of 4 banks.
template <int R>
__device__ __forceinline__ void ac_task4(const double* __restrict__ xw, int n0, int segLen, int m0, double* acc) {
    static_assert(R % 2 == 0, "pairs of steps");
    double W[R];
#pragma unroll
    for (int j = 0; j < R; j += 2) {
        const double2 w2 = *reinterpret_cast<const double2*>(xw + n0 + m0 + j);
        acc[j] = 0.0; acc[j + 1] = 0.0; W[j] = w2.x; W[j + 1] = w2.y;
    }
    const double* p = xw + n0;            // a = x[n]
    const double* pw = p + m0 + R - 1;    // newest window element of step u: pw[u]
    const int full = segLen / R;
    for (int r = 0; r < full; ++r, p += R, pw += R) {
#pragma unroll
        for (int u = 0; u < R; u += 2) {
            const double2 a = *reinterpret_cast<const double2*>(p + u);
#pragma unroll
            for (int j = 0; j < R; ++j) acc[j] = fma(a.x, W[(u + j) % R], acc[j]);
            const double2 w2 = *reinterpret_cast<const double2*>(pw + u + 1);   // newest elements of steps u + 1 and u + 2
            W[u % R] = w2.x;
#pragma unroll
            for (int j = 0; j < R; ++j) acc[j] = fma(a.y, W[(u + 1 + j) % R], acc[j]);
            W[(u + 1) % R] = w2.y;
        }
    }
    const int rem = segLen - full * R;  // even; the last, partial round runs only its own steps
#pragma unroll
    for (int u = 0; u < R; u += 2) {
        if (u >= rem) break;  // warp-uniform
        const double2 a = *reinterpret_cast<const double2*>(p + u);
#pragma unroll
        for (int j = 0; j < R; ++j) acc[j] = fma(a.x, W[(u + j) % R], acc[j]);
        const double2 w2 = *reinterpret_cast<const double2*>(pw + u + 1);
        W[u % R] = w2.x;
#pragma unroll
        for (int j = 0; j < R; ++j) acc[j] = fma(a.y, W[(u + 1 + j) % R], acc[j]);
        W[(u + 1) % R] = w2.y;
    }
}

// ---------------------------------------------------------------------------
// v2 (default): one WARP per frame; a warp walks AV_BATCH consecutive frames of one stream. Each frame's raw samples are
// loaded coalesced in predicated batches, windowed into two FP64 copies in shared memory (voice, side-chain), and the warp
// runs lane = (segment of 8) x (lag group of 4: voice lags 0-13, side-chain lags 0-13, voice lags 14-27, 27-40) with the
// same register-window task as above. Only warp-level synchronisation.
// ---------------------------------------------------------------------------
#ifndef AV_WARPS
#define AV_WARPS 10  // 10 x 10.3 KB + window: two CTAs per SM = 20 warps (registers capped at 96 by the launch bounds)
#endif
#define AV_BATCH 32  // consecutive frames per warp (cache locality of the 4x overlapping frame reads)
#ifndef AV_STAGE_UNROLL
#define AV_STAGE_UNROLL 9  // raw samples per signal and lane loaded at once, predicated batches (a 556-sample frame at 48 kHz = 2 x 9 x 32)
#endif
constexpr int kStageUnroll = AV_STAGE_UNROLL;
#ifndef AV_TREDUCE
#define AV_TREDUCE 1  // transposed reduction over the segments (0: butterfly on every accumulator)
#endif
#ifndef AV_V4
#define AV_V4 0  // 1: 128-bit shared loads in the lag sums (ac_task4, half the load instructions). Measured [B200]: 129.7 ms against 128.2 for the 64-bit form -- the loop is not bound by its load issue
#endif
#ifndef AV_PREFETCH
#define AV_PREFETCH 0  // 1: the loads of frame k + 1 are issued before the lag sums of frame k (registers held across them).
                       // Measured [B200], default workload, autocorrelation timed alone: 0 -> 128.2 ms; 1 with 8 / 10 / 12 / 15
                       // loads ahead -> 128.2 / 132.0 / 131.3 / 142.6 (spills): the load latency is already covered by the
                       // other 19 warps of the SM, so the default keeps the simple form.
#endif

// A warp walks AV_BATCH consecutive frames of one stream and builds each frame's windowed FP64 copies straight from global
// memory (a sample is read by the 4 frames that overlap it, back to back by the same warp: L1 / L2 hits). An earlier
// version kept the raw samples in a shared-memory ring (every sample loaded once); dropping it cut the warp's shared
// memory from 14.7 to 10.3 KB, i.e. 20 instead of 14 resident warps per SM, and that is worth more (143 -> 130 ms): with
// 3-4 warps per scheduler the FP64 pipe idles whenever all of them are in a non-DFMA stretch.
__global__ void __launch_bounds__(32 * AV_WARPS, 2) k_voc_autocorr2(VPGeom g, VPTables tb, const float* __restrict__ voice,
                                                                 const float* __restrict__ synth, double* __restrict__ rV,
                                                                 double* __restrict__ rS, int segLen, int FS, int ringLen,
                                                                 int batchesPerStream, int S) {
    extern __shared__ __align__(16) double smA[];
    double* sm = smA;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int hop = g.hopV, wlen = g.wlenV;
    double* wv = sm;  // [wlen] analysis window, shared by the CTA
    for (int i = threadIdx.x; i < wlen; i += blockDim.x) wv[i] = tb.wV[i];
    __syncthreads();
    const long long wid = (long long)blockIdx.x * AV_WARPS + warp;
    if (wid >= (long long)batchesPerStream * S) return;
    const int s = (int)(wid / batchesPerStream);
    const int k0 = (int)(wid - (long long)s * batchesPerStream) * AV_BATCH;
    double* xw = sm + ((wlen + 1) & ~1) + (size_t)warp * (2 * FS + ringLen);  // [FS] voice * window (zero padded)
    double* sw = xw + FS;                                                     // [FS] synth ch0 * window
    const VPRow v = vp_row(voice, g.histV, s, g), y = vp_row(synth, g.histS, s, g);
    for (int j = wlen + lane; j < FS; j += 32) { xw[j] = 0.0; sw[j] = 0.0; }
    // lane groups of 8 segments: 0 = voice lags 0-13, 1 = side-chain lags 0-13, 2 = voice lags 14-27, 3 = voice lags 27-40
    // (lag 27 is computed twice, identically). Bank layout of the 64-bit loads, which go out per half-warp over 16 banks:
    // segLen = 2 (mod 4) spreads the 8 segments of a group over the 8 even (or 8 odd) banks. Half-warp 0 = voice group 0 +
    // side-chain: the side-chain copy starts an ODD number of doubles after the voice copy (FS = 1 mod 16), so its `a` loads
    // sit on the odd banks and its window loads (+13) on the even ones, opposite to voice group 0. Half-warp 1 = voice
    // groups 2 and 3: their `a` loads are the same addresses (broadcast), their window loads start 27 and 40 doubles on.
    // (Round 1 paired voice group 2 with the side-chain at an even offset: their `a` loads met on the even banks -- the
    // 14 % conflict wavefronts of profiles/ncu_r01fin4_kernels.md.)
    const int seg = lane & (AC_SEGS - 1), grp = lane >> 3;
    const bool isSynth = grp == 1;
    const double* sig = isSynth ? sw : xw;
#if AV_V4
    const int m0 = (grp == 2) ? AC_R : (grp == 3) ? 2 * AC_R : 0;        // even offsets: 128-bit window loads (ac_task4)
#else
    const int m0 = (grp == 2) ? AC_R : (grp == 3) ? 2 * AC_R - 1 : 0;
#endif
    const int order = isSynth ? g.ordS : g.ordV;
    // The raw samples of a frame are loaded into registers in one go (kStageUnroll loads per signal and lane = 32 kStageUnroll
    // samples: whole frames up to 48 kHz, the head of longer ones; predicated, so 44.1 kHz frames of 441 samples take the same
    // path), then windowed into the FP64 copies. Round 2 measured 6 loads at a time + remainder loop at 149.6 ms, this form at
    // 140.5 ms (mark chain alongside in both). AV_PREFETCH = 1 issues them one frame ahead instead (no gain, see above).
    float rv[kStageUnroll], rs[kStageUnroll];
    auto frame_src = [&](int k, const float*& pv, const float*& ps) -> bool {
        const long long t0 = (long long)k * hop + g.offV - g.lat;
        pv = v.x + t0; ps = y.x + t0;
        return k < g.nFramesV && t0 >= 0 && t0 + wlen <= g.n;   // the frame lies inside this call's input (else: history / zeros, slow path)
    };
    auto prefetch = [&](const float* pv, const float* ps, int j0) {
#pragma unroll
        for (int i = 0; i < kStageUnroll; ++i) {
            const int j = j0 + lane + 32 * i;
            rv[i] = (j < wlen) ? __ldg(pv + j) : 0.0f;
            rs[i] = (j < wlen) ? __ldg(ps + j) : 0.0f;
        }
    };
    auto convert = [&](int j0) {
#pragma unroll
        for (int i = 0; i < kStageUnroll; ++i) {
            const int j = j0 + lane + 32 * i;
            if (j < wlen) {
                const double w = wv[j];
                xw[j] = (double)rv[i] * w;
                sw[j] = (double)rs[i] * w;
            }
        }
    };
    const float *pv = nullptr, *ps = nullptr;
    bool pre = false;
#if AV_PREFETCH
    pre = frame_src(k0, pv, ps);
    if (pre) prefetch(pv, ps, 0);
#endif
    for (int fb = 0; fb < AV_BATCH; ++fb) {
        const int k = k0 + fb;
        if (k >= g.nFramesV) break;
        const long long u0 = (long long)k * hop + g.offV;
        __syncwarp();
#if !AV_PREFETCH
        pre = frame_src(k, pv, ps);
        if (pre) prefetch(pv, ps, 0);
#endif
        // ---- windowed FP64 copies of this frame
        if (pre) {
            convert(0);
            for (int j0 = 32 * kStageUnroll; j0 < wlen; j0 += 32 * kStageUnroll) {  // further batches of a frame longer than one
                prefetch(pv, ps, j0);
                convert(j0);
            }
        } else {
            for (int j = lane; j < wlen; j += 32) {
                const double w = wv[j];
                xw[j] = (double)vp_x(v, u0 + j, g) * w;
                sw[j] = (double)vp_x(y, u0 + j, g) * w;
            }
        }
        __syncwarp();
#if AV_PREFETCH
        pre = (fb + 1 < AV_BATCH) && frame_src(k + 1, pv, ps);
        if (pre) prefetch(pv, ps, 0);
#endif
        double acc[AC_R];
#if AV_V4
        ac_task4<AC_R>(sig, seg * segLen, segLen, m0, acc);
#else
        ac_task<AC_R>(sig, seg * segLen, segLen, m0, acc);
#endif
        double* rowV = rV + ((size_t)s * g.nFramesV + k) * (size_t)vp_rowlen(g.ordV);
        double* rowS = rS + ((size_t)s * g.nFramesV + k) * (size_t)vp_rowlen(g.ordS);
#if AV_TREDUCE
        // Sum over the 8 segments, transposed: at each of the three exchange steps a lane keeps half of its values and trades
        // the other half with its partner, so the 14 sums cost 13 exchanges (26 shuffles) instead of 42 (84) -- a shuffle
        // holds the scheduler like a shared-memory load does. Same pairs added at every step as in the butterfly
        // ((s0 + s1) + (s2 + s3)) + ((s4 + s5) + (s6 + s7)): bit-identical sums. Afterwards lane (b2 b1 b0) of a group
        // holds the sums of lags m0 + 7 b0 + 4 b1 + 2 b2 + {0, 1} (index 7 of a half is padding).
        {
            static_assert(AC_R == 14, "the exchange pattern below is written for 14 lags per group");
            const bool b0 = (seg & 1) != 0, b1 = (seg & 2) != 0, b2 = (seg & 4) != 0;
            double t7[8];
#pragma unroll
            for (int j = 0; j < 7; ++j) {
                const double keep = b0 ? acc[j + 7] : acc[j], send = b0 ? acc[j] : acc[j + 7];
                t7[j] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
            }
            t7[7] = 0.0;
            double t4[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double keep = b1 ? t7[j + 4] : t7[j], send = b1 ? t7[j] : t7[j + 4];
                t4[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
            }
            double* r = isSynth ? rowS : rowV;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const double keep = b2 ? t4[j + 2] : t4[j], send = b2 ? t4[j] : t4[j + 2];
                const double sum = keep + __shfl_xor_sync(0xffffffffu, send, 4);
                const int li = (b1 ? 4 : 0) + (b2 ? 2 : 0) + j;
                const int m = m0 + (b0 ? 7 : 0) + li;
                if (li < 7 && m <= order) r[m] = sum;  // raw sum; the Levinson kernel applies the 1/wlen of LPC.cpp:93-96
            }
        }
#else
#pragma unroll
        for (int j = 0; j < AC_R; ++j) {
            double a = acc[j];
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            a += __shfl_xor_sync(0xffffffffu, a, 4);
            acc[j] = a;
        }
        if (seg == 0) {
            double* r = isSynth ? rowS : rowV;
#pragma unroll
            for (int j = 0; j < AC_R; ++j) {
                const int m = m0 + j;
                if (m <= order) r[m] = acc[j];  // raw sum; the Levinson kernel applies the 1/wlen of LPC.cpp:93-96
            }
        }
#endif
        // the frame's last `order` windowed samples, appended to its row (coalesced)
        for (int t = lane; t < g.ordV; t += 32) rowV[g.ordV + 1 + t] = (wlen - g.ordV + t >= 0) ? xw[wlen - g.ordV + t] : 0.0;
        for (int t = lane; t < g.ordS; t += 32) rowS[g.ordS + 1 + t] = (wlen - g.ordS + t >= 0) ? sw[wlen - g.ordS + t] : 0.0;
        __syncwarp();
    }
}

void vp_launch_voc_autocorr(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                            const float* synth, const uint8_t* gate, double* rV, double* rS) {
    (void)gate;
    int segLen = (g.wlenV + AC_SEGS - 1) / AC_SEGS;
    while ((segLen & 3) != 2) ++segLen;
    const int Gv = (g.ordV + 1 + AC_R - 1) / AC_R, Gs = (g.ordS + 1 + AC_R - 1) / AC_R;
    // window reads reach n + m0 + 2R: pad, then round the frame stride to 1 (mod 16)
    int FS = AC_SEGS * segLen + (Gv > Gs ? Gv : Gs) * AC_R + 2 * AC_R + 2;
    while ((FS & 15) != 1) ++FS;
    // (the streaming form always runs its three voice lag groups, whatever the order: pad for lag offsets up to 27 + 2 R)
    int FSv = AC_SEGS * segLen + 3 * AC_R + 2 * AC_R + 2;
    if (FSv < FS) FSv = FS;
#if AV_V4
    const int FS2 = (FSv + 1) & ~1;            // even: the voice and the side-chain copy both 16-byte aligned (ac_task4)
#else
    const int FS2 = (FSv + 15) / 16 * 16 + 1;  // odd distance between the voice and the side-chain copy (see k_voc_autocorr2)
#endif
    const int ringLen = 0;   // (no raw-sample ring any more: see k_voc_autocorr2)
    const size_t smem2 = ((size_t)((g.wlenV + 1) & ~1) + (size_t)AV_WARPS * (2 * FS2 + ringLen)) * sizeof(double);
    // the streaming form needs its seven warps' windows + rings in shared memory (fits up to 88.2 kHz frames)
    // (any voice order up to 40 and side-chain order up to 13: lags beyond an order are computed and not stored)
    if (g.ordV + 1 <= 3 * AC_R - 1 && Gs == 1 && smem2 <= (size_t)200 * 1024) {
        FS = FS2;
        const size_t smem = smem2;
        const int batchesPerStream = (g.nFramesV + AV_BATCH - 1) / AV_BATCH;
        const long long warps = (long long)batchesPerStream * S;
        cudaFuncSetAttribute(k_voc_autocorr2, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        VP_LAUNCH(k_voc_autocorr2<<<(unsigned)((warps + AV_WARPS - 1) / AV_WARPS), 32 * AV_WARPS, smem, st>>>(
            g, tb, voice, synth, rV, rS, segLen, FS, ringLen, batchesPerStream, S));
        return;
    }
    const size_t smem = (size_t)2 * AC_FRAMES * FS * sizeof(double);
    cudaFuncSetAttribute(k_voc_autocorr, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    dim3 grid((g.nFramesV + AC_FRAMES - 1) / AC_FRAMES, S);
    VP_LAUNCH(k_voc_autocorr<<<grid, 32 * (Gv + Gs), smem, st>>>(g, tb, voice, synth, rV, rS, segLen, FS, Gv));
}

// ---------------------------------------------------------------------------
// Levinson-Durbin (LPC.cpp:107-148) + residual energies, one thread per frame.
// The energy of the zero-state FIR residual over the frame
// (VocoderProcess.cpp:235-251) is evaluated in closed form:
//   E = wlen * (r0 + sum_k a_k r_k)  -  sum_{i=wlen}^{wlen+p-1} e_full[i]^2
// (total energy of the full convolution minus its tail past the frame end),
// 41 + p^2/2 DFMAs instead of wlen*(p+1). Verified to ~1e-14 relative against
// the reference's direct sum (DESIGN.md).
// ---------------------------------------------------------------------------
__device__ void lev_solve(const double* r, double* a, int order) {
    // |r0| < 1e-9 -> a = [1, 0, ...]   (LPC.cpp:110-114)
    a[0] = 1.0;
    if (fabs(r[0]) < 1e-9) {
        for (int i = 1; i <= order; ++i) a[i] = 0.0;
        return;
    }
    a[1] = r[1] / r[0];
    for (int p = 2; p <= order; ++p) {
        double rho = 0.0, ra = 0.0;
        for (int i = 1; i < p; ++i) { rho = fma(r[p - i], a[i], rho); ra = fma(r[i], a[i], ra); }
        const double k = (r[p] - rho) / (r[0] - ra);  // error energy recomputed every order (LPC.cpp:131-136)
        for (int i = 1; 2 * i <= p; ++i) {
            const double t1 = a[i], t2 = a[p - i];
            a[i] = fma(-k, t2, t1);
            if (i != p - i) a[p - i] = fma(-k, t1, t2);
        }
        a[p] = k;
    }
    for (int i = 1; i <= order; ++i) a[i] = -a[i];
}

// residual energy of the zero-state FIR over the frame in closed form (see above); xt = the frame's last `order`
// windowed samples (appended to the autocorrelation row by the autocorr kernels)
__device__ double fir_energy(const double* r, const double* a, int order, int wlen, const double* __restrict__ xt) {
    double q = r[0];
    for (int k = 1; k <= order; ++k) q = fma(a[k], r[k], q);
    // tail of the full convolution: i = wlen + d, d = 0..order-1, taps k = d+1..order on xw[wlen + d - k]
    double tail = 0.0;
    for (int d = 0; d < order; ++d) {
        double e = 0.0;
        for (int k = d + 1; k <= order; ++k) e = fma(a[k], xt[order + d - k], e);
        tail = fma(e, e, tail);
    }
    // q wlen rounded on its own, then the tail subtracted (spelled out: k_voc_levinson_static's per-frame form must round
    // exactly like this for the orders that run here)
    const double E = __dsub_rn(__dmul_rn(q, (double)wlen), tail);
    return E > 0.0 ? E : 0.0;
}

__global__ void __launch_bounds__(128) k_voc_levinson(VPGeom g, VPTables tb, const uint8_t* __restrict__ gate,
                                                      const double* __restrict__ rV, const double* __restrict__ rS,
                                                      double* __restrict__ aV, double* __restrict__ aS,
                                                      double* __restrict__ EeV, double* __restrict__ EeS, int S) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)S * g.nFramesV) return;
    const int s = (int)(idx / g.nFramesV), k = (int)(idx - (long long)s * g.nFramesV);
    const size_t row = vp_vrow(g, s, k);
    const int b = (int)(((unsigned)k * (unsigned)g.hopV + (unsigned)g.offV) / (unsigned)g.B);  // block of the frame's start
    // the frame's own orders: the stream's at its start block (VocoderProcess.cpp:193-194) when the call's streams differ;
    // the rows are g.ordV / g.ordS wide, and their tails hold the LAST g.ordV / g.ordS windowed samples
    int pv = g.ordV, ps = g.ordS;
    if (g.ordTab) { const VPStreamParam& q = vp_sp(tb, b, s); pv = q.ordV; ps = q.ordS; }
    double r[VP_ORDER_MAX + 1], a[VP_ORDER_MAX + 1];
    {
        const double* rp = rV + (size_t)idx * vp_rowlen(g.ordV);
        for (int m = 0; m <= pv; ++m) r[m] = rp[m] / (double)g.wlenV;
        lev_solve(r, a, pv);
        double* ap = aV + row * (g.synV + 1);
        for (int m = 0; m <= g.synV; ++m) ap[m] = (m <= pv) ? a[m] : 0.0;  // zero padded up to the call's row order
        EeV[row] = fir_energy(r, a, pv, g.wlenV, rp + g.ordV + 1 + (g.ordV - pv));
    }
    {
        const double* rp = rS + (size_t)idx * vp_rowlen(g.ordS);
        for (int m = 0; m <= ps; ++m) r[m] = rp[m] / (double)g.wlenV;
        lev_solve(r, a, ps);
        double* ap = aS + row * (g.synS + 1);
        for (int m = 0; m <= g.synS; ++m) ap[m] = (m <= ps) ? a[m] : 0.0;
        const double eS = fir_energy(r, a, ps, g.wlenV, rp + g.ordS + 1 + (g.ordS - ps));
        // a frame skipped by the silence gate (VocoderProcess.cpp:199-204) is marked with EeSynth = -1
        const bool gated = (gate[(size_t)s * g.nBlocks + b] & (VP_GATE_VOICE | VP_GATE_SYNTH)) != 0;
        EeS[row] = gated ? -1.0 : eS;
    }
}

// rp / ap / xt point into SHARED memory (row of this thread, odd stride): the CTA stages them with coalesced,
// batched global accesses, because 232 registers per thread leave no room to keep dozens of global loads in flight.
// ord <= P: the frame's own order. The recursion stops there and the taps beyond it are +0.0, so the energy sums below
// append exact zero terms (fma(+0, x, e) == e) after the real ones: bit-identical to solving at order `ord` (lev_solve /
// fir_energy); the tail samples xt[P + d - k] are the same windowed samples wlen + d - k whatever the row's width.
// fused: E = q wlen - tail in one rounding, as this kernel has always computed it at its own orders; else the product is
// rounded first, as fir_energy does -- a frame gets the rounding of the kernel a call at its orders alone would run.
template <int P>
__device__ __forceinline__ double lev_energy_static(const double* __restrict__ rp, double* __restrict__ ap, int wlen,
                                                    const double* __restrict__ xts, int ord, bool fused) {
    double r[P + 1], a[P + 1];
    const double dw = (double)wlen, iw = 1.0 / dw;
#pragma unroll
    for (int m = 0; m <= P; ++m) r[m] = vp_div_const(rp[m], dw, iw);  // biased autocorrelation: r / wlen (LPC.cpp:93-96)
    a[0] = 1.0;
    if (fabs(r[0]) < 1e-9) {
#pragma unroll
        for (int i = 1; i <= P; ++i) a[i] = 0.0;
    } else {
        a[1] = r[1] / r[0];
#pragma unroll
        for (int p = 2; p <= P; ++p) {
            if (p <= ord) {
                double rho = 0.0, ra = 0.0;
#pragma unroll
                for (int i = 1; i < p; ++i) { rho = fma(r[p - i], a[i], rho); ra = fma(r[i], a[i], ra); }
                const double k = (r[p] - rho) / (r[0] - ra);
#pragma unroll
                for (int i = 1; 2 * i <= p; ++i) {
                    const double t1 = a[i], t2 = a[p - i];
                    a[i] = fma(-k, t2, t1);
                    if (i != p - i) a[p - i] = fma(-k, t1, t2);
                }
                a[p] = k;
            }
        }
#pragma unroll
        for (int i = 1; i <= P; ++i) a[i] = (i <= ord) ? -a[i] : 0.0;
    }
#pragma unroll
    for (int m = 0; m <= P; ++m) ap[m] = a[m];
    double q = r[0];
#pragma unroll
    for (int k = 1; k <= P; ++k) q = fma(a[k], r[k], q);
    double xt[P];  // xt[t] = windowed sample wlen - P + t
#pragma unroll
    for (int t = 0; t < P; ++t) xt[t] = xts[t];
    double tail = 0.0;
#pragma unroll
    for (int d = 0; d < P; ++d) {
        double e = 0.0;
#pragma unroll
        for (int k = d + 1; k <= P; ++k) e = fma(a[k], xt[P + d - k], e);
        tail = fma(e, e, tail);
    }
    const double E = fused ? fma(q, dw, -tail) : __dsub_rn(__dmul_rn(q, dw), tail);
    return E > 0.0 ? E : 0.0;
}

#define LV_THREADS 64

// TAB: the call's streams have different orders (g.ordTab) -- each frame is solved at its own. A separate instantiation:
// at uniform 40 / 5 the per-frame form measured 2.1 ms per step slower (21.6 vs 19.5 ms, profiles/ab_stream_orders_r06.txt).
template <int PV, int PS, bool TAB>
__global__ void __launch_bounds__(LV_THREADS) k_voc_levinson_static(VPGeom g, VPTables tb, const float* __restrict__ voice,
                                                                    const float* __restrict__ synth, const uint8_t* __restrict__ gate,
                                                                    const double* __restrict__ rV, const double* __restrict__ rS,
                                                                    double* __restrict__ aV, double* __restrict__ aS,
                                                                    double* __restrict__ EeV, double* __restrict__ EeS, long long tot) {
    constexpr int RV = 2 * PV + 1, RSY = 2 * PS + 1;  // workspace rows: lags 0..P then the last P windowed samples
    constexpr int NR = RV + RSY;
    constexpr int RS = NR | 1;                        // odd row stride in shared memory
    extern __shared__ double sm[];
    __shared__ size_t sRow[LV_THREADS];
    double* sR = sm;                                  // [LV_THREADS][RS]  rows in; the coefficient rows go out through it
    const int tid = threadIdx.x;
    const long long f0 = (long long)blockIdx.x * LV_THREADS;
    const int nF = (int)((tot - f0 < LV_THREADS) ? tot - f0 : LV_THREADS);
    const int wlen = g.wlenV;
    // ---- coalesced staging (rows of consecutive frames are contiguous in global memory)
    // asynchronous 8-byte copies: all of a thread's ~90 elements are in flight at once, no register round trip
    for (int i = tid; i < nF * RV; i += LV_THREADS) __pipeline_memcpy_async(sR + (i / RV) * RS + (i % RV), rV + f0 * RV + i, 8);
    for (int i = tid; i < nF * RSY; i += LV_THREADS) __pipeline_memcpy_async(sR + (i / RSY) * RS + RV + (i % RSY), rS + f0 * RSY + i, 8);
    __pipeline_commit();
    __pipeline_wait_prior(0);
    __syncthreads();
    if (tid < nF) {
        const long long idx = f0 + tid;
        const int s = (int)(idx / g.nFramesV), k = (int)(idx - (long long)s * g.nFramesV);
        const size_t orow = vp_vrow(g, s, k);
        sRow[tid] = orow;
        double* row = sR + tid * RS;
        const int b = (int)(((unsigned)k * (unsigned)g.hopV + (unsigned)g.offV) / (unsigned)g.B);  // block of the frame's start
        // the frame's own orders when the call's streams differ (VocoderProcess.cpp:193-194: read at the frame start)
        int pv = PV, ps = PS;
        if (TAB) { const VPStreamParam& q = vp_sp(tb, b, s); pv = q.ordV; ps = q.ordS; }
        const bool fused = pv == PV && ps == PS;  // (other orders alone run k_voc_levinson)
        const double eS = lev_energy_static<PS>(row + RV, row + RV, wlen, row + RV + PS + 1, ps, fused);
        // a frame skipped by the silence gate (VocoderProcess.cpp:199-204) is marked with EeSynth = -1: the synthesis
        // kernel then needs no gate lookups for its 10-frame energy history
        const bool gated = (gate[(size_t)s * g.nBlocks + b] & (VP_GATE_VOICE | VP_GATE_SYNTH)) != 0;
        EeS[orow] = gated ? -1.0 : eS;
        EeV[orow] = lev_energy_static<PV>(row, row, wlen, row + PV + 1, pv, fused);
    }
    __syncthreads();
    // coalesced coefficient rows out; the workspace row of each frame (carry rows per stream in front) was noted by its thread
    for (int i = tid; i < nF * (PV + 1); i += LV_THREADS) {
        const int fi = i / (PV + 1), m = i % (PV + 1);
        aV[sRow[fi] * (PV + 1) + m] = sR[fi * RS + m];
    }
    for (int i = tid; i < nF * (PS + 1); i += LV_THREADS) {
        const int fi = i / (PS + 1), m = i % (PS + 1);
        aS[sRow[fi] * (PS + 1) + m] = sR[fi * RS + RV + m];
    }
}

void vp_launch_voc_levinson(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                            const float* synth, const uint8_t* gate, const double* rV, const double* rS, double* aV,
                            double* aS, double* EeV, double* EeS) {
    const long long tot = (long long)S * g.nFramesV;
    // (a call with per-stream orders all <= 40 / <= 5 has 40 / 5 rows and takes this kernel too, in its per-frame form)
    if (g.ordV == 40 && g.ordS == 5 && g.synV == 40 && g.synS == 5 && g.wlenV >= 40)
    {
        const size_t smem = (size_t)LV_THREADS * ((vp_rowlen(40) + vp_rowlen(5)) | 1) * sizeof(double);
        const unsigned grid = (unsigned)((tot + LV_THREADS - 1) / LV_THREADS);
        if (g.ordTab) {
            cudaFuncSetAttribute(k_voc_levinson_static<40, 5, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            VP_LAUNCH(k_voc_levinson_static<40, 5, true><<<grid, LV_THREADS, smem, st>>>(g, tb, voice, synth, gate, rV, rS, aV, aS, EeV, EeS, tot));
        } else {
            cudaFuncSetAttribute(k_voc_levinson_static<40, 5, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            VP_LAUNCH(k_voc_levinson_static<40, 5, false><<<grid, LV_THREADS, smem, st>>>(g, tb, voice, synth, gate, rV, rS, aV, aS, EeV, EeS, tot));
        }
    }
    else
        VP_LAUNCH(k_voc_levinson<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(g, tb, gate, rV, rS, aV, aS, EeV, EeS, S));
}

// ---------------------------------------------------------------------------
// Gain + all-pole resynthesis + sine-window overlap-add
// (VocoderProcess.cpp:260-297). One thread per frame, one warp per tile of 32
// consecutive frames of one stream: the recursion is serial in i, so frames
// are the parallel axis. The tile's side-chain samples and its overlap-add
// accumulator live in shared memory with a +1-per-hop skew so that lanes
// (hop apart) hit distinct banks.
// ---------------------------------------------------------------------------
#define VS_WARPS 2

// Skewed shared-memory index of tile position pos = lane*hop + i: pos + sk * floor(pos / hop), sk = 1 for an even hop
// (lane stride hop + 1 odd) and 0 for an odd hop (lane stride already odd) -> lanes always hit 32 distinct banks.
__device__ __forceinline__ int vs_idx(int lane, int i, int hop, int sk) {
    return lane * hop + i + sk * (lane + (i >= hop) + (i >= 2 * hop) + (i >= 3 * hop) + (i >= 4 * hop));
}
__device__ __forceinline__ int vs_skew(int pos, int hop, int sk) { return pos + sk * (pos / hop); }

// Gain of every frame (VocoderProcess.cpp:264-276, :301-327): g = sqrt(sum EeVoice / sum EeSynth) over the last 10
// PROCESSED frames, newest first (a gated frame -- EeSynth < 0 -- neither shifts the histories nor gets a gain).
// One thread per frame scans back over this call's frames and, if the call started fewer than 10 processed frames
// ago, continues into the stream's carried histories hist[s] = {EeVoice[10], EeSynth[10]} (newest first).
__global__ void __launch_bounds__(128) k_voc_gain(VPGeom g, VPTables tb, const double* __restrict__ EeV,
                                                  const double* __restrict__ EeS, double* __restrict__ G, double* __restrict__ Gs,
                                                  const double* __restrict__ hist, long long tot) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= tot) return;
    const int s = (int)(idx / g.nFramesV), k = (int)(idx - (long long)s * g.nFramesV);
    const size_t row0 = vp_vrow(g, s, 0);
    const double es = EeS[row0 + k];
    double gain = 0.0;
    if (es > 1e-4) {
        double sv = 0.0, ss = 0.0;
        int cnt = 0;
        for (int q = k; q >= 0 && cnt < 10; --q) {
            const double eq = EeS[row0 + q];
            if (eq >= 0.0) { sv += EeV[row0 + q]; ss += eq; ++cnt; }
        }
        const double* h = hist + (size_t)s * 20;
        for (int i = 0; cnt < 10; ++i, ++cnt) { sv += h[i]; ss += h[10 + i]; }  // zero entries = "never processed"
        gain = sqrt(sv / ss);
    }
    G[row0 + k] = gain;
    // what the synthesis applies: g times the frame's own gainVoc (its stream's, read once per frame in the block the frame
    // starts in, VocoderProcess.cpp:291-294), so a frame that is finished by a later call keeps the gain of that block
    const int blk = (int)(((long long)k * g.hopV + g.offV) / g.B);
    Gs[row0 + k] = gain * (double)vp_sp(tb, blk, s).gainVocF;
}

// the carried histories after this call: the 10 newest processed frames of (old history ++ this call's frames)
__global__ void __launch_bounds__(64) k_voc_gain_carry(VPGeom g, const double* __restrict__ EeV, const double* __restrict__ EeS,
                                                       double* __restrict__ hist, int S) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const size_t row0 = vp_vrow(g, s, 0);
    double hv[10], hs[10];
    int cnt = 0;
    for (int q = g.nFramesV - 1; q >= 0 && cnt < 10; --q) {
        const double eq = EeS[row0 + q];
        if (eq >= 0.0) { hv[cnt] = EeV[row0 + q]; hs[cnt] = eq; ++cnt; }
    }
    double* h = hist + (size_t)s * 20;
    for (int i = 0; cnt < 10; ++i, ++cnt) { hv[cnt] = h[i]; hs[cnt] = h[10 + i]; }
    for (int i = 0; i < 10; ++i) { h[i] = hv[i]; h[10 + i] = hs[i]; }
}

void vp_launch_voc_gain(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const double* EeV, const double* EeS, double* G,
                        double* Gs, double* hist) {
    const long long tot = (long long)S * g.nFramesV;
    if (tot > 0) VP_LAUNCH(k_voc_gain<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(g, tb, EeV, EeS, G, Gs, hist, tot));
    VP_LAUNCH(k_voc_gain_carry<<<(S + 63) / 64, 64, 0, st>>>(g, EeV, EeS, hist, S));
}

// ---------------------------------------------------------------------------
// Lock-step streaming synthesis (default for row orders 40 / 5). wlen = 4 hop, so exactly four frames overlap any output
// position. A group of 4 lanes owns one stream, lane phase phi runs the frames k = phi (mod 4) back to back, and all four
// lanes step through the SAME output position t in lock step:
//   * the overlap-add out[t] = sum of the four lanes' windowed outputs is a transpose-reduce of three shuffles per four
//     positions -- no accumulator buffer, no atomics, no pre-zeroed output, every position written exactly once,
//   * coefficients are (re)loaded once per frame, states restart at zero (VocoderProcess.cpp:243-247, :280-285); the
//     recursion is in transposed direct form II: P independent DFMAs per sample, states and coefficients in registers.
// A warp = 8 streams x one segment of frames; a segment starts 3 rows early (the 3 frames that still overlap its first
// position) and only emits its own positions.
// Round 2 rebuilt the step (round 1: k_voc_synth_stream, same arithmetic -- FIR32 = false is bit-identical to it; 146.7 ->
// 103 ms per step of the default workload) around what the pipe microbenchmark
// (tools/ubench_mix.cu, profiles/ubench_mix_r02a.txt) measured on the B200: next to DFMAs NO other instruction issues for
// free -- an FFMA, an integer op or a load each cost their own issue cycle, an F2F about 2.7 -- so the step is trimmed to
// its 40 + 6 DFMAs plus the fewest possible other instructions:
//   * the side-chain samples of a hop-row (8 streams x hop floats per warp) are copied global -> shared by cp.async one
//     row ahead (each lane copies a quarter of its stream's row: 0.25 copy instructions per sample instead of one load
//     with 64-bit address arithmetic and range tests), and a block of 4 positions reads them with ONE 128-bit load;
//   * window rows are padded so that a block reads its 4 weights with 128-bit loads at immediate offsets;
//   * frame parameters land in one zone per STREAM (only one of a stream's four phases starts a frame per row), copied by
//     the stream's four lanes together;
//   * segments are sized so that the grid is a whole number of waves of resident CTAs (the round-1 launch left a third,
//     nearly empty wave).
// FIR32 = true moves the order-PS whitening FIR and both window multiplies to the idle FP32 pipe (the all-pole recursion,
// its state and its input sum stay FP64); SURVEY.md App. C.4 measured that split at >= 117 dB on the clean voice.
// ---------------------------------------------------------------------------
#define VR_WARPS 2

__host__ __device__ inline int vr_pad4odd(int n) {  // smallest multiple of 4 with an odd quotient, >= n rounded up to 4
    int q = (n + 3) >> 2;
    if ((q & 1) == 0) ++q;
    return 4 * q;
}

template <int P, int PS, bool FIR32>
__global__ void __launch_bounds__(32 * VR_WARPS) k_voc_synth_rows(VPGeom g, VPTables tb, const float* __restrict__ synth,
                                                                  const double* __restrict__ aV, const double* __restrict__ aS,
                                                                  const double* __restrict__ EeS, const double* __restrict__ G,
                                                                  float* __restrict__ outV, int S, int nSeg, int segFrames,
                                                                  int wPad, int xPad, int wsOff) {
    using WT = typename std::conditional<FIR32, float, double>::type;  // window / FIR arithmetic type
    extern __shared__ __align__(16) unsigned char vr_smem[];
    constexpr int CF_AS = P + 1, CF_G = P + PS + 2, CF_ES = CF_G + 1, CF_N = CF_ES + 1;
    constexpr int CF_STRIDE = CF_N | 1;  // odd stride: the 64-bit reads of a warp's 8 zones hit distinct banks
    const int hop = g.hopV;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float* xsAll = reinterpret_cast<float*>(vr_smem);                         // [VR_WARPS][2][8][xPad] side-chain rows
    // [4][wPad] analysis-window rows, then -- wsOff != 0: the "hann" window type, whose synthesis window differs
    // (VocoderProcess.cpp:116-124) -- [4][wPad] synthesis-window rows; for "sine" both are the same table
    WT* wv = reinterpret_cast<WT*>(xsAll + (size_t)VR_WARPS * 2 * 8 * xPad);
    double* cfAll = reinterpret_cast<double*>(wv + (size_t)4 * wPad + wsOff);  // [VR_WARPS][8][CF_STRIDE] frame parameters
    for (int i = threadIdx.x; i < 4 * wPad; i += blockDim.x) {
        const int r = i / wPad, c = i - r * wPad;
        wv[i] = (c < hop) ? (WT)tb.wV[r * hop + c] : (WT)0;
        if (wsOff) wv[wsOff + i] = (c < hop) ? (WT)tb.wS[r * hop + c] : (WT)0;
    }
    __syncthreads();
    const long long wid = (long long)blockIdx.x * VR_WARPS + warp;
    const int groups = (S + 7) / 8;
    if (wid >= (long long)groups * nSeg) return;
    const int grp = (int)(wid / nSeg), seg = (int)(wid - (long long)grp * nSeg);
    const int phi = lane & 3, j8 = lane >> 2;
    int s = grp * 8 + j8;
    const bool sOk = s < S;
    if (!sOk) s = S - 1;  // idle group: runs along on a valid stream, stores are masked
    // rows / segments exactly as in k_voc_synth_stream
    const int kS = seg * segFrames;
    const int nRowsAll = (int)((g.n - g.offV + hop - 1) / hop);
    if (seg > 0 && kS >= nRowsAll) return;
    const bool lastSeg = (seg == nSeg - 1) || (kS + segFrames >= nRowsAll);
    const int kE = lastSeg ? nRowsAll : kS + segFrames;
    const long long emit0 = (seg == 0) ? 0 : (long long)kS * hop + g.offV;
    const long long emit1 = lastSeg ? g.n : (long long)kE * hop + g.offV;
    const int rho0 = (seg == 0) ? -VP_VC : kS - 3;
    const VPRow y = vp_row(synth, g.histS, s, g);
    float* o = outV + (size_t)s * g.vstride;
    double* cf = cfAll + ((size_t)warp * 8 + j8) * CF_STRIDE;
    float* xs0 = xsAll + ((size_t)(warp * 2) * 8 + j8) * xPad;  // this stream's row, buffer 0; buffer 1 is 8 xPad further
    const int xbuf = 8 * xPad;
    double a[P + 1], st[P + 1];
    WT as[PS + 1], t[PS + 1];
#pragma unroll
    for (int j = 0; j <= P; ++j) { a[j] = 0.0; st[j] = 0.0; }
#pragma unroll
    for (int j = 0; j <= PS; ++j) { as[j] = (WT)0; t[j] = (WT)0; }
    int wrow = 0;
    auto frameOk = [&](int k) { return k + g.kV0 >= 0 && k < g.nFramesV; };
    // ---- asynchronous copies for row r: the stream's hop side-chain samples (this lane: positions phi, phi + 4, ...) and,
    // by the stream's four lanes together, the parameters of the frame that starts at row r
    auto stage = [&](int r, int buf) {
        float* dst = xs0 + buf * xbuf;
        const long long tIn = (long long)r * hop + g.offV - g.lat;  // input index of the row's first position
        if (tIn >= 0 && tIn + hop <= g.n) {
            const float* src = y.x + tIn;
#pragma unroll 4
            for (int i = phi; i < hop; i += 4) __pipeline_memcpy_async(dst + i, src + i, 4);
        } else {  // history before the call / beyond its input: plain stores (the __syncwarp after the wait orders them)
            const long long u0 = (long long)r * hop + g.offV;
            for (int i = phi; i < hop; i += 4) dst[i] = vp_x(y, u0 + i, g);
        }
        if (frameOk(r)) {
            const size_t row = vp_vrow(g, s, r);
            const double* ap = aV + row * (P + 1);
            const double* sp = aS + row * (PS + 1);
#pragma unroll
            for (int q0 = 0; q0 < CF_N; q0 += 4) {
                const int q = q0 + phi;
                if (q < CF_N) {
                    const double* src = (q <= P) ? ap + q : (q < CF_G) ? sp + (q - CF_AS) : (q == CF_G) ? G + row : EeS + row;
                    __pipeline_memcpy_async(cf + q, src, 8);
                }
            }
        }
        __pipeline_commit();
    };
    stage(rho0, 0);
    int cur = 0;
    for (int rho = rho0; rho < kE; ++rho, cur ^= 1) {
        __pipeline_wait_prior(0);
        __syncwarp();
        // ---- frame start for the phase that begins at this row
        if (((rho + 4 * VP_VC) & 3) == phi) {
#pragma unroll
            for (int j = 0; j <= P; ++j) st[j] = 0.0;
#pragma unroll
            for (int j = 0; j <= PS; ++j) t[j] = (WT)0;
            const bool active = frameOk(rho) && cf[CF_ES] >= 0.0;  // a gated frame carries EeSynth < 0
            if (active) {
                const double gain = cf[CF_G];
#pragma unroll
                for (int j = 1; j <= P; ++j) a[j] = cf[j];
#pragma unroll
                for (int j = 0; j <= PS; ++j) as[j] = (WT)(gain * cf[CF_AS + j]);  // gain folded into the FIR taps
            } else {
#pragma unroll
                for (int j = 1; j <= P; ++j) a[j] = 0.0;
#pragma unroll
                for (int j = 0; j <= PS; ++j) as[j] = (WT)0;
            }
            wrow = 0;
        }
        __syncwarp();  // the zone has been read before the next frame's parameters are copied into it
        if (rho + 1 < kE) stage(rho + 1, cur ^ 1);
        const float* xr = xs0 + cur * xbuf;
        const WT* wr = wv + wrow * wPad;
        const WT* wo = wr + wsOff;  // synthesis-window row
        const long long tBase = (long long)rho * hop + g.offV;
        const bool rowEmit = sOk && tBase >= emit0 && tBase + hop <= emit1;  // whole row inside the emission range
        const int nblk = (hop + 3) >> 2;
        const int nFull = hop >> 2;  // full blocks of 4 positions; block nFull (if any) is the row's partial last block
        // The row body exists twice: EALL = every position of the row is emitted (steady state: stores are plain
        // pointer + immediate, no range test) and the general form (segment halo rows, first / last rows of a call).
        auto rowBody = [&](auto emitTag) {
            constexpr bool EALL = decltype(emitTag)::value;
            float* op = o + tBase + phi;  // this lane's position in block 0
            WT eA[4], eB[4];
            float cA[4], cB[4];
            // whitening FIR (transposed form) of the block at row offset i1 with nb1 valid positions -> e
            auto fir = [&](auto fullTag, WT* e, int i1, int nb1) {
                constexpr bool FULL = decltype(fullTag)::value;
                const float4 x4 = *reinterpret_cast<const float4*>(xr + i1);
                const float xv[4] = {x4.x, x4.y, x4.z, x4.w};
                WT w4[4];
                if (FIR32) {
                    const float4 q = *reinterpret_cast<const float4*>(wr + i1);
                    w4[0] = (WT)q.x; w4[1] = (WT)q.y; w4[2] = (WT)q.z; w4[3] = (WT)q.w;
                } else {
                    const double2 q0 = *reinterpret_cast<const double2*>(wr + i1), q1 = *reinterpret_cast<const double2*>(wr + i1 + 2);
                    w4[0] = (WT)q0.x; w4[1] = (WT)q0.y; w4[2] = (WT)q1.x; w4[3] = (WT)q1.y;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    e[j] = (WT)0;
                    if (FULL || j < nb1) {
                        const WT x = (WT)xv[j] * w4[j];
                        e[j] = fma(as[0], x, t[0]);
#pragma unroll
                        for (int qq = 0; qq < PS; ++qq) t[qq] = fma(as[qq + 1], x, t[qq + 1]);
                    }
                }
            };
            // all-pole recursion of the block at row offset i0 (transposed direct form II: P independent DFMAs per sample)
            auto iir = [&](auto fullTag, const WT* e, float* c, int i0, int nb) {
                constexpr bool FULL = decltype(fullTag)::value;
                WT w4[4];
                if (FIR32) {
                    const float4 q = *reinterpret_cast<const float4*>(wo + i0);
                    w4[0] = (WT)q.x; w4[1] = (WT)q.y; w4[2] = (WT)q.z; w4[3] = (WT)q.w;
                } else {
                    const double2 q0 = *reinterpret_cast<const double2*>(wo + i0), q1 = *reinterpret_cast<const double2*>(wo + i0 + 2);
                    w4[0] = (WT)q0.x; w4[1] = (WT)q0.y; w4[2] = (WT)q1.x; w4[3] = (WT)q1.y;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (FULL || j < nb) {
                        const double ov = (double)e[j] + st[0];
#pragma unroll
                        for (int kk = 0; kk < P; ++kk) st[kk] = fma(-a[kk + 1], ov, st[kk + 1]);
                        if (FIR32) c[j] = (float)ov * (float)w4[j];
                        else c[j] = (float)(ov * (double)w4[j]);
                    } else c[j] = 0.0f;
                }
            };
            // overlap-add of the 4 phase lanes for the 4 positions of the block at row offset iP (nbP valid positions):
            // transpose-reduce, 3 shuffles; lane phi ends with the sum over the group for position iP + phi
            auto ola = [&](const float* c, int iP, int nbP) {
                const bool hi = (phi & 2) != 0, od = (phi & 1) != 0;
                const float s0 = hi ? c[0] : c[2], s1 = hi ? c[1] : c[3];
                const float k0 = hi ? c[2] : c[0], k1 = hi ? c[3] : c[1];
                const float r0 = k0 + __shfl_xor_sync(0xffffffffu, s0, 2);
                const float r1 = k1 + __shfl_xor_sync(0xffffffffu, s1, 2);
                const float snd = od ? r0 : r1, kp = od ? r1 : r0;
                const float tot = kp + __shfl_xor_sync(0xffffffffu, snd, 1);
                if (EALL) {
                    if (nbP == 4 || phi < nbP) op[iP] = tot;
                } else {
                    const long long tp = tBase + iP + phi;
                    if (sOk && phi < nbP && tp >= emit0 && tp < emit1) op[iP] = tot;
                }
            };
            // step k: recursion of block k (its FIR output is in e), overlap-add + store of block k - 1 (its shuffle
            // latencies hide under the recursion), then the FIR of block k + 1 into the same e (each e[j] is dead as soon as
            // sample j entered the recursion, so one set of registers serves both). Even k writes cA, odd k cB.
            WT* const e = eA;
            (void)eB;
            int k = 0;
            if (nFull >= 2) {
                fir(std::true_type{}, e, 0, 4);
                iir(std::true_type{}, e, cA, 0, 4);
                fir(std::true_type{}, e, 4, 4);
                k = 1;
                for (; k + 2 < nFull; k += 2) {  // blocks k, k + 1, k + 2 are full
                    iir(std::true_type{}, e, cB, 4 * k, 4);
                    ola(cA, 4 * k - 4, 4);
                    fir(std::true_type{}, e, 4 * k + 4, 4);
                    iir(std::true_type{}, e, cA, 4 * k + 4, 4);
                    ola(cB, 4 * k, 4);
                    fir(std::true_type{}, e, 4 * k + 8, 4);
                }
            } else {
                fir(std::false_type{}, e, 0, min(4, hop));
            }
            // remaining blocks (at most 3 + the partial one), parity tracked at run time; k = next block to run through the
            // recursion (its FIR output is in e); block k - 1 (if k > 0) awaits its overlap-add
            for (; k < nblk; ++k) {
                const int nb = min(4, hop - 4 * k), nb1 = min(4, hop - 4 * k - 4);
                if (k & 1) {
                    iir(std::false_type{}, e, cB, 4 * k, nb);
                    ola(cA, 4 * k - 4, 4);
                } else {
                    iir(std::false_type{}, e, cA, 4 * k, nb);
                    if (k > 0) ola(cB, 4 * k - 4, 4);
                }
                if (k + 1 < nblk) fir(std::false_type{}, e, 4 * k + 4, nb1);
            }
            {   // drain: the row's last block
                const int kl = nblk - 1;
                ola((kl & 1) ? cB : cA, 4 * kl, min(4, hop - 4 * kl));
            }
        };
        if (rowEmit) rowBody(std::true_type{});
        else rowBody(std::false_type{});
        ++wrow;
    }
}

// Generic-order fallback (orders other than the plug-in defaults): same tiling,
// histories in local memory.
__global__ void __launch_bounds__(32 * VS_WARPS) k_voc_synth_generic(VPGeom g, VPTables tb, const float* __restrict__ synth,
                                                                     const double* __restrict__ aV,
                                                                     const double* __restrict__ aS,
                                                                     const double* __restrict__ EeS,
                                                                     const double* __restrict__ G, float* __restrict__ outV,
                                                                     int tilesPerStream, int S, int spanPad, int sk) {
    extern __shared__ float smf[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long tile = (long long)blockIdx.x * VS_WARPS + warp;
    const bool live = tile < (long long)tilesPerStream * S;
    const int s = live ? (int)(tile / tilesPerStream) : 0;
    // tiles start VP_VC frames early: the previous call's last frames (carry rows) still reach into this call
    const int k0 = (live ? (int)(tile - (long long)s * tilesPerStream) * 32 : 0) - VP_VC;
    const int P = g.synV, PS = g.synS;  // row orders (>= the frames' own analysis orders; rows are zero padded)
    float* sbuf = smf + (size_t)warp * 2 * spanPad;
    float* obuf = sbuf + spanPad;
    const int hop = g.hopV, wlen = g.wlenV;
    const int span = 31 * hop + wlen;
    const VPRow y = vp_row(synth, g.histS, s, g);
    const long long uBase = (long long)k0 * hop + g.offV;
    if (live) {
        for (int i = lane; i < span; i += 32) sbuf[vs_skew(i, hop, sk)] = vp_x(y, uBase + i, g);
        for (int i = lane; i < span; i += 32) obuf[vs_skew(i, hop, sk)] = 0.0f;
    }
    __syncwarp();
    const int k = k0 + lane;
    const size_t fidx = vp_vrow(g, s, k);
    bool active = live && k < g.nFramesV && k + g.kV0 >= 0;
    if (active && EeS[fidx] < 0.0) active = false;  // gated frame (marked by the Levinson kernel)
    const double gain = active ? G[fidx] : 0.0;
    const double* ap = aV + fidx * (size_t)(P + 1);
    const double* sp = aS + fidx * (size_t)(PS + 1);
    double h[VP_ORDER_MAX];
    for (int j = 0; j < P; ++j) h[j] = 0.0;
    for (int i = 0; i < wlen; ++i) {
        const double w = tb.wS[i];
        double o = 0.0;
        if (active) {
            double e = 0.0;
            for (int q = 0; q <= PS && q <= i; ++q)
                e = fma(sp[q], (double)sbuf[vs_idx(lane, i - q, hop, sk)] * tb.wV[i - q], e);
            o = gain * e;
            for (int kk = 1; kk <= P && kk <= i; ++kk) o = fma(-ap[kk], h[(i - kk) % P], o);
            h[i % P] = o;
            obuf[vs_idx(lane, i, hop, sk)] += (float)(o * w);
        }
        if ((i & 31) == 31) __syncwarp();
    }
    __syncwarp();
    if (live) {
        float* o = outV + (size_t)s * g.vstride;
        const int ov = wlen - hop;
        for (int i = lane; i < span; i += 32) {
            const long long u = uBase + i;
            if (u >= g.n) break;
            if (u < 0) continue;
            const float v = obuf[vs_skew(i, hop, sk)];
            if (i < ov || i >= 32 * hop) atomicAdd(o + u, v);
            else o[u] = v;
        }
    }
}

bool vp_voc_synth_needs_clear(const VPGeom& g) { return !(g.synV == 40 && g.synS == 5); }

// ---------------------------------------------------------------------------
// Frames of earlier calls that are off this call's frame grid (VPGeom::orphPos): finished from their carried rows, one
// thread per stream, frames in slot order, added to the plane the grid kernel has already written. Rare (only around a
// vocBool toggle) and short (at most 4 live frames per stream), so it is written for clarity: the same transposed-form
// FIR + IIR with the states in local memory.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(64) k_voc_orphans(VPGeom g, VPTables tb, const float* __restrict__ synth,
                                                    const double* __restrict__ oAV, const double* __restrict__ oAS,
                                                    const double* __restrict__ oEeS, const double* __restrict__ oG,
                                                    float* __restrict__ outV, int S, int capV, int capS) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const VPRow y = vp_row(synth, g.histS, s, g);
    float* o = outV + (size_t)s * g.vstride;
    double st[VP_ORDER_MAX + 1], t[32];
    for (int j = 0; j < VP_ORPH; ++j) {
        const int pos = g.orphPos[j];
        if (pos == VP_NOFRAME || pos + g.wlenV <= 0 || pos >= g.n) continue;
        const size_t slot = (size_t)s * VP_ORPH + j;
        if (oEeS[slot] < 0.0) continue;  // gated frame
        const int P = g.orphOrdV[j], PS = g.orphOrdS[j];
        const double* a = oAV + slot * (size_t)(capV + 1);
        const double* as = oAS + slot * (size_t)(capS + 1);
        const double gain = oG[slot];
        for (int k = 0; k <= P; ++k) st[k] = 0.0;
        for (int k = 0; k <= PS; ++k) t[k] = 0.0;
        for (int i = 0; i < g.wlenV; ++i) {
            const long long u = (long long)pos + i;
            if (u >= g.n) break;
            const double x = (double)vp_x(y, u, g) * tb.wV[i];
            const double w = tb.wS[i];
            const double e = fma(gain * as[0], x, t[0]);
            for (int q = 0; q < PS; ++q) t[q] = fma(gain * as[q + 1], x, t[q + 1]);
            const double ov = e + st[0];
            for (int k = 0; k < P; ++k) st[k] = fma(-a[k + 1], ov, st[k + 1]);
            if (u >= 0) o[u] += (float)(ov * w);
        }
    }
}

void vp_launch_voc_orphans(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* synth, const double* oAV,
                           const double* oAS, const double* oEeS, const double* oG, float* outV, int capV, int capS) {
    VP_LAUNCH(k_voc_orphans<<<(S + 63) / 64, 64, 0, st>>>(g, tb, synth, oAV, oAS, oEeS, oG, outV, S, capV, capS));
}

// segments per stream group such that the grid is (at most) `waves` full waves of resident warps. Measured on the default
// workload (ms per step of this kernel): 1 wave 126.8, 2 waves 109.3, 3 waves 105.4, 4 waves 103.0 -- shorter segments let
// the hardware's CTA scheduler even out the warps' run times; the 3-row halo of a segment stays below 1 %
static int vs_segments(const VPGeom& g, int groups, int residentWarps, int* segFramesOut) {
    static int waves = 0;
    if (waves == 0) { const char* w = getenv("VP_SYNTH_WAVES"); waves = (w && atoi(w) > 0) ? atoi(w) : 4; }
    int nSeg = (waves * residentWarps) / groups;                        // whole waves of resident warps: the last one (nearly) full
    if (nSeg < 1) nSeg = 1;
    int segFrames = (g.nFramesV + nSeg - 1) / nSeg;
    if (segFrames < 16) segFrames = 16;                                  // keep the 3-row halo a small fraction
    nSeg = (g.nFramesV + segFrames - 1) / segFrames;
    if (nSeg < 1) nSeg = 1;                                              // no new frame: the carried frames still emit
    *segFramesOut = segFrames;
    return nSeg;
}

template <bool FIR32>
static void launch_synth_rows(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* synth,
                              const double* aV, const double* aS, const double* EeS, const double* G, float* outV) {
    auto kern = k_voc_synth_rows<40, 5, FIR32>;
    const int groups = (S + 7) / 8;
    const int nblk = (g.hopV + 3) >> 2;
    const int xPad = vr_pad4odd(g.hopV);
    int wPad;
    if (FIR32) wPad = vr_pad4odd(g.hopV);
    else { wPad = 4 * nblk; if (((wPad >> 1) & 1) == 0) wPad += 2; }     // doubles: 16-byte rows, row stride / 16 B odd
    const int cfStride = (40 + 1 + 5 + 1 + 2) | 1;
    const int wsOff = (tb.wS != tb.wV) ? 4 * wPad : 0;  // "hann": a second table for the synthesis window
    const size_t smem = (size_t)VR_WARPS * 2 * 8 * xPad * sizeof(float) + (size_t)(4 * wPad + wsOff) * (FIR32 ? sizeof(float) : sizeof(double)) +
                        (size_t)VR_WARPS * 8 * cfStride * sizeof(double);
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    int perSM = 4, dev = 0, nSM = 148;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, kern, 32 * VR_WARPS, smem);
    if (perSM < 1) perSM = 1;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nSM, cudaDevAttrMultiProcessorCount, dev);
    int segFrames = 0;
    const int nSeg = vs_segments(g, groups, nSM * perSM * VR_WARPS, &segFrames);
    const long long warps = (long long)groups * nSeg;
    VP_LAUNCH(kern<<<(unsigned)((warps + VR_WARPS - 1) / VR_WARPS), 32 * VR_WARPS, smem, st>>>(
        g, tb, synth, aV, aS, EeS, G, outV, S, nSeg, segFrames, wPad, xPad, wsOff));
}

// VP_SYNTH = rows (default) | rows32 (FP32 whitening FIR + window multiplies: 102.5 vs 109.3 ms per step at 2 waves, worst
// stream 124 dB instead of 146 dB against the reference) | generic (the any-order kernel, for A/B)
static int vs_variant() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("VP_SYNTH");
        v = (e && strcmp(e, "generic") == 0) ? 2 : (e && strcmp(e, "rows32") == 0) ? 1 : 0;
    }
    return v;
}

void vp_launch_voc_synth(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* synth,
                         const double* aV, const double* aS, const double* EeS, const double* G, float* outV) {
    if (g.synV == 40 && g.synS == 5 && vs_variant() != 2 && g.hopV >= 8) {
        if (vs_variant() == 1) launch_synth_rows<true>(st, g, tb, S, synth, aV, aS, EeS, G, outV);
        else launch_synth_rows<false>(st, g, tb, S, synth, aV, aS, EeS, G, outV);
        return;
    }
    const int tilesPerStream = (g.nFramesV + VP_VC + 31) / 32;
    const int span = 31 * g.hopV + g.wlenV + VP_ORDER_MAX;
    const int sk = (g.hopV & 1) ? 0 : 1;
    int spanPad = span + span / g.hopV + 8;
    spanPad = (spanPad + 31) & ~31;
    const long long tiles = (long long)tilesPerStream * S;
    const unsigned grid = (unsigned)((tiles + VS_WARPS - 1) / VS_WARPS);
    const size_t smem = (size_t)VS_WARPS * 2 * spanPad * sizeof(float);
    cudaFuncSetAttribute(k_voc_synth_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    VP_LAUNCH(k_voc_synth_generic<<<grid, 32 * VS_WARPS, smem, st>>>(g, tb, synth, aV, aS, EeS, G, outV, tilesPerStream, S, spanPad, sk));
}
