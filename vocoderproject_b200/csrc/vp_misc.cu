// Mix/egress, synthetic-input generation and issue-rate microbenchmarks.
#include <algorithm>

#include "vp_common.cuh"
#include "vp_synth.h"

// ---------------------------------------------------------------------------
// Mix + egress (PluginProcessor.cpp:226-232, MyBuffer.cpp:113-133, :309-448):
// out = vocoder OLA + pitch OLA (+ gainVoice * delayed voice) (+ gainSynth *
// delayed synth), cast to float. Output sample u carries input time u - latency.
// ---------------------------------------------------------------------------
// Each stream mixes with its own dry gains, those of the output sample's block (PluginProcessor.cpp:226-230 reads them per
// block); a path that is off adds nothing (not 0 * x, which would turn -0 into +0).
__global__ void __launch_bounds__(256) k_mix(VPGeom g, VPTables tb, const float* __restrict__ voice,
                                             const float* __restrict__ synthL, const float* __restrict__ synthR,
                                             const float* __restrict__ outV, const float* __restrict__ outP,
                                             float* __restrict__ outL, float* __restrict__ outR) {
    const int s = blockIdx.y;
    const VPStreamParam p0 = tb.sp[s];
    const bool perBlock = tb.spStride != 0;
    const size_t row = (size_t)s * g.stride, wrow = (size_t)s * g.wstride;
    const long long step = (long long)gridDim.x * blockDim.x;
    constexpr int MU = 4;  // independent loads in flight per thread and plane
    for (long long u0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; u0 < g.n; u0 += step * MU) {
        float a[MU], b[MU];
#pragma unroll
        for (int k = 0; k < MU; ++k) {
            const long long u = u0 + k * step;
            a[k] = (g.vocMix && u < g.n) ? __ldg(outV + wrow + u) : 0.0f;
            b[k] = (g.pitchMix && u < g.n) ? __ldg(outP + wrow + u) : 0.0f;
        }
#pragma unroll
        for (int k = 0; k < MU; ++k) {
            const long long u = u0 + k * step;
            if (u >= g.n) break;
            float l = 0.0f;
            if (g.vocMix) l += a[k];
            if (g.pitchMix) l += b[k];
            float r = l;
            const VPStreamParam p = perBlock ? vp_sp(tb, (int)(u / g.B), s) : p0;
            if (p.dryOn) {
                const float d = p.gainVoiceF * vp_x(vp_row(voice, g.histV, s, g), u, g);
                l += d; r += d;
            }
            if (p.synthOn) {
                l += p.gainSynthF * vp_x(vp_row(synthL, g.histS, s, g), u, g);
                r += p.gainSynthF * (synthR ? vp_x(vp_row(synthR, g.histR, s, g), u, g) : vp_x(vp_row(synthL, g.histS, s, g), u, g));
            }
            outL[row + u] = l;
            if (outR) outR[row + u] = r;
        }
    }
}

// The common case -- no stream of the call with a dry path on, rows 16-byte aligned -- as 128-bit accesses with 32-bit indexing inside a row: 4 output
// samples per thread and iteration for 2 loads, 4 adds and 1 (2) stores; the general kernel above spends ~57 instructions
// per sample on 64-bit index arithmetic (ncu, profiles/ncu_mix_r02e.json), 2.9 % of the whole step's instruction issue.
template <bool VOC, bool PITCH>
__global__ void __launch_bounds__(256) k_mix4(const float4* __restrict__ outV, const float4* __restrict__ outP, float4* __restrict__ outL,
                                              float4* __restrict__ outR, int n4, int stride4, int wstride4) {
    const int s = blockIdx.y;
    const float4* a = outV + (size_t)s * wstride4;
    const float4* b = outP + (size_t)s * wstride4;
    float4* l = outL + (size_t)s * stride4;
    float4* r = outR ? outR + (size_t)s * stride4 : nullptr;
    const int step = gridDim.x * blockDim.x;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += 2 * step) {
        const int i2 = i + step;
        const bool two = i2 < n4;
        float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0, p0 = v0, p1 = v0;
        if (VOC) { v0 = __ldg(a + i); if (two) v1 = __ldg(a + i2); }
        if (PITCH) { p0 = __ldg(b + i); if (two) p1 = __ldg(b + i2); }
        // (0 + voc) + pitch, the order of the general kernel: bit-identical
        const float4 o0 = make_float4((0.0f + v0.x) + p0.x, (0.0f + v0.y) + p0.y, (0.0f + v0.z) + p0.z, (0.0f + v0.w) + p0.w);
        l[i] = o0;
        if (r) r[i] = o0;
        if (two) {
            const float4 o1 = make_float4((0.0f + v1.x) + p1.x, (0.0f + v1.y) + p1.y, (0.0f + v1.z) + p1.z, (0.0f + v1.w) + p1.w);
            l[i2] = o1;
            if (r) r[i2] = o1;
        }
    }
}

void vp_launch_mix(cudaStream_t st, const VPGeom& g, const VPTables& tb, bool anyDry, int S, const float* voice, const float* synthL,
                   const float* synthR, const float* outV, const float* outP, float* outL, float* outR) {
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    if (!anyDry && (g.n & 3) == 0 && (g.stride & 3) == 0 && (g.wstride & 3) == 0 && g.n / 4 < (1LL << 30) && al16(outV) &&
        al16(outP) && al16(outL) && al16(outR)) {
        const int n4 = (int)(g.n / 4);
        int bx = (n4 + 2 * 256 - 1) / (2 * 256);
        if (bx > 2048) bx = 2048;
        if (bx < 1) bx = 1;
        dim3 grid((unsigned)bx, S);
        const float4 *a = reinterpret_cast<const float4*>(outV), *b = reinterpret_cast<const float4*>(outP);
        float4 *l = reinterpret_cast<float4*>(outL), *r = reinterpret_cast<float4*>(outR);
        const int s4 = (int)(g.stride / 4), w4 = (int)(g.wstride / 4);
        if (g.vocMix && g.pitchMix) VP_LAUNCH(k_mix4<true, true><<<grid, 256, 0, st>>>(a, b, l, r, n4, s4, w4));
        else if (g.vocMix) VP_LAUNCH(k_mix4<true, false><<<grid, 256, 0, st>>>(a, b, l, r, n4, s4, w4));
        else if (g.pitchMix) VP_LAUNCH(k_mix4<false, true><<<grid, 256, 0, st>>>(a, b, l, r, n4, s4, w4));
        else VP_LAUNCH(k_mix4<false, false><<<grid, 256, 0, st>>>(a, b, l, r, n4, s4, w4));
        return;
    }
    long long bx = (g.n + 4 * 256 - 1) / (4 * 256);
    if (bx > 4096) bx = 4096;
    if (bx < 1) bx = 1;
    dim3 grid((unsigned)bx, S);
    VP_LAUNCH(k_mix<<<grid, 256, 0, st>>>(g, tb, voice, synthL, synthR, outV, outP, outL, outR));
}

// ---------------------------------------------------------------------------
// Block-indexed parameter table of a call with scheduled changes (vp_engine_schedule_stream_params): out[b][s] = the value
// stream s has in force at call-local block b -- its last event at or before b, else its value at the call's start cur[s].
// Grid: x over streams (a warp writes 32 consecutive 32-byte entries of one block row), y over tiles of EX_TILE blocks; a
// thread finds the value at its tile's start by binary search in its stream's events and walks the tile.
// ---------------------------------------------------------------------------
#define EX_TILE 64
__global__ void __launch_bounds__(128) k_expand_stream_params(const VPStreamParam* __restrict__ cur, const int* __restrict__ off,
                                                              const int* __restrict__ evBlk, const VPStreamParam* __restrict__ evVal,
                                                              VPStreamParam* __restrict__ out, int S, int nBlocks) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    const int b0 = blockIdx.y * EX_TILE, b1 = min(b0 + EX_TILE, nBlocks);
    const int k0 = off[s], k1 = off[s + 1];
    int lo = k0, hi = k1;  // first event after b0
    while (lo < hi) {
        const int m = (lo + hi) >> 1;
        if (evBlk[m] <= b0) lo = m + 1;
        else hi = m;
    }
    VPStreamParam v = (lo > k0) ? evVal[lo - 1] : cur[s];
    int k = lo;
    for (int b = b0; b < b1; ++b) {
        if (k < k1 && evBlk[k] == b) v = evVal[k++];
        out[(size_t)b * S + s] = v;
    }
}
void vp_launch_expand_stream_params(cudaStream_t st, const VPStreamParam* cur, const int* off, const int* evBlk,
                                    const VPStreamParam* evVal, VPStreamParam* out, int S, int nBlocks) {
    const dim3 grid((unsigned)((S + 127) / 128), (unsigned)((nBlocks + EX_TILE - 1) / EX_TILE));
    VP_LAUNCH(k_expand_stream_params<<<grid, 128, 0, st>>>(cur, off, evBlk, evVal, out, S, nBlocks));
}

// ---------------------------------------------------------------------------
// Carried per-stream state between calls (consecutive process calls = consecutive processBlock calls).
// A frame-indexed workspace array holds, per stream, C carry rows followed by the rows of this call. carry_in copies the
// stream's C stored rows in front; carry_out stores the LAST C rows of (carry ++ new) = rows [nNew, nNew + C).
// Rows are counted in 4-byte words.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_carry_in(uint32_t* __restrict__ ws, const uint32_t* __restrict__ carry, int S,
                                                  int wsWords, int cWords, int C, long long wsRowsPerStream) {
    const long long tot = (long long)S * C * wsWords;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
        const int s = (int)(i / ((long long)C * wsWords));
        const long long r = i - (long long)s * C * wsWords;
        const int row = (int)(r / wsWords), w = (int)(r - (long long)row * wsWords);
        ws[(size_t)s * wsRowsPerStream * wsWords + r] = (w < cWords) ? carry[((size_t)s * C + row) * cWords + w] : 0u;
    }
}
__global__ void __launch_bounds__(256) k_carry_out(uint32_t* __restrict__ carry, const uint32_t* __restrict__ ws, int S,
                                                   int wsWords, int cWords, int C, long long nNew, long long wsRowsPerStream) {
    const long long tot = (long long)S * C * cWords;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
        const int s = (int)(i / ((long long)C * cWords));
        const long long r = i - (long long)s * C * cWords;
        const int row = (int)(r / cWords), w = (int)(r - (long long)row * cWords);
        carry[i] = (w < wsWords) ? ws[((size_t)s * wsRowsPerStream + nNew + row) * wsWords + w] : 0u;
    }
}
void vp_launch_carry_in(cudaStream_t st, void* ws, const void* carry, int S, int wsRowBytes, int carryRowBytes, int C,
                        long long wsRowsPerStream) {
    const long long tot = (long long)S * C * (wsRowBytes / 4);
    if (tot <= 0) return;
    VP_LAUNCH(k_carry_in<<<(unsigned)std::min<long long>((tot + 255) / 256, 4096), 256, 0, st>>>((uint32_t*)ws, (const uint32_t*)carry, S,
                                                                                       wsRowBytes / 4, carryRowBytes / 4, C, wsRowsPerStream));
}
void vp_launch_carry_out(cudaStream_t st, void* carry, const void* ws, int S, int wsRowBytes, int carryRowBytes, int C, long long nNew,
                         long long wsRowsPerStream) {
    const long long tot = (long long)S * C * (carryRowBytes / 4);
    if (tot <= 0) return;
    VP_LAUNCH(k_carry_out<<<(unsigned)std::min<long long>((tot + 255) / 256, 4096), 256, 0, st>>>((uint32_t*)carry, (const uint32_t*)ws, S,
                                                                                        wsRowBytes / 4, carryRowBytes / 4, C, nNew, wsRowsPerStream));
}

// row `srcRow` of every stream's C-row store -> slot `dstSlot` of its D-slot store
__global__ void __launch_bounds__(256) k_row_move(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, int S, int words,
                                                  int C, int srcRow, int D, int dstSlot) {
    const long long tot = (long long)S * words;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
        const int s = (int)(i / words), w = (int)(i - (long long)s * words);
        dst[((size_t)s * D + dstSlot) * words + w] = src[((size_t)s * C + srcRow) * words + w];
    }
}
void vp_launch_row_move(cudaStream_t st, void* dst, const void* src, int S, int rowBytes, int C, int srcRow, int D, int dstSlot) {
    const long long tot = (long long)S * (rowBytes / 4);
    if (tot <= 0) return;
    VP_LAUNCH(k_row_move<<<(unsigned)std::min<long long>((tot + 255) / 256, 4096), 256, 0, st>>>((uint32_t*)dst, (const uint32_t*)src, S,
                                                                                       rowBytes / 4, C, srcRow, D, dstSlot));
}

// ---------------------------------------------------------------------------
// Silent state of listed streams (vp_engine_reset_streams; every stream at prepare / reset): what a stream holds that has
// received zeros on every input since prepare. The engine lists the carried arrays and their silent values (VPResetSegs);
// one launch fills all of them. Grid: x over a stream's 16-byte units of all segments, y over the listed streams.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_reset_streams(VPResetSegs segs, const int* __restrict__ list, int count) {
    const int unit = blockIdx.x * blockDim.x + threadIdx.x;
    if (unit >= segs.unitsPerStream) return;
    int j = 0, u = unit;
    while (u >= segs.seg[j].units) { u -= segs.seg[j].units; ++j; }
    const VPResetSeg sg = segs.seg[j];
    double2 v;
    if (sg.kind == VP_FILL_ONE_AT) v = make_double2(2 * u == sg.oneAt ? 1.0 : 0.0, 2 * u + 1 == sg.oneAt ? 1.0 : 0.0);
    else v.x = v.y = (sg.kind == VP_FILL_GATED) ? -1.0 : 0.0;
    for (int i = blockIdx.y; i < count; i += gridDim.y) {
        const size_t s = list ? (size_t)__ldg(list + i) : (size_t)i;
        reinterpret_cast<double2*>(sg.base)[s * (size_t)sg.units + u] = v;
    }
}
void vp_launch_reset_streams(cudaStream_t st, const VPResetSegs& segs, const int* list, int count) {
    if (count <= 0 || segs.unitsPerStream <= 0) return;
    const dim3 grid((unsigned)((segs.unitsPerStream + 255) / 256), (unsigned)std::min(count, 65535));
    VP_LAUNCH(k_reset_streams<<<grid, 256, 0, st>>>(segs, list, count));
}

// Stream snapshots (vp_engine_save_streams / vp_engine_load_streams): the same segments, gathered into / scattered from a
// packed staging buffer [count][unitsPerStream] of 16-byte units (a stream's units in segment order). Same grid as
// k_reset_streams; one 16-byte load and one 16-byte store per unit.
__device__ __forceinline__ double2* vp_seg_unit(const VPResetSegs& segs, int unit, size_t s) {
    int j = 0, u = unit;
    while (u >= segs.seg[j].units) { u -= segs.seg[j].units; ++j; }
    return reinterpret_cast<double2*>(segs.seg[j].base) + s * (size_t)segs.seg[j].units + u;
}
__global__ void __launch_bounds__(256) k_save_streams(VPResetSegs segs, const int* __restrict__ list, int count,
                                                      double2* __restrict__ stage) {
    const int unit = blockIdx.x * blockDim.x + threadIdx.x;
    if (unit >= segs.unitsPerStream) return;
    for (int i = blockIdx.y; i < count; i += gridDim.y) {
        const double2* src = vp_seg_unit(segs, unit, (size_t)__ldg(list + i));
        stage[(size_t)i * segs.unitsPerStream + unit] = *src;
    }
}
__global__ void __launch_bounds__(256) k_load_streams(VPResetSegs segs, const int* __restrict__ list, int count,
                                                      const double2* __restrict__ stage) {
    const int unit = blockIdx.x * blockDim.x + threadIdx.x;
    if (unit >= segs.unitsPerStream) return;
    for (int i = blockIdx.y; i < count; i += gridDim.y)
        *vp_seg_unit(segs, unit, (size_t)__ldg(list + i)) = __ldg(stage + (size_t)i * segs.unitsPerStream + unit);
}
void vp_launch_snapshot_streams(cudaStream_t st, const VPResetSegs& segs, const int* list, int count, void* stage, bool save) {
    if (count <= 0 || segs.unitsPerStream <= 0) return;
    const dim3 grid((unsigned)((segs.unitsPerStream + 255) / 256), (unsigned)std::min(count, 65535));
    if (save) VP_LAUNCH(k_save_streams<<<grid, 256, 0, st>>>(segs, list, count, (double2*)stage));
    else VP_LAUNCH(k_load_streams<<<grid, 256, 0, st>>>(segs, list, count, (const double2*)stage));
}

// PitchProcess::silence() (PitchProcess.cpp:146-158) for every stream: both mark vectors cleared (their storage keeps its
// values), pitch = prevPitch = 0, period = prevPeriod = 0. prevVoicedPeriod, periodNew and beta are not touched.
__global__ void __launch_bounds__(128) k_marks_silence(VPMarkState* __restrict__ carry, int S) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    VPMarkState* c = carry + s;
    c->nAn = 0; c->nSt = 0;
    c->period = 0; c->prevPeriod = 0;
    c->voiced = 0; c->prevVoiced = 0;
}
void vp_launch_marks_silence(cudaStream_t st, VPMarkState* carry, int S) {
    VP_LAUNCH(k_marks_silence<<<(S + 127) / 128, 128, 0, st>>>(carry, S));
}

// ---------------------------------------------------------------------------
// 16-bit PCM on the host link (vp_engine_process_host_pcm16): exactly vp_wav.hpp's conversions -- int16 / 32768 in (exact),
// clamp(nearbyint(x * 32768)) out (round to nearest even) -- so a PCM16 file run through the WAV front-end gives the same
// bytes whichever side converts. 8 samples per thread, 16-byte accesses; the tail is scalar.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pcm16_to_float(float* __restrict__ dst, const int16_t* __restrict__ src, long long count) {
    const long long n8 = count >> 3;
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += step) {
        const int4 v = __ldg(reinterpret_cast<const int4*>(src) + i);
        const int w[4] = {v.x, v.y, v.z, v.w};
        float f[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f[2 * k] = (float)(short)(w[k] & 0xffff) * (1.0f / 32768.0f);
            f[2 * k + 1] = (float)(short)(w[k] >> 16) * (1.0f / 32768.0f);
        }
        float4* d = reinterpret_cast<float4*>(dst) + 2 * i;
        d[0] = make_float4(f[0], f[1], f[2], f[3]);
        d[1] = make_float4(f[4], f[5], f[6], f[7]);
    }
    for (long long i = (n8 << 3) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += step)
        dst[i] = (float)src[i] * (1.0f / 32768.0f);
}
__device__ __forceinline__ int vp_pcm16(float v) {
    float s = rintf(v * 32768.0f);
    s = fminf(fmaxf(s, -32768.0f), 32767.0f);
    return (int)s;
}
__global__ void __launch_bounds__(256) k_float_to_pcm16(int16_t* __restrict__ dst, const float* __restrict__ src, long long count) {
    const long long n8 = count >> 3;
    const long long step = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += step) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(src) + 2 * i), b = __ldg(reinterpret_cast<const float4*>(src) + 2 * i + 1);
        const float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        int w[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = (vp_pcm16(f[2 * k]) & 0xffff) | (vp_pcm16(f[2 * k + 1]) << 16);
        reinterpret_cast<int4*>(dst)[i] = make_int4(w[0], w[1], w[2], w[3]);
    }
    for (long long i = (n8 << 3) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += step)
        dst[i] = (int16_t)vp_pcm16(src[i]);
}
void vp_launch_pcm16_to_float(cudaStream_t st, float* dst, const int16_t* src, long long count) {
    if (count <= 0) return;
    VP_LAUNCH(k_pcm16_to_float<<<(unsigned)std::min<long long>((count / 8 + 255) / 256 + 1, 148 * 16), 256, 0, st>>>(dst, src, count));
}
void vp_launch_float_to_pcm16(cudaStream_t st, int16_t* dst, const float* src, long long count) {
    if (count <= 0) return;
    VP_LAUNCH(k_float_to_pcm16<<<(unsigned)std::min<long long>((count / 8 + 255) / 256 + 1, 148 * 16), 256, 0, st>>>(dst, src, count));
}

// history update: the H input samples that precede the NEXT call = the last H of (old history ++ this call's input)
__global__ void __launch_bounds__(256) k_hist_update(float* __restrict__ hNew, const float* __restrict__ hOld,
                                                     const float* __restrict__ x, int S, int H, long long n, long long stride) {
    const long long tot = (long long)S * H;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
        const int s = (int)(i / H);
        const int j = (int)(i - (long long)s * H);
        const long long t = n - H + j;
        hNew[i] = (t >= 0) ? __ldg(x + (size_t)s * stride + t) : hOld[(size_t)s * H + H + t];
    }
}
void vp_launch_hist_update(cudaStream_t st, float* hNew, const float* hOld, const float* x, int S, int H, long long n,
                           long long stride) {
    const long long tot = (long long)S * H;
    VP_LAUNCH(k_hist_update<<<(unsigned)std::min<long long>((tot + 255) / 256, 8192), 256, 0, st>>>(hNew, hOld, x, S, H, n, stride));
}

// ---------------------------------------------------------------------------
// Synthetic inputs: one thread per stream (the formant cascade is a serial
// recursion), 32 samples buffered per thread and written through a shared
// transpose so that global stores are 128-byte rows.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_synth(const vp_synth_stream* __restrict__ streams, int nStreams, long long nSamples,
                                              long long stride, float* __restrict__ voice, float* __restrict__ synthL,
                                              float* __restrict__ synthR) {
    __shared__ float tv[32][33], tl[32][33], tr[32][33];
    const int lane = threadIdx.x;
    const int s0 = blockIdx.x * 32;
    const int s = s0 + lane;
    vp_synth_stream p;
    vp_synth_state st;
    const bool live = s < nStreams;
    if (live) { p = streams[s]; vps_init(&p, &st); }
    for (long long i0 = 0; i0 < nSamples; i0 += 32) {
        if (live) {
            for (int j = 0; j < 32; ++j) {
                float a, b, c;
                vps_step(&p, &st, i0 + j, &a, &b, &c);
                tv[lane][j] = a; tl[lane][j] = b; tr[lane][j] = c;
            }
        }
        __syncwarp();
        for (int r = 0; r < 32; ++r) {
            const int sr = s0 + r;
            const long long i = i0 + lane;
            if (sr < nStreams && i < nSamples) {
                voice[(size_t)sr * stride + i] = tv[r][lane];
                if (synthL) synthL[(size_t)sr * stride + i] = tl[r][lane];
                if (synthR) synthR[(size_t)sr * stride + i] = tr[r][lane];
            }
        }
        __syncwarp();
    }
}

void vp_launch_synth(cudaStream_t st, const void* streams, int nStreams, long long nSamples, long long stride,
                     float* voice, float* synthL, float* synthR) {
    VP_LAUNCH(k_synth<<<(nStreams + 31) / 32, 32, 0, st>>>((const vp_synth_stream*)streams, nStreams, nSamples, stride, voice,
                                                 synthL, synthR));
}

// ---------------------------------------------------------------------------
// Issue-rate microbenchmarks: 8 independent FMA chains per thread.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_peak(T* sink, int iters) {
    T a0 = (T)threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const T m = (T)0.999999, c = (T)1e-3;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
            a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
            a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
        }
    }
    const T r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == (T)123456789) sink[0] = r;
}

// Same issue-rate measurement with the operand pattern of the engine's inner loops: acc_i = fma(x, b_i, acc_i) -- one
// operand shared by all chains (operand-reuse cache), TWO distinct register operands per FMA (b_i and acc_i).
template <typename T>
__global__ void __launch_bounds__(256) k_peak2(T* sink, int iters) {
    T a[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { a[i] = (T)(threadIdx.x + i); b[i] = (T)1e-3 * (T)(i + 1 + (threadIdx.x & 3)); }
    T x = (T)0.999 + (T)1e-6 * (T)threadIdx.x;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 16; ++u) {
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] = fma(x, b[i], a[i]);
        }
        x = -x;
    }
    T r = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) r += a[i];
    if (r == (T)123456789) sink[0] = r;
}

void vp_launch_peak2_fp32(cudaStream_t st, float* sink, int iters, int blocks, int threads) {
    VP_LAUNCH(k_peak2<float><<<blocks, threads, 0, st>>>(sink, iters));
}
void vp_launch_peak2_fp64(cudaStream_t st, double* sink, int iters, int blocks, int threads) {
    VP_LAUNCH(k_peak2<double><<<blocks, threads, 0, st>>>(sink, iters));
}

void vp_launch_peak_fp32(cudaStream_t st, float* sink, int iters, int blocks, int threads) {
    VP_LAUNCH(k_peak<float><<<blocks, threads, 0, st>>>(sink, iters));
}
void vp_launch_peak_fp64(cudaStream_t st, double* sink, int iters, int blocks, int threads) {
    VP_LAUNCH(k_peak<double><<<blocks, threads, 0, st>>>(sink, iters));
}
