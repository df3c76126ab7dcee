// Shared definitions for the sm_100a kernels and the engine host code.
// Timeline convention (SURVEY.md App. A.1): everything is indexed on the
// *delayed timeline* u = input time + latency. Output sample u of a stream is
// the sum of all frame contributions at delayed position u; input before time
// 0 is zero (MyBuffer.cpp:56-58 clears the rings).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/vp_engine.h"

#define VP_ORDER_MAX 100  // PluginProcessor.cpp:53-59 (parameter range ends)
#define VP_SLOTS 32       // >= anCap (20 at 44.1/48 kHz); one warp lane per storage slot
#define VP_VC 4           // vocoder frames of earlier calls that can still overlap a call's first positions (wlen = 4 hop)
#define VP_PC 2           // pitch frames of earlier calls that can still own output positions of a call (L = 4 chunks, hop = 3)
#define VP_ORPH 8         // slots for vocoder frames that are off the current frame grid (see VPGeom::orphPos)
#define VP_NOFRAME (-(1 << 30))

// Geometry + parameters of one prepared engine, passed by value to kernels.
struct VPGeom {
    double fs;
    int B, hopV, wlenV, hopP, L, c, tauMin, tauMax, lat, keep, inSize, anCap;
    int nBlocks;       // blocks in this call
    long long n;       // nBlocks * B samples per stream
    long long stride;  // row stride of the I/O arrays (floats)
    long long wstride; // row stride of the engine's own per-sample intermediates (outV, outP)
    long long vstride; // row stride of the array the vocoder synthesis writes (wstride, or the caller's stride in direct mode)
    long long pstride; // same for the pitch path
    int nFramesV;      // vocoder frames with start < n   (VocoderProcess.cpp:176)
    int nFramesP;      // pitch frames with start < n     (PitchProcess.cpp:169)
    int ordV, ordS, ordP;  // analysis row orders of the call's frames (every frame's own order when ordTab is 0)
    int ordTab;            // 1: the streams' orders differ -- the Levinson kernels take each frame's own orders from the
                           // parameter table at its start block (VPStreamParam::ordV / ordS <= ordV / ordS)
    int ordTabP;           // 1: the streams' pitch orders differ -- rows are ordP + 1 wide (zero padded), the pitch Levinson and
                           // all-pole kernels take each frame's own order from VPTables::ordP (<= ordP)
    int vocOn, pitchOn;
    double yinEps;  // relative margin below which the FP32 YIN decision is re-done in FP64
    // ---- continuation (consecutive process calls = consecutive processBlock calls). Kernels work in CALL-LOCAL
    // coordinates: delayed position 0 = first output sample of this call (global position u0 = blocks done * B).
    const float* histV;  // [S][H] the H input samples that precede this call, per stream (zeros before time 0)
    const float* histS;  //        same for side-chain channel 0
    const float* histR;  //        same for side-chain channel 1 (only when the dry side-chain is mixed in)
    int H;               // history length in samples (>= latency + frameLenP + 3 chunk + max LPC order)
    int offV, offP;      // local position of the first vocoder / pitch frame that starts inside this call
    int kV0, fP0;        // global index of that frame (frames before it belong to earlier calls)
    int hasPrev;         // 1 = an earlier call exists (carry rows / pending pitch frame are valid)
    // ---- parameters that change between calls of a running stream (VocoderProcess.cpp:193-194, PluginProcessor.cpp:214-221)
    // Coefficient rows of this call are synV + 1 / synS + 1 doubles wide: the analysis order of the call's own frames
    // (ordV / ordS) or, when a frame carried from an earlier call had a larger order, that one -- rows are zero padded,
    // and a zero tap changes neither the whitening FIR nor the all-pole recursion.
    int synV, synS;
    int defined;           // VP_MODE_DEFINED: bounds-correct behaviour at the reference's undefined-behaviour sites
    int vocMix, pitchMix;  // the mix adds the vocoder / pitch plane: the path is on, or frames of earlier calls still emit
    // Vocoder frames of earlier calls that are NOT on this call's frame grid: VocoderProcess::process was skipped for some
    // blocks in between (vocBool off), and its startSample -- hence the grid -- froze relative to the block. Their output
    // was already in the reference's ring; here a small kernel finishes them from their carried rows ("orphan" store).
    int orphPos[VP_ORPH];            // call-local start (VP_NOFRAME = empty slot)
    int orphOrdV[VP_ORPH], orphOrdS[VP_ORPH];
    // Carried pitch frames (slot j <-> frame index f = j - VP_PC): call-local start and how many of their 4 chunks are ever
    // processed -- PitchProcess::silence() (pitchBool off, PitchProcess.cpp:146-158) clears the marks, and the chunks of the
    // frame in flight that had not been handled yet then do nothing (processChunkCont, :253-271).
    int carryPosP[VP_PC], carryLimP[VP_PC];
};

// start of pitch frame f in call-local coordinates / number of its chunks that are processed
__host__ __device__ inline long long vp_ppos(const VPGeom& g, int f) {
    return f >= 0 ? (long long)f * g.hopP + g.offP : (long long)g.carryPosP[f + VP_PC];
}
__host__ __device__ inline int vp_plim(const VPGeom& g, int f) { return f >= 0 ? 4 : g.carryLimP[f + VP_PC]; }

// Per-frame row of the vocoder's autocorrelation workspace: lags 0..order (raw sums) followed by the frame's last
// `order` windowed samples (the Levinson kernel's residual-energy correction reads them instead of re-gathering).
__host__ __device__ inline int vp_rowlen(int order) { return 2 * order + 1; }

// gate flags per (stream, block)
#define VP_GATE_VOICE 1
#define VP_GATE_SYNTH 2
#define VP_GATE_NEAR 4

// Frame-indexed vocoder workspace (coefficient rows, energies, gains): per stream VP_VC carry rows (the last frames
// of the previous call: they still overlap this call's first output positions) followed by this call's frames.
__host__ __device__ inline size_t vp_vrow(const VPGeom& g, int s, int k) { return (size_t)s * (size_t)(g.nFramesV + VP_VC) + VP_VC + k; }
// Pitch frames: two carry slots (the last two frames of earlier calls can still own output positions of this call:
// frame length 4 chunks, hop 3 chunks), then this call's frames.
__host__ __device__ inline size_t vp_prow(const VPGeom& g, int s, int f) { return (size_t)s * (size_t)(g.nFramesP + VP_PC) + VP_PC + f; }

// PitchProcess state that survives from one frame to the next (PitchProcess.cpp:76-92, :415-425) and therefore from one
// call to the next: pitch history, and the STORAGE of the analysis / synthesis mark vectors (slot values survive clear()).
struct VPMarkState {
    int period, prevPeriod, prevVoicedPeriod, periodNew, voiced, prevVoiced, nAn, nSt;
    double beta;
    int an[VP_SLOTS], st[VP_SLOTS];
    int pad[2];  // a whole number of 16-byte units per stream (k_reset_streams)
};
static_assert(sizeof(VPMarkState) % 16 == 0, "k_reset_streams writes 16-byte units");

// One stream's input as seen by a call: x = the samples handed to this call, h = the H samples before them.
struct VPRow {
    const float* x;
    const float* h;
};
__device__ __forceinline__ VPRow vp_row(const float* base, const float* hist, int s, const VPGeom& g) {
    VPRow r;
    r.x = base + (size_t)s * g.stride;
    r.h = hist + (size_t)s * g.H;
    return r;
}

// Voice / synth sample at (call-local) delayed position u of a stream (MyBuffer.cpp:142-172): input index u - latency;
// negative indices reach into the carried history (the ring's samplesToKeep + latency part), zeros beyond it.
__device__ __forceinline__ float vp_x(const VPRow& row, long long u, const VPGeom& g) {
    const long long t = u - g.lat;
    if (t >= 0) return (t < g.n) ? __ldg(row.x + t) : 0.0f;
    return (t >= -(long long)g.H) ? __ldg(row.h + g.H + t) : 0.0f;
}

// Cooperative staging of `count` consecutive samples (delayed positions u0 .. u0+count-1) of a stream into shared
// memory by `nthr` threads. Loads are issued in batches of UN per thread BEFORE the first store, so a thread has UN
// global loads in flight instead of one (a plain `for (...) dst[j] = vp_x(...)` loop serialises on the load latency).
template <int UN, typename T>
__device__ __forceinline__ void vp_stage(T* __restrict__ dst, const VPRow& row, long long u0, int count, const VPGeom& g,
                                         int tid, int nthr) {
    const long long t0 = u0 - g.lat;
    const bool inside = t0 >= 0 && t0 + count <= g.n;
    for (int base = tid; base < count; base += nthr * UN) {
        float tmp[UN];
#pragma unroll
        for (int k = 0; k < UN; ++k) {
            const int j = base + k * nthr;
            if (inside) tmp[k] = (j < count) ? __ldg(row.x + t0 + j) : 0.0f;
            else tmp[k] = (j < count) ? vp_x(row, u0 + j, g) : 0.0f;
        }
#pragma unroll
        for (int k = 0; k < UN; ++k) {
            const int j = base + k * nthr;
            if (j < count) dst[j] = (T)tmp[k];
        }
    }
}

// x / d for a divisor d that is reused many times: with inv = RN(1 / d), q = RN(x inv) is within 1 ulp of x / d and
// q' = fma(fma(-q, d, x), inv, q) is the correctly rounded quotient (Markstein) -- bit-identical to x / d, 3 FP64 ops.
__device__ __forceinline__ double vp_div_const(double x, double d, double inv) {
    const double q = x * inv;
    return fma(fma(-q, d, x), inv, q);
}

__device__ __forceinline__ double vp_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Every kernel launch goes through VP_LAUNCH: a launch that the runtime refuses (configuration, shared memory, ...) is
// recorded -- first one wins -- and turns the engine call that issued it into VP_E_CUDA (vp_take_launch_error).
extern thread_local cudaError_t g_vpLaunchError;
inline void vp_note_launch() {
    const cudaError_t err = cudaPeekAtLastError();
    if (err != cudaSuccess && g_vpLaunchError == cudaSuccess) g_vpLaunchError = err;
}
inline cudaError_t vp_take_launch_error() {
    const cudaError_t err = g_vpLaunchError;
    g_vpLaunchError = cudaSuccess;
    if (err != cudaSuccess) cudaGetLastError();  // clear the runtime's copy as well
    return err;
}
#define VP_LAUNCH(...) do { __VA_ARGS__; vp_note_launch(); } while (0)

#define VP_CUDA_OK(call)                                                        \
    do {                                                                        \
        cudaError_t _e = (call);                                                \
        if (_e != cudaSuccess) return vp_fail(e, _e, #call, __FILE__, __LINE__); \
    } while (0)

// The per-instance parameters of one stream (vp_stream_params) as the kernels read them: gains already converted with
// decibelsToGain<float>(dB, -59) (PluginProcessor.cpp:226-230, VocoderProcess.cpp:291, PitchProcess.cpp:336), the key, and
// whether each dry path is mixed in (> -59 dB). Device table [nStreams], indexed by the engine's global stream; a call with
// scheduled changes (vp_engine_schedule_stream_params) reads a block-indexed table [nBlocks][nStreams] instead.
struct __align__(16) VPStreamParam {
    float gainVocF, gainPitchF, gainVoiceF, gainSynthF;
    int key;             // Notes::key 0..12: row of the note LUTs
    int dryOn, synthOn;  // dry voice / dry side-chain mixed in
    int16_t ordV, ordS;  // vocoder LPC orders (vp_stream_orders): read by the Levinson kernels when VPGeom::ordTab is set
};
static_assert(sizeof(VPStreamParam) == 32, "one table entry is 32 bytes");

// ---- kernel launchers (one per .cu file) -------------------------------------
struct VPTables {
    const double* wV;        // vocoder analysis window [wlenV]        VocoderProcess.cpp:116-130 ("sine": the sine window; "hann": ones)
    const double* wS;        // vocoder synthesis window [wlenV]       ("sine": the same table; "hann": Hann x overlap factor)
    const double* stP;       // pitch synthesis window [L]             PitchProcess.cpp:889-905
    const double* hann;      // PSOLA Hann tables, all T               PitchProcess.cpp:878-882
    const int* hannOff;      // offset of table T in hann[], [tauMax+1]
    const double* lutBeta;   // [13 keys][tauMax+1] per period: closestFreq / pitch   PitchProcess.cpp:594-596
    const int* lutPeriodNew; // [13][tauMax+1] per period: round(period / beta)
    const int* lutNote;      // [13][tauMax+1] per period: snapped note index         Notes.cpp:79-110
    const VPStreamParam* sp; // per-stream parameters of the pass's streams (table + streamBase): sp[blk * spStride + s], s = stream
                             // of the pass, blk = call-local block of the read site's delayed-timeline position (vp_sp)
    int spStride;            // 0: one entry per stream for the whole call; nStreams: a call with scheduled changes
    const int16_t* ordP;     // lpcPitch in force for each stream of the pass (vp_engine_set_stream_pitch_orders), read when
                             // VPGeom::ordTabP is set: fixed between two starts of a stream, so one entry per stream and call
};
// the parameters of stream s (of the pass) in force at call-local block blk
__device__ __forceinline__ const VPStreamParam& vp_sp(const VPTables& tb, int blk, int s) {
    return tb.sp[(size_t)blk * (size_t)tb.spStride + s];
}

int vp_gate_carry_rows(const VPGeom& g);
void vp_launch_gate(cudaStream_t st, const VPGeom& g, int S, const float* voice, const float* synth, uint8_t* gate,
                    double* part /* [S][partRows][4]: carry rows then this call's blocks */, int partRows);
void vp_launch_voc_gain(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const double* EeV, const double* EeS, double* G,
                        double* Gs, double* hist);

void vp_launch_voc_autocorr(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                            const float* synth, const uint8_t* gate, double* rV, double* rS);
void vp_launch_voc_levinson(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                            const float* synth, const uint8_t* gate, const double* rV, const double* rS, double* aV,
                            double* aS, double* EeV, double* EeS);
bool vp_voc_synth_needs_clear(const VPGeom& g);  // false: the kernel writes every output position itself
void vp_launch_voc_synth(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* synth,
                         const double* aV, const double* aS, const double* EeS, const double* G, float* outV);

void vp_launch_yin(cudaStream_t st, const VPGeom& g, int S, const float* voice, const uint8_t* gate, int* period,
                   uint32_t* yflags, int* recheckList, int* recheckCount, int maxList);
// correlation-form YIN (default): chunk partials P [S][3 nFramesP + 1][lagPad] floats, then the per-frame decision
int vp_yin_corr_lagpad(const VPGeom& g);
int vp_yin_corr_chunks(const VPGeom& g);
int vp_yin_corr_tiles(const VPGeom& g);
void vp_launch_yin_corr(cudaStream_t st, const VPGeom& g, int S, const float* voice, float* P, double* Ech, int lagBegin,
                        int lagEnd, const int* tileList, const int* tileCount);
int vp_yin_phase_split(const VPGeom& g);
void vp_launch_yin_decide(cudaStream_t st, const VPGeom& g, int S, const float* voice, const uint8_t* gate, const float* P, const double* Ech,
                          int* period, uint32_t* yflags, int* recheckList, int* recheckCount, int maxList, int kLimit, int phase,
                          int* pendList, int* pendCount, int* tileFlag, int* tileList, int* tileCount);
void vp_launch_yin_recheck(cudaStream_t st, const VPGeom& g, int S, const float* voice, const uint8_t* gate, int* period,
                           uint32_t* yflags, const int* recheckList, const int* recheckCount, int maxList);
void vp_launch_marks(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                     const uint8_t* gate, const int* period, const uint32_t* yflags, vp_pitch_frame* frames,
                     VPMarkState* carry);
void vp_launch_pitch_lpc(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                         const vp_pitch_frame* frames, double* rP, double* aP);
void vp_launch_pitch_psola(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* voice,
                           vp_pitch_frame* frames, const double* aP, float* outE);
// gainUniform: the gainPitch (as a gain) every stream has in every block of the call and that every carried chunk was
// emitted with, or NULL to read each chunk's from the table. pgIn / pgOut [S][VP_PC][4]: the gain each chunk of the carried
// pitch frames was emitted with, before / after the call (pgOut: the last VP_PC frames of carried ++ new)
void vp_launch_pitch_iir(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const vp_pitch_frame* frames,
                         const double* aP, const float* outE, float* outP, const float* gainUniform, const float* pgIn,
                         float* pgOut);
// anyDry: some stream of the call has a dry path on (then the general kernel, which tests each stream's own flags)
void vp_launch_mix(cudaStream_t st, const VPGeom& g, const VPTables& tb, bool anyDry, int S, const float* voice, const float* synthL,
                   const float* synthR, const float* outV, const float* outP, float* outL, float* outR);

// rows of wsRowBytes in the workspace <-> rows of carryRowBytes in the carried store (the shorter length is copied, the rest
// of the destination row is zero filled)
void vp_launch_carry_in(cudaStream_t st, void* ws, const void* carry, int S, int wsRowBytes, int carryRowBytes, int C,
                        long long wsRowsPerStream);
void vp_launch_carry_out(cudaStream_t st, void* carry, const void* ws, int S, int wsRowBytes, int carryRowBytes, int C, long long nNew,
                         long long wsRowsPerStream);
// row `srcRow` of every stream's C-row carried store -> slot `dstSlot` of its D-slot store (same row bytes)
void vp_launch_row_move(cudaStream_t st, void* dst, const void* src, int S, int rowBytes, int C, int srcRow, int D, int dstSlot);
void vp_launch_marks_silence(cudaStream_t st, VPMarkState* carry, int S);
// The per-stream state carried from call to call, as k_reset_streams sees it: arrays [nStreams][units * 16 bytes], each with
// the value a stream that has heard only silence since prepare holds in it.
#define VP_FILL_ZERO 0    // all bits zero
#define VP_FILL_GATED 1   // doubles = -1.0: EeSynth of a gated vocoder frame (k_voc_levinson*), which no kernel synthesises
#define VP_FILL_ONE_AT 2  // zeros, except double oneAt of each stream's run = 1.0 (VPMarkState::beta)
#define VP_RESET_MAXSEG 16
struct VPResetSeg {
    void* base;
    int units;  // 16-byte units per stream
    int kind, oneAt;
};
struct VPResetSegs {
    VPResetSeg seg[VP_RESET_MAXSEG];
    int nSeg, unitsPerStream;
};
// one launch: the silent state of streams list[0 .. count) (list == NULL: streams 0 .. count - 1) in every segment
void vp_launch_reset_streams(cudaStream_t st, const VPResetSegs& segs, const int* list, int count);
// one launch: streams list[0 .. count) of every segment -> stage [count][unitsPerStream] x 16 bytes (save), or back (load)
void vp_launch_snapshot_streams(cudaStream_t st, const VPResetSegs& segs, const int* list, int count, void* stage, bool save);
// the [nBlocks][S] table of a call with scheduled changes: entry (b, s) = the last event of stream s at or before call-local
// block b (events of s: evBlk / evVal[off[s] .. off[s + 1]), ascending blocks), else cur[s]
void vp_launch_expand_stream_params(cudaStream_t st, const VPStreamParam* cur, const int* off, const int* evBlk,
                                    const VPStreamParam* evVal, VPStreamParam* out, int S, int nBlocks);
// 16-bit PCM <-> float exactly as vp_wav.hpp converts on the host: x / 32768 in, clamp(rint(x * 32768)) out
void vp_launch_pcm16_to_float(cudaStream_t st, float* dst, const int16_t* src, long long count);
void vp_launch_float_to_pcm16(cudaStream_t st, int16_t* dst, const float* src, long long count);
void vp_launch_voc_orphans(cudaStream_t st, const VPGeom& g, const VPTables& tb, int S, const float* synth, const double* oAV,
                           const double* oAS, const double* oEeS, const double* oG, float* outV, int capV, int capS);
void vp_launch_hist_update(cudaStream_t st, float* hNew, const float* hOld, const float* x, int S, int H, long long n,
                           long long stride);

void vp_launch_synth(cudaStream_t st, const void* streams, int nStreams, long long nSamples, long long stride,
                     float* voice, float* synthL, float* synthR);
void vp_launch_peak_fp32(cudaStream_t st, float* sink, int iters, int blocks, int threads);
void vp_launch_peak_fp64(cudaStream_t st, double* sink, int iters, int blocks, int threads);
void vp_launch_peak2_fp32(cudaStream_t st, float* sink, int iters, int blocks, int threads);
void vp_launch_peak2_fp64(cudaStream_t st, double* sink, int iters, int blocks, int threads);
