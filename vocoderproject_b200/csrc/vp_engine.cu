// Engine host code + C ABI (include/vp_engine.h). Plain C++ over the CUDA
// runtime; no PyTorch, no NCCL (streams are independent: SURVEY.md 8(e)).
// The reference-side meaning of each entry point is documented in the header.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <limits.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "vp_common.cuh"
#include "vp_synth.h"
#include "vp_synth_host.hpp"

enum { ST_GATE = 0, ST_VOC_AC, ST_VOC_LEV, ST_VOC_SYN, ST_YIN, ST_YIN64, ST_MARKS, ST_PFRAME, ST_PIIR, ST_MIX, ST_CLEAR, ST_OTHER,
       ST_YIN_DECIDE, ST_PLPC, ST_SPARE2, ST_SPARE3 };
static const char* kStageNames[VP_NSTAGES] = {"gate", "voc_autocorr", "voc_levinson", "voc_synth", "yin_fp32", "yin_fp64_recheck",
                                              "marks", "pitch_psola", "pitch_iir", "mix", "clear", "other",
                                              "yin_decide", "pitch_lpc", "", ""};

thread_local cudaError_t g_vpLaunchError = cudaSuccess;  // per host thread: engines driven from different threads do not see each other's launch failures

// ---------------------------------------------------------------------------
// Frame grids: absolute positions on the delayed timeline. Every stream of an engine shares them (the parameters that move
// the grids -- vocBool, pitchBool -- are per engine; the key, the gains and the LPC orders are per stream and move no
// grid), so this is plain host state; it is what VocoderProcess::startSample, PitchProcess::startSample and
// PitchProcess::nChunk are in the reference, plus the bookkeeping of the frames that outlive the call they started in.
// Pure host logic (no CUDA): vp_grid_plan runs it stand-alone.
// ---------------------------------------------------------------------------
struct GridState {
    int B = 0;
    vp_sizes z;
    long long blocksDone = 0;          // host blocks processed since prepare / reset
    long long nextFrameV = 0;          // start of the next vocoder frame = block start + VocoderProcess::startSample
    int alignedV = 0;                  // carried vocoder frames that lie on the current grid: carry rows VP_VC - alignedV .. VP_VC - 1
    int alignedOrdV[VP_VC] = {0}, alignedOrdS[VP_VC] = {0};  // their analysis row orders (largest over the streams), by carry row
    long long orphAbs[VP_ORPH];        // frames left off the grid by a vocBool-off stretch: absolute start, -1 = free slot
    int orphOrdV[VP_ORPH] = {0}, orphOrdS[VP_ORPH] = {0};
    long long nextChunkP = 0;          // start of the next pitch chunk = block start + PitchProcess::startSample
    int nChunk = 0;                    // PitchProcess::nChunk
    long long carryAbsP[VP_PC];        // carried pitch frames: absolute start (-1 = none) and chunks that are processed at all
    int carryLimP[VP_PC] = {0};
    void reset() {
        blocksDone = 0; nextFrameV = 0; alignedV = 0; nextChunkP = 0; nChunk = 0;
        for (int j = 0; j < VP_ORPH; ++j) orphAbs[j] = -1;
        for (int j = 0; j < VP_PC; ++j) { carryAbsP[j] = -1; carryLimP[j] = 0; }
    }
};
struct GridMove { int srcRow, dstSlot; };  // carry row -> orphan slot (device rows follow the host bookkeeping)

struct vp_engine {
    int device = 0;
    bool prepared = false;
    int mode = VP_MODE_PARITY;  // vp_engine_set_mode
    int lutMode = -1;
    bool failed = false;  // a process call failed half way: the carried state is undefined until vp_engine_reset / vp_engine_prepare
    cudaStream_t st = nullptr, stIn = nullptr, stOut = nullptr;
    cudaStream_t st2 = nullptr;   // the sequential pitch-mark chain runs here, under the vocoder kernels of the same pass
    cudaEvent_t evFork = nullptr, evJoin = nullptr;
    cudaEvent_t evYin[2] = {nullptr}, evMarks[2] = {nullptr}, evSideDone[2] = {nullptr}, evMix[2] = {nullptr};  // pass phases, by pass parity
    bool sidePending = false, mixPending = false;  // an earlier pass of this call recorded evMarks / evMix
    std::vector<cudaEvent_t> evSide;  // (start, end) pairs of the side-stream kernels when stage timing is on
    std::vector<int> evSideStage;
    size_t evSideUsed = 0;
    bool overlapMarks = true;
    bool forkEarly = false;   // VP_OVERLAP=y (developer A/B): fork the mark chain before the autocorrelation instead of after it
    std::string err;
    vp_params prm;
    vp_sizes sz;
    double fs = 0;
    int B = 0, S = 0, maxBlocks = 0;
    int Sc = 0;  // streams per pass
    size_t workspace = 0;
    VPGeom geom;
    // tables (device)
    double *dWS = nullptr;  // synthesis window when it differs from the analysis window ("hann")
    int window = VP_WINDOW_SINE;
    double *dWV = nullptr, *dStP = nullptr, *dHann = nullptr, *dLutBeta = nullptr;
    int *dHannOff = nullptr, *dLutPeriodNew = nullptr, *dLutNote = nullptr;  // note LUTs: [13 keys][tauMax + 1]
    // ---- per-stream parameters (vp_engine_set_stream_params): what each stream's plug-in instance holds, in dB, and the
    // table the kernels read (spTab on the host, dSP on the device, [S]). A changed table goes up through the pinned staging
    // buffer spPinned on the engine's stream before the next call's first kernel; evSpUp marks when that copy has read it.
    // The vocoder orders of each stream (vp_engine_set_stream_orders) are kept beside them (sord) and ride in the same table.
    std::vector<vp_stream_params> sprm;
    std::vector<vp_stream_orders> sord;
    std::vector<VPStreamParam> spTab;
    VPStreamParam *spPinned = nullptr, *dSP = nullptr;
    cudaEvent_t evSpUp = nullptr;
    bool spDirty = false;
    bool anyDry = false, anySynth = false;  // some stream has a dry path (voice or side-chain) / the dry side-chain on
    bool pitchGainUniform = true;           // every stream has the same gainPitch (k_pitch_iir then takes it as an argument)
    bool ordUniform = true;                 // every stream has the orders of spTab[0]
    int ordMaxV = 0, ordMaxS = 0;           // largest orders over the streams
    bool capturing = false;                 // a streaming graph is being captured: nothing table-derived may be baked in
    // ---- per-stream lpcPitch (vp_engine_set_stream_pitch_orders), read when a stream starts (PitchProcess::prepare, :70):
    // pordNext = the order each stream starts with, pordIn = the order its next block runs at. pordIn changes only for a
    // stream that has processed no block since its start, so no frame in flight ever sees a change. It goes up with the
    // parameter table (through pordPinned, behind evSpUp) into dOrdP [S], which the kernels read when the orders differ.
    std::vector<int> pordIn, pordNext;
    int16_t *pordPinned = nullptr, *dOrdP = nullptr;
    bool pordDirty = false;
    bool pordUniform = true;  // every stream has pordIn[0]
    int pordMax = 0;          // largest pordIn
    // ---- scheduled per-stream changes (vp_engine_schedule_stream_params): pending events by (absolute block, stream). A call
    // takes those at its first block into the [S] table (= vp_engine_set_stream_params before it) and those after it into
    // callEv; a call with callEv non-empty reads the block-indexed table dSPB [nBlocks][S], which k_expand_stream_params
    // builds from dSP and the events (uploaded through the pinned staging buffer schPinned; evSchUp marks when that copy
    // has read it). dSPB is allocated at the first such call, outside the workspace budget. Parameter and order events
    // (vp_engine_schedule_stream_orders) of one (block, stream) share an entry; a CallEvent holds the full values in force.
    struct Pending { bool hasP = false, hasO = false; vp_stream_params p; vp_stream_orders o; };
    struct CallEvent { int blk, stream; vp_stream_params p; vp_stream_orders o; VPStreamParam v; };
    std::map<std::pair<long long, int>, Pending> sched;
    std::vector<CallEvent> callEv;
    VPStreamParam* dSPB = nullptr;
    uint8_t *schPinned = nullptr, *dSch = nullptr;
    size_t schPinnedCap = 0, dSchCap = 0;
    cudaEvent_t evSchUp = nullptr;
    // what the call being issued reads (the [S] table or dSPB) and its flags over all of its blocks: some stream has a dry path
    // on / the dry side-chain on in some block, every stream has gainPitch callPg in every block
    const VPStreamParam* callSP = nullptr;
    int callStride = 0;
    bool callAnyDry = false, callAnySynth = false, callPgUniform = true;
    float callPg = 0.0f;
    // the call's vocoder orders: every stream has callOrdV / callOrdS in every block (callOrdTab false), else the largest
    bool callOrdTab = false;
    int callOrdV = 0, callOrdS = 0;
    // workspace (device), sized for Sc streams x maxBlocks
    uint8_t* dGate = nullptr;
    double* dGatePart = nullptr;
    // ---- state carried from call to call, for all S streams (vp_engine_reset zeroes it = prepareToPlay)
    int H = 0;                         // input history length
    int gateCarry = 0;                 // carried gate block partials per stream (inSize / B + 1)
    int histCur = 0;                   // which of the two history buffers is current
    float* cHist[2][3] = {{nullptr}};  // [buffer][voice, synth ch0, synth ch1][S][H]
    double *cGate = nullptr, *cAV = nullptr, *cAS = nullptr, *cEeS = nullptr, *cG = nullptr, *cGainHist = nullptr;
    vp_pitch_frame* cFrames = nullptr; // [S][VP_PC]
    VPMarkState* cMarks = nullptr;     // [S]
    // gain each chunk of the carried pitch frames was emitted with, [S][VP_PC][4], read / written by k_pitch_iir: current =
    // cPG[histCur], the call writes the other one. pgCarry >= 0: every carried chunk of every stream went out with that gain
    // (then k_pitch_iir may take a uniform gain as its argument); pgCarryAny: nothing has been emitted since prepare / reset.
    float* cPG[2] = {nullptr, nullptr};
    float pgCarry = -1.0f;
    bool pgCarryAny = true;
    // ---- per-stream resets (vp_engine_reset_streams): the streams listed since the last process call (rsMark dedupes), put on
    // the device through the pinned staging list rsPinned, like the parameter table; evRsUp marks when that copy has read it
    std::vector<uint8_t> rsMark;
    std::vector<int> rsList;
    int *rsPinned = nullptr, *dRsList = nullptr;
    cudaEvent_t evRsUp = nullptr;
    // ---- stream snapshots (vp_engine_save_streams / vp_engine_load_streams): packed records [count][unitsPerStream] followed
    // by the stream list, staged through pinned host memory (snapPinned) and device memory (dSnap) of snapCap bytes each,
    // allocated at the first save / load that needs them, outside the workspace budget. evSnapUp marks when the last upload
    // has read snapPinned; evSnapSide orders a save behind the side stream's mark chain.
    uint8_t *snapPinned = nullptr, *dSnap = nullptr;
    size_t snapCap = 0;
    cudaEvent_t evSnapUp = nullptr, evSnapSide = nullptr;
    double *dRV = nullptr, *dRS = nullptr, *dAV = nullptr, *dAS = nullptr, *dEeV = nullptr, *dEeS = nullptr, *dG = nullptr, *dGs = nullptr;
    int *dPeriod = nullptr, *dList = nullptr, *dListCount = nullptr;
    uint32_t* dYFlags = nullptr;
    vp_pitch_frame* dFrames = nullptr;
    double *dAP = nullptr, *dRP = nullptr;
    float* dOutE = nullptr;
    float* dYinP = nullptr;   // correlation-form YIN chunk partials
    int* dYinTiles = nullptr;     // two-phase YIN: [1 count | tile flags | tile list]
    int* dYinPending = nullptr;  // list of the frames whose decision needs the upper lags
    size_t yinTilesPerStreamCap = 0;
    bool yinTwoPhase = true;  // VP_YIN_PHASES=1: one pass over all lags
    double* dYinE = nullptr;  // chunk energies
    int yinDirect = 0;        // VP_YIN_MODE=direct: FP32 direct-form (a-b)^2 kernel instead
    float *dOutV = nullptr, *dOutP = nullptr;
    int maxList = 0;
    // decisions kept for the whole batch (all S streams) of the last call
    vp_pitch_frame* dFramesAll = nullptr;
    uint8_t* dGateAll = nullptr;
    double *dEeVAll = nullptr, *dEeSAll = nullptr, *dGAll = nullptr;
    bool keepDecisions = true;
    int lastBlocks = 0;
    VPGeom lastG;  // geometry of the most recent process call (frame counts depend on where the timeline stood)
    // ---- low-latency streaming (one host block per call): pinned host I/O, fixed device I/O, one CUDA graph per block phase
    float *sHostV = nullptr, *sHostS = nullptr, *sHostO = nullptr;  // pinned [S][B]
    float *sDevV = nullptr, *sDevS = nullptr, *sDevO = nullptr;     // device [S][B]
    std::map<std::vector<long long>, cudaGraphExec_t> graphs;
    uint64_t graphLaunches = 0, graphCaptures = 0;
    // host-path staging (device), 3 slices
    int Sh = 0;
    float* hIn[3][3] = {{nullptr}};
    float* hOut[3][2] = {{nullptr}};
    int16_t* pIn[3][3] = {{nullptr}};   // 16-bit PCM landing buffers of vp_engine_process_host_pcm16
    int16_t* pOut[3][2] = {{nullptr}};
    cudaEvent_t evIn[3] = {nullptr}, evComp[3] = {nullptr}, evOut[3] = {nullptr};
    // stats / timing
    uint64_t launches = 0, yinRechecked = 0, yinFrames = 0;
    int passCount = 0;      // passes of the current call
    int capV = 0, capS = 0, capP = 0;  // LPC orders the workspace was sized for
    int reserveV = 0, reserveS = 0;    // vp_engine_reserve_orders: largest lpcVoice / lpcSynth that may be set mid-stream
    int reserveP = 0;                  // vp_engine_reserve_pitch_order: largest per-stream lpcPitch
    GridState gs;                      // frame grids and carried-frame bookkeeping (host side, shared by all streams)
    double *oAV = nullptr, *oAS = nullptr, *oEeS = nullptr, *oG = nullptr;  // orphan store [S][VP_ORPH][...]
    std::vector<cudaEvent_t> ev;
    std::vector<int> evStage;
    size_t evUsed = 0;
    cudaEvent_t evT0 = nullptr, evT1 = nullptr;
    bool stageTiming = false;
    bool timingOpen = false;
    bool timingAccumulate = false;  // vp_engine_timing_reset(e, 1): stage times accumulate over calls  // evT0 already recorded since the last vp_engine_timing_reset
    cudaEvent_t evTimer[8] = {nullptr};
};

static int vp_fail(vp_engine* e, cudaError_t ce, const char* what, const char* file, int line) {
    char buf[512];
    snprintf(buf, sizeof buf, "CUDA error %d (%s) at %s:%d: %s", (int)ce, cudaGetErrorString(ce), file, line, what);
    if (e) e->err = buf;
    return ce == cudaErrorMemoryAllocation ? VP_E_NOMEM : VP_E_CUDA;
}
static int vp_err(vp_engine* e, int code, const char* msg) {
    if (e) e->err = msg;
    return code;
}

// ---------------------------------------------------------------------------
// Host-side restatement of the sizes and tables the reference derives in
// prepareToPlay / prepare (PluginProcessor.cpp:160-176, PitchProcess.cpp:62-128,
// VocoderProcess.cpp:95-135, Notes.cpp:43-110).
// ---------------------------------------------------------------------------
static const double kPiVoc = 3.14159265;              // VocoderProcess.cpp:13
static const double kPi = 3.14159265358979323846;     // juce::MathConstants<double>::pi

static int notes_table(int key, double fMin, double fMax, double* freq /* [128] */) {
    static const int intervals[7] = {2, 2, 1, 2, 2, 2, 1};
    int n = 0, i = 0;
    double f = 27.5;
    f = f * pow(2, (double)key / 12.0);
    const double semi = pow(2, 1.0 / 12);
    while (n == 0 || freq[n - 1] < fMax) {
        if (key != 12) f = f * pow(semi, intervals[i % 7]);
        else f = f * semi;
        if (f > fMin && n < 127) freq[n++] = f;
        i += 1;
    }
    return n - 1;  // pop_back(); freq[n-1] keeps the popped value (Notes.cpp:69, SURVEY App. B U6)
}

extern "C" void vp_default_params(vp_params* p) {
    if (!p) return;
    p->gainPitch = 0.f; p->gainVoice = -60.f; p->gainSynth = -60.f; p->gainVoc = 0.f;
    p->lpcVoice = 40; p->lpcPitch = 15; p->lpcSynth = 5; p->keyPitch = 12; p->pitchBool = 1; p->vocBool = 1;
}

extern "C" int vp_sizes_for(double fs, int B, int keyPitch, vp_sizes* s) {
    if (!s || !(fs >= 8000.0) || fs > 400000.0 || B <= 0 || keyPitch < 0 || keyPitch > 12) return VP_E_ARG;
    const double ratio = fs / 44100.0;
    s->hopV = (int)floor(128.0 * ratio);
    s->wlenV = 4 * s->hopV;
    const int c256 = (int)floor(256.0 * ratio);
    s->hopP = 3 * c256;
    s->frameLenP = 4 * c256;
    s->chunk = s->frameLenP - s->hopP;
    s->tauMin = (int)floor(fs / 800.0);
    s->tauMax = (int)ceil(fs / 100.0);
    s->latency = std::max(s->frameLenP, s->wlenV);
    s->keep = s->frameLenP;
    s->inSize = s->keep + B + s->latency;
    s->outSize = B + s->latency;
    s->anCap = (int)ceil(s->frameLenP * 800.0 / fs) + 1;
    double freq[128];
    s->nFreq = notes_table(keyPitch, 100.0, 800.0, freq);
    return VP_OK;
}

extern "C" int vp_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

static float db_to_gain(float db) { return db > -59.0f ? powf(10.0f, db * 0.05f) : 0.0f; }

template <typename T>
static int upload(vp_engine* e, T** dst, const std::vector<T>& src) {
    if (*dst) { cudaFree(*dst); *dst = nullptr; }
    VP_CUDA_OK(cudaMalloc((void**)dst, std::max<size_t>(src.size(), 1) * sizeof(T)));
    VP_CUDA_OK(cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    return VP_OK;
}

static int build_note_lut(vp_engine* e) {
    // closestFreq / beta / periodNew / note are pure functions of (period, key):
    // pitch = fS / tau (PitchProcess.cpp:441), Notes::getClosestFreq (Notes.cpp:79-110),
    // beta = closestFreq / pitch, periodNew = round(period / beta) (PitchProcess.cpp:594-596).
    // One row per key (every stream reads the row of its own key); the rows depend on the mode (Notes.cpp:99, U6).
    const int tauMax = e->sz.tauMax, row = tauMax + 1;
    std::vector<double> beta((size_t)13 * row, 1.0);
    std::vector<int> pnew((size_t)13 * row, 0), note((size_t)13 * row, -1);
    for (int key = 0; key <= 12; ++key) {
        double freq[128];
        const int nf = notes_table(key, 100.0, 800.0, freq);
        for (int tau = 1; tau <= tauMax; ++tau) {
            const double pitch = e->fs / tau;
            const int idx = (int)(std::lower_bound(freq, freq + nf, pitch) - freq);
            int pick;
            if (idx > 0) pick = (fabs(freq[idx] - pitch) <= fabs(freq[idx - 1] - pitch)) ? idx : idx - 1;  // idx == nf reads the popped slot
            else pick = idx;
            if (e->mode == VP_MODE_DEFINED && idx == nf) pick = nf - 1;  // above the table the closest note is the last one
            const double closest = freq[pick];
            const size_t i = (size_t)key * row + tau;
            beta[i] = closest / pitch;
            pnew[i] = (int)round(tau / beta[i]);
            note[i] = pick;
        }
    }
    int rc;
    if ((rc = upload(e, &e->dLutBeta, beta))) return rc;
    if ((rc = upload(e, &e->dLutPeriodNew, pnew))) return rc;
    if ((rc = upload(e, &e->dLutNote, note))) return rc;
    e->lutMode = e->mode;
    return VP_OK;
}

static int build_tables(vp_engine* e) {
    const vp_sizes& z = e->sz;
    std::vector<double> wV(z.wlenV), wS, stP(z.frameLenP, 1.0);
    {
        const double overlap = (double)(z.wlenV - z.hopV) / (double)z.wlenV;
        double factor = 1.0;
        if (fabs(overlap - 0.75) < pow(10, -10)) factor = 1.0 / sqrt(2);
        if (e->window == VP_WINDOW_HANN) {
            // VocoderProcess.cpp:116-124: juce hann table (normalise = false) x overlapFactor for synthesis, no analysis window
            wS.resize(z.wlenV);
            for (int i = 0; i < z.wlenV; ++i) {
                wS[i] = (0.5 - 0.5 * cos((double)(2 * i) * kPi / (double)(z.wlenV - 1))) * factor;
                wV[i] = 1.0;
            }
        } else {
            for (int i = 0; i < z.wlenV; ++i) wV[i] = factor * sin((i + 0.5) * kPiVoc / (double)z.wlenV);
        }
    }
    {
        const double overlap = ((double)(z.frameLenP - z.hopP)) / ((double)z.frameLenP);
        const int h = (int)round(overlap * z.frameLenP);
        for (int i = 0; i < 2 * h; ++i) {
            const double w = 0.5 - 0.5 * cos((double)(2 * i) * kPi / (double)(2 * h - 1));
            if (i < h) stP[i] = w;
            else stP[z.frameLenP - 2 * h + i] = w;
        }
    }
    std::vector<int> off(z.tauMax + 2, 0);
    size_t tot = 0;
    for (int T = 0; T <= z.tauMax; ++T) { off[T] = (int)tot; tot += (size_t)(2 * T + 1); }
    std::vector<double> hann(tot);
    for (int T = 1; T <= z.tauMax; ++T) {
        double* h = hann.data() + off[T];
        const int len = 2 * T + 1;
        for (int i = 0; i < len; ++i) h[i] = 0.5 - 0.5 * cos((double)(2 * i) * kPi / (double)(len - 1));
    }
    int rc;
    if ((rc = upload(e, &e->dWV, wV))) return rc;
    if (e->dWS) { cudaFree(e->dWS); e->dWS = nullptr; }
    if (!wS.empty() && (rc = upload(e, &e->dWS, wS))) return rc;
    if ((rc = upload(e, &e->dStP, stP))) return rc;
    if ((rc = upload(e, &e->dHann, hann))) return rc;
    if ((rc = upload(e, &e->dHannOff, off))) return rc;
    return build_note_lut(e);
}

static void free_workspace(vp_engine* e) {
    void** cptrs[] = {(void**)&e->cGate, (void**)&e->cAV, (void**)&e->cAS, (void**)&e->cEeS, (void**)&e->cG, (void**)&e->cGainHist,
                      (void**)&e->cFrames, (void**)&e->cMarks, (void**)&e->oAV, (void**)&e->oAS, (void**)&e->oEeS, (void**)&e->oG};
    for (void** p : cptrs) if (*p) { cudaFree(*p); *p = nullptr; }
    for (int i = 0; i < 2; ++i) for (int j = 0; j < 3; ++j) if (e->cHist[i][j]) { cudaFree(e->cHist[i][j]); e->cHist[i][j] = nullptr; }
    for (int i = 0; i < 2; ++i) if (e->cPG[i]) { cudaFree(e->cPG[i]); e->cPG[i] = nullptr; }
    if (e->dSPB) { cudaFree(e->dSPB); e->dSPB = nullptr; }
    if (e->dSch) { cudaFree(e->dSch); e->dSch = nullptr; }
    if (e->schPinned) { cudaFreeHost(e->schPinned); e->schPinned = nullptr; }
    e->dSchCap = e->schPinnedCap = 0;
    e->sched.clear();
    e->callEv.clear();
    if (e->spPinned) { cudaFreeHost(e->spPinned); e->spPinned = nullptr; }
    if (e->pordPinned) { cudaFreeHost(e->pordPinned); e->pordPinned = nullptr; }
    if (e->rsPinned) { cudaFreeHost(e->rsPinned); e->rsPinned = nullptr; }
    if (e->snapPinned) { cudaFreeHost(e->snapPinned); e->snapPinned = nullptr; }
    if (e->dSnap) { cudaFree(e->dSnap); e->dSnap = nullptr; }
    e->snapCap = 0;
    void** ptrs[] = {(void**)&e->dSP, (void**)&e->dOrdP, (void**)&e->dRsList, (void**)&e->dGate, (void**)&e->dRV, (void**)&e->dRS, (void**)&e->dAV, (void**)&e->dAS, (void**)&e->dEeV,
                     (void**)&e->dEeS, (void**)&e->dG, (void**)&e->dGs, (void**)&e->dPeriod, (void**)&e->dList, (void**)&e->dListCount,
                     (void**)&e->dYFlags, (void**)&e->dFrames, (void**)&e->dAP, (void**)&e->dOutE, (void**)&e->dOutV,
                     (void**)&e->dOutP, (void**)&e->dFramesAll, (void**)&e->dGateAll, (void**)&e->dEeVAll, (void**)&e->dEeSAll,
                     (void**)&e->dGAll, (void**)&e->dGatePart, (void**)&e->dYinP, (void**)&e->dYinE, (void**)&e->dRP, (void**)&e->dYinTiles, (void**)&e->dYinPending};
    for (void** p : ptrs) if (*p) { cudaFree(*p); *p = nullptr; }
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) if (e->hIn[i][j]) { cudaFree(e->hIn[i][j]); e->hIn[i][j] = nullptr; }
        for (int j = 0; j < 2; ++j) if (e->hOut[i][j]) { cudaFree(e->hOut[i][j]); e->hOut[i][j] = nullptr; }
        for (int j = 0; j < 3; ++j) if (e->pIn[i][j]) { cudaFree(e->pIn[i][j]); e->pIn[i][j] = nullptr; }
        for (int j = 0; j < 2; ++j) if (e->pOut[i][j]) { cudaFree(e->pOut[i][j]); e->pOut[i][j] = nullptr; }
    }
    e->Sh = 0;
    for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
    e->graphs.clear();
    if (e->sHostV) { cudaFreeHost(e->sHostV); e->sHostV = nullptr; }
    if (e->sHostS) { cudaFreeHost(e->sHostS); e->sHostS = nullptr; }
    if (e->sHostO) { cudaFreeHost(e->sHostO); e->sHostO = nullptr; }
    if (e->sDevV) { cudaFree(e->sDevV); e->sDevV = nullptr; }
    if (e->sDevS) { cudaFree(e->sDevS); e->sDevS = nullptr; }
    if (e->sDevO) { cudaFree(e->sDevO); e->sDevO = nullptr; }
}

extern "C" int vp_engine_create(vp_engine** out, int device) {
    if (!out) return VP_E_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { cudaGetLastError(); return VP_E_CUDA; }
    if (device < 0 || device >= n) return VP_E_ARG;
    vp_engine* e = new vp_engine();
    e->device = device;
    vp_default_params(&e->prm);
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&e->st, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&e->stIn, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&e->stOut, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&e->st2, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->evFork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->evJoin, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreate(&e->evT0) != cudaSuccess || cudaEventCreate(&e->evT1) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->evSpUp, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->evRsUp, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->evSchUp, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->evSnapUp, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&e->evSnapSide, cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        delete e;
        return VP_E_CUDA;
    }
    for (int i = 0; i < 3; ++i) {
        cudaEventCreateWithFlags(&e->evIn[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->evComp[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->evOut[i], cudaEventDisableTiming);
    }
    for (int i = 0; i < 8; ++i) cudaEventCreate(&e->evTimer[i]);
    for (int i = 0; i < 2; ++i) {
        cudaEventCreateWithFlags(&e->evYin[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->evMarks[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->evSideDone[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&e->evMix[i], cudaEventDisableTiming);
    }
    { const char* ov = getenv("VP_OVERLAP"); e->overlapMarks = !(ov && ov[0] == '0'); e->forkEarly = ov && ov[0] == 'y'; }
    { const char* yp = getenv("VP_YIN_PHASES"); e->yinTwoPhase = !(yp && yp[0] == '1'); }
    const char* pt = getenv("VP_STAGE_TIMING");
    e->stageTiming = pt && pt[0] == '1';
    *out = e;
    return VP_OK;
}

extern "C" void vp_engine_destroy(vp_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    free_workspace(e);
    void** t[] = {(void**)&e->dWS, (void**)&e->dWV, (void**)&e->dStP, (void**)&e->dHann, (void**)&e->dHannOff, (void**)&e->dLutBeta,
                  (void**)&e->dLutPeriodNew, (void**)&e->dLutNote};
    for (void** p : t) if (*p) cudaFree(*p);
    for (auto ev : e->ev) cudaEventDestroy(ev);
    for (int i = 0; i < 3; ++i) { cudaEventDestroy(e->evIn[i]); cudaEventDestroy(e->evComp[i]); cudaEventDestroy(e->evOut[i]); }
    cudaEventDestroy(e->evT0); cudaEventDestroy(e->evT1);
    for (int i = 0; i < 8; ++i) cudaEventDestroy(e->evTimer[i]);
    for (auto ev : e->evSide) cudaEventDestroy(ev);
    cudaEventDestroy(e->evFork); cudaEventDestroy(e->evJoin); cudaEventDestroy(e->evSpUp); cudaEventDestroy(e->evRsUp); cudaEventDestroy(e->evSchUp);
    cudaEventDestroy(e->evSnapUp); cudaEventDestroy(e->evSnapSide);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(e->evYin[i]); cudaEventDestroy(e->evMarks[i]); cudaEventDestroy(e->evSideDone[i]); cudaEventDestroy(e->evMix[i]); }
    cudaStreamDestroy(e->st); cudaStreamDestroy(e->stIn); cudaStreamDestroy(e->stOut); cudaStreamDestroy(e->st2);
    delete e;
}

extern "C" const char* vp_last_error(const vp_engine* e) { return e ? e->err.c_str() : "null engine"; }

static bool gain_ok(float g) { return g >= -60.0f && g <= 6.0f; }  // (false for NaN)

static int check_params(const vp_params* p) {
    if (!p) return VP_E_ARG;
    if (p->lpcVoice < 2 || p->lpcVoice > 100 || p->lpcPitch < 2 || p->lpcPitch > 100 || p->lpcSynth < 2 || p->lpcSynth > 30)
        return VP_E_RANGE;
    if (p->keyPitch < 0 || p->keyPitch > 12) return VP_E_RANGE;
    const float gs[4] = {p->gainPitch, p->gainVoice, p->gainSynth, p->gainVoc};
    for (float g : gs) if (!gain_ok(g)) return VP_E_RANGE;
    return VP_OK;
}

extern "C" int vp_engine_set_window(vp_engine* e, int window) {
    if (!e) return VP_E_ARG;
    if (window != VP_WINDOW_SINE && window != VP_WINDOW_HANN) return vp_err(e, VP_E_ARG, "unknown window type");
    if (window != e->window) {
        if (e->prepared && e->gs.blocksDone > 0) return vp_err(e, VP_E_STATE, "the window type is an argument of prepare (VocoderProcess.cpp:35-71): vp_engine_reset first");
        e->window = window;
        e->prepared = false;  // the tables are built by vp_engine_prepare
    }
    return VP_OK;
}

extern "C" int vp_engine_set_mode(vp_engine* e, int mode) {
    if (!e) return VP_E_ARG;
    if (mode != VP_MODE_PARITY && mode != VP_MODE_DEFINED) return vp_err(e, VP_E_ARG, "unknown mode");
    if (mode != e->mode) {
        for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);  // the mode is baked into the captured kernel arguments
        e->graphs.clear();
    }
    e->mode = mode;
    if (e->prepared && e->lutMode != mode) {
        cudaSetDevice(e->device);
        cudaStreamSynchronize(e->st);
        return build_note_lut(e);
    }
    return VP_OK;
}

extern "C" int vp_engine_reserve_orders(vp_engine* e, int maxLpcVoice, int maxLpcSynth) {
    if (!e) return VP_E_ARG;
    if (maxLpcVoice < 0 || maxLpcVoice > 100 || maxLpcSynth < 0 || maxLpcSynth > 30) return vp_err(e, VP_E_RANGE, "order outside the plug-in's range");
    e->reserveV = maxLpcVoice; e->reserveS = maxLpcSynth;
    if (e->prepared && (maxLpcVoice > e->capV || maxLpcSynth > e->capS)) {
        if (e->gs.blocksDone > 0) return vp_err(e, VP_E_STATE, "vp_engine_reserve_orders on a running stream: call it before vp_engine_prepare");
        e->prepared = false;
    }
    return VP_OK;
}

extern "C" int vp_engine_reserve_pitch_order(vp_engine* e, int maxLpcPitch) {
    if (!e) return VP_E_ARG;
    if (maxLpcPitch < 0 || maxLpcPitch > 100) return vp_err(e, VP_E_RANGE, "order outside the plug-in's range");
    if (e->prepared && maxLpcPitch > e->capP && e->gs.blocksDone > 0)
        return vp_err(e, VP_E_STATE, "vp_engine_reserve_pitch_order on a running stream: call it before vp_engine_prepare");
    e->reserveP = maxLpcPitch;
    if (e->prepared && maxLpcPitch > e->capP) e->prepared = false;
    return VP_OK;
}

// after pordIn changed: the next call uploads the orders, the batch-wide flags are recomputed
static void pitch_orders_changed(vp_engine* e) {
    e->pordDirty = true;
    e->pordUniform = true;
    e->pordMax = 0;
    for (int p : e->pordIn) {
        e->pordUniform = e->pordUniform && p == e->pordIn[0];
        e->pordMax = std::max(e->pordMax, p);
    }
}

extern "C" int vp_engine_set_stream_pitch_orders(vp_engine* e, int firstStream, int count, const int* lpcPitch) {
    if (!e) return VP_E_ARG;
    if (!e->prepared) return vp_err(e, VP_E_STATE, "vp_engine_prepare has not been called");
    if (firstStream < 0 || count < 0 || firstStream > e->S - count || (count > 0 && !lpcPitch))
        return vp_err(e, VP_E_ARG, "stream range outside [0, nStreams), or NULL values");
    for (int i = 0; i < count; ++i)
        if (lpcPitch[i] < 2 || lpcPitch[i] > 100) return vp_err(e, VP_E_RANGE, "order outside the plug-in's range");
    for (int i = 0; i < count; ++i)
        if (lpcPitch[i] > e->capP)
            return vp_err(e, VP_E_STATE, "lpcPitch beyond what vp_engine_prepare sized: vp_engine_reserve_pitch_order before vp_engine_prepare");
    // a stream that has processed no block since its start (none since prepare / reset, or a reset of it pending) starts with
    // the new value at the next call; any other stream keeps its order until its next start
    const bool fresh = e->gs.blocksDone == 0;
    bool changed = false;
    for (int i = 0; i < count; ++i) {
        const int s = firstStream + i;
        e->pordNext[s] = lpcPitch[i];
        if ((fresh || e->rsMark[s]) && e->pordIn[s] != lpcPitch[i]) { e->pordIn[s] = lpcPitch[i]; changed = true; }
    }
    if (changed) pitch_orders_changed(e);
    return VP_OK;
}

extern "C" int vp_engine_get_stream_pitch_orders(const vp_engine* e, int firstStream, int count, int* inForce, int* next) {
    if (!e) return VP_E_ARG;
    if (!e->prepared) return VP_E_STATE;
    if (firstStream < 0 || count < 0 || firstStream > e->S - count) return VP_E_ARG;
    for (int i = 0; i < count; ++i) {
        if (inForce) inForce[i] = e->pordIn[firstStream + i];
        if (next) next[i] = e->pordNext[firstStream + i];
    }
    return VP_OK;
}

static VPStreamParam stream_table_entry(const vp_stream_params& p, const vp_stream_orders& o) {
    VPStreamParam q;
    memset(&q, 0, sizeof q);
    q.gainVocF = db_to_gain(p.gainVoc); q.gainPitchF = db_to_gain(p.gainPitch);
    q.gainVoiceF = db_to_gain(p.gainVoice); q.gainSynthF = db_to_gain(p.gainSynth);
    q.key = p.keyPitch;
    q.dryOn = p.gainVoice > -59.0f; q.synthOn = p.gainSynth > -59.0f;
    q.ordV = (int16_t)o.lpcVoice; q.ordS = (int16_t)o.lpcSynth;
    return q;
}

// stream s takes the values v and the orders o; true when its table entry changed
static bool put_one_stream(vp_engine* e, int s, const vp_stream_params& v, const vp_stream_orders& o) {
    const VPStreamParam t = stream_table_entry(v, o);
    e->sprm[s] = v;
    e->sord[s] = o;
    if (memcmp(&e->spTab[s], &t, sizeof t) == 0) return false;
    e->spTab[s] = t;
    return true;
}

// after table entries changed: the next call uploads the table, the batch-wide flags are recomputed
static void stream_table_changed(vp_engine* e) {
    e->spDirty = true;
    e->anyDry = e->anySynth = false;
    e->pitchGainUniform = e->ordUniform = true;
    e->ordMaxV = e->ordMaxS = 0;
    for (const VPStreamParam& t : e->spTab) {
        e->anyDry = e->anyDry || t.dryOn || t.synthOn;
        e->anySynth = e->anySynth || t.synthOn;
        e->pitchGainUniform = e->pitchGainUniform && t.gainPitchF == e->spTab[0].gainPitchF;
        e->ordUniform = e->ordUniform && t.ordV == e->spTab[0].ordV && t.ordS == e->spTab[0].ordS;
        e->ordMaxV = std::max(e->ordMaxV, (int)t.ordV); e->ordMaxS = std::max(e->ordMaxS, (int)t.ordS);
    }
}

// streams [first, first + count) take the values p[0 .. count) (p == NULL: keep theirs) and the orders o[0 .. count)
// (o == NULL: keep theirs); only a changed table entry makes the next call upload
static void put_streams(vp_engine* e, int first, int count, const vp_stream_params* p, size_t pStep, const vp_stream_orders* o,
                        size_t oStep) {
    bool changed = false;
    for (int i = 0; i < count; ++i) {
        const int s = first + i;
        changed = put_one_stream(e, s, p ? p[(size_t)i * pStep] : e->sprm[s], o ? o[(size_t)i * oStep] : e->sord[s]) || changed;
    }
    if (changed) stream_table_changed(e);
}

static vp_stream_params stream_part(const vp_params& p) {
    vp_stream_params q;
    q.gainPitch = p.gainPitch; q.gainVoice = p.gainVoice; q.gainSynth = p.gainSynth; q.gainVoc = p.gainVoc; q.keyPitch = p.keyPitch;
    return q;
}
static vp_stream_orders order_part(const vp_params& p) { return vp_stream_orders{p.lpcVoice, p.lpcSynth}; }

// VP_E_RANGE outside the plug-in's ranges, VP_E_STATE above what the workspace rows were sized for
static int check_orders(vp_engine* e, const vp_stream_orders* o, size_t step, int count) {
    for (int i = 0; i < count; ++i) {
        const vp_stream_orders& q = o[(size_t)i * step];
        if (q.lpcVoice < 2 || q.lpcVoice > 100 || q.lpcSynth < 2 || q.lpcSynth > 30) return vp_err(e, VP_E_RANGE, "order outside the plug-in's range");
    }
    for (int i = 0; i < count; ++i) {
        const vp_stream_orders& q = o[(size_t)i * step];
        if (q.lpcVoice > e->capV || q.lpcSynth > e->capS)
            return vp_err(e, VP_E_STATE, "lpcVoice / lpcSynth beyond what vp_engine_prepare sized: vp_engine_reserve_orders before "
                                         "vp_engine_prepare");
    }
    return VP_OK;
}

// The table goes up before the first kernel of a call, on the engine's stream. The staging buffer is rewritten only after
// the previous upload has read it: a call that is still queued (vp_engine_process_device returns before it runs) keeps the
// values it was issued with.
// The per-stream lpcPitch values travel the same way.
static int upload_stream_params(vp_engine* e) {
    if (!e->spDirty && !e->pordDirty) return VP_OK;
    VP_CUDA_OK(cudaEventSynchronize(e->evSpUp));
    if (e->spDirty) {
        const size_t bytes = e->spTab.size() * sizeof(VPStreamParam);
        memcpy(e->spPinned, e->spTab.data(), bytes);
        VP_CUDA_OK(cudaMemcpyAsync(e->dSP, e->spPinned, bytes, cudaMemcpyHostToDevice, e->st));
    }
    if (e->pordDirty) {
        for (size_t s = 0; s < e->pordIn.size(); ++s) e->pordPinned[s] = (int16_t)e->pordIn[s];
        VP_CUDA_OK(cudaMemcpyAsync(e->dOrdP, e->pordPinned, e->pordIn.size() * sizeof(int16_t), cudaMemcpyHostToDevice, e->st));
    }
    VP_CUDA_OK(cudaEventRecord(e->evSpUp, e->st));
    e->spDirty = e->pordDirty = false;
    return VP_OK;
}

static bool stream_params_ok(const vp_stream_params& p) {
    return p.keyPitch >= 0 && p.keyPitch <= 12 && gain_ok(p.gainPitch) && gain_ok(p.gainVoice) && gain_ok(p.gainSynth) &&
           gain_ok(p.gainVoc);
}

extern "C" int vp_engine_set_stream_params(vp_engine* e, int firstStream, int count, const vp_stream_params* p) {
    if (!e || !p) return VP_E_ARG;
    if (!e->prepared) return vp_err(e, VP_E_STATE, "vp_engine_prepare has not been called");
    if (firstStream < 0 || count < 0 || firstStream > e->S - count) return vp_err(e, VP_E_ARG, "stream range outside [0, nStreams)");
    for (int i = 0; i < count; ++i)
        if (!stream_params_ok(p[i])) return vp_err(e, VP_E_RANGE, "parameter outside the plug-in's range");
    put_streams(e, firstStream, count, p, 1, nullptr, 0);
    return VP_OK;
}

extern "C" int vp_engine_set_stream_orders(vp_engine* e, int firstStream, int count, const vp_stream_orders* o) {
    if (!e || !o) return VP_E_ARG;
    if (!e->prepared) return vp_err(e, VP_E_STATE, "vp_engine_prepare has not been called");
    if (firstStream < 0 || count < 0 || firstStream > e->S - count) return vp_err(e, VP_E_ARG, "stream range outside [0, nStreams)");
    const int rc = check_orders(e, o, 1, count);
    if (rc) return rc;
    put_streams(e, firstStream, count, nullptr, 0, o, 1);
    return VP_OK;
}

extern "C" int vp_engine_get_stream_orders(const vp_engine* e, int firstStream, int count, vp_stream_orders* out) {
    if (!e || !out) return VP_E_ARG;
    if (!e->prepared) return VP_E_STATE;
    if (firstStream < 0 || count < 0 || firstStream > e->S - count) return VP_E_ARG;
    for (int i = 0; i < count; ++i) out[i] = e->sord[firstStream + i];
    return VP_OK;
}

static_assert(sizeof(vp_stream_order_event) == 24 && sizeof(vp_stream_order_event) % sizeof(vp_stream_orders) == 0 &&
              offsetof(vp_stream_order_event, o) % sizeof(vp_stream_orders) == 0, "event orders are checked as a strided list");

// the checks every schedule call shares: state, list, streams, blocks not yet issued
template <typename Ev>
static int check_events(vp_engine* e, const Ev* ev, int count) {
    if (!e->prepared) return vp_err(e, VP_E_STATE, "vp_engine_prepare has not been called");
    if (count < 0 || (count > 0 && !ev)) return vp_err(e, VP_E_ARG, "events must be non-null and count >= 0");
    for (int i = 0; i < count; ++i) {
        if (ev[i].stream < 0 || ev[i].stream >= e->S) return vp_err(e, VP_E_ARG, "stream index outside [0, nStreams)");
        if (ev[i].block < e->gs.blocksDone) return vp_err(e, VP_E_ARG, "event for a block that has already been issued");
    }
    return VP_OK;
}

extern "C" int vp_engine_schedule_stream_params(vp_engine* e, const vp_stream_event* ev, int count) {
    if (!e) return VP_E_ARG;
    int rc = check_events(e, ev, count);
    if (rc) return rc;
    for (int i = 0; i < count; ++i)
        if (!stream_params_ok(ev[i].p)) return vp_err(e, VP_E_RANGE, "parameter outside the plug-in's range");
    for (int i = 0; i < count; ++i) {  // a later (stream, block) replaces an earlier one
        vp_engine::Pending& q = e->sched[{ev[i].block, ev[i].stream}];
        q.hasP = true; q.p = ev[i].p;
    }
    return VP_OK;
}

extern "C" int vp_engine_schedule_stream_orders(vp_engine* e, const vp_stream_order_event* ev, int count) {
    if (!e) return VP_E_ARG;
    int rc = check_events(e, ev, count);
    if (rc) return rc;
    if ((rc = check_orders(e, count > 0 ? &ev[0].o : nullptr, sizeof(vp_stream_order_event) / sizeof(vp_stream_orders), count))) return rc;
    for (int i = 0; i < count; ++i) {
        vp_engine::Pending& q = e->sched[{ev[i].block, ev[i].stream}];
        q.hasO = true; q.o = ev[i].o;
    }
    return VP_OK;
}

extern "C" int vp_engine_get_stream_params(const vp_engine* e, int firstStream, int count, vp_stream_params* out) {
    if (!e || !out) return VP_E_ARG;
    if (!e->prepared) return VP_E_STATE;
    if (firstStream < 0 || count < 0 || firstStream > e->S - count) return VP_E_ARG;
    for (int i = 0; i < count; ++i) out[i] = e->sprm[firstStream + i];
    return VP_OK;
}

extern "C" int vp_engine_set_params(vp_engine* e, const vp_params* p) {
    if (!e) return VP_E_ARG;
    int rc = check_params(p);
    if (rc) return vp_err(e, rc, "parameter outside the plug-in's range");
    vp_params q = *p;
    const bool running = e->prepared && e->gs.blocksDone > 0;
    // lpcPitch is read in PitchProcess::prepare only (PitchProcess.cpp:70): a change on a running stream has no effect until
    // the next prepareToPlay, exactly as in the reference. It is the engine-wide value every stream gets at vp_engine_prepare;
    // the per-stream values (vp_engine_set_stream_pitch_orders) are never overwritten here.
    if (running) q.lpcPitch = e->prm.lpcPitch;
    // The workspace rows are sized for capV / capS (the orders at vp_engine_prepare, or vp_engine_reserve_orders). On a running
    // stream an order within that range takes effect at the next vocoder frame (VocoderProcess.cpp:193-194); beyond it the
    // reference would run past its orderMax vectors (its assert at :141-147) and the engine refuses.
    if (e->prepared && (q.lpcVoice > e->capV || q.lpcSynth > e->capS || q.lpcPitch != e->prm.lpcPitch)) {
        if (running)
            return vp_err(e, VP_E_STATE, "lpcVoice / lpcSynth beyond what vp_engine_prepare sized: vp_engine_reserve_orders before "
                                         "vp_engine_prepare, or vp_engine_reset, set the parameters, vp_engine_prepare");
        e->prepared = false;  // freshly prepared / reset engine: accepted, the workspace must be sized again (vp_engine_prepare)
    }
    // Every parameter is read where the reference reads it: gains per block / frame / chunk, keyPitch per pitch frame, the
    // LPC orders per vocoder frame, vocBool / pitchBool per block (PluginProcessor.cpp:214-221).
    // The engine-wide fields are baked into the captured graphs' kernel arguments; the per-instance ones are table data.
    if (q.lpcVoice != e->prm.lpcVoice || q.lpcPitch != e->prm.lpcPitch || q.lpcSynth != e->prm.lpcSynth ||
        q.pitchBool != e->prm.pitchBool || q.vocBool != e->prm.vocBool) {
        for (auto& kv : e->graphs) cudaGraphExecDestroy(kv.second);
        e->graphs.clear();
    }
    e->prm = q;
    if (e->prepared) {
        double freq[128];
        e->sz.nFreq = notes_table(q.keyPitch, 100.0, 800.0, freq);
    }
    // the per-instance part and the orders go to every stream (a caller that never sets streams one by one gets one set)
    const vp_stream_params sp = stream_part(q);
    const vp_stream_orders so = order_part(q);
    put_streams(e, 0, (int)e->sprm.size(), &sp, 0, &so, 0);
    return VP_OK;
}

template <typename T>
static int wsalloc(vp_engine* e, T** p, size_t count) {
    VP_CUDA_OK(cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T)));
    return VP_OK;
}

static void frame_counts(const vp_sizes& z, long long n, int* nV, int* nP) {
    *nV = (int)((n + z.hopV - 1) / z.hopV);
    *nP = (int)((n + z.hopP - 1) / z.hopP);
}

// Every array a stream carries from one call to the next, with the value it holds after silence since prepare: rings and
// histories zero (MyBuffer.cpp:56-58), no marks, beta = 1 (PitchProcess.cpp:76-92), and the frames still on the grids gated:
// a vocoder frame with EeSynth < 0 (carried and orphan rows; k_voc_synth_rows / k_voc_orphans skip it, k_voc_gain never
// counts it), a pitch record without VP_PF_HAS_MARKS (pf_live). Silence is a fixed point of this state (a gated vocoder
// frame shifts no energy history, a gated pitch frame only empties anMarks), so it is also the state of a stream that has
// received zeros since prepare, whatever the grids' phase.
static VPResetSegs carried_state(vp_engine* e) {
    VPResetSegs r;
    memset(&r, 0, sizeof r);
    auto add = [&](void* base, size_t bytesPerStream, int kind, int oneAt) {
        r.seg[r.nSeg++] = VPResetSeg{base, (int)(bytesPerStream / 16), kind, oneAt};
        r.unitsPerStream += (int)(bytesPerStream / 16);
    };
    const size_t d = sizeof(double);
    for (int j = 0; j < 3; ++j) add(e->cHist[e->histCur][j], (size_t)e->H * sizeof(float), VP_FILL_ZERO, 0);  // H % 4 == 0
    add(e->cGate, (size_t)e->gateCarry * 4 * d, VP_FILL_ZERO, 0);
    add(e->cAV, (size_t)VP_VC * (e->capV + 1) * d, VP_FILL_ZERO, 0);
    add(e->cAS, (size_t)VP_VC * (e->capS + 1) * d, VP_FILL_ZERO, 0);
    add(e->cEeS, (size_t)VP_VC * d, VP_FILL_GATED, 0);
    add(e->cG, (size_t)VP_VC * d, VP_FILL_ZERO, 0);
    add(e->cGainHist, 20 * d, VP_FILL_ZERO, 0);
    add(e->cFrames, (size_t)VP_PC * sizeof(vp_pitch_frame), VP_FILL_ZERO, 0);
    add(e->cMarks, sizeof(VPMarkState), VP_FILL_ONE_AT, (int)(offsetof(VPMarkState, beta) / d));
    add(e->cPG[e->histCur], (size_t)VP_PC * 4 * sizeof(float), VP_FILL_ZERO, 0);  // (a silent frame has no marks: never emitted)
    add(e->oAV, (size_t)VP_ORPH * (e->capV + 1) * d, VP_FILL_ZERO, 0);
    add(e->oAS, (size_t)VP_ORPH * (e->capS + 1) * d, VP_FILL_ZERO, 0);
    add(e->oEeS, (size_t)VP_ORPH * d, VP_FILL_GATED, 0);
    add(e->oG, (size_t)VP_ORPH * d, VP_FILL_ZERO, 0);
    return r;
}
static_assert((VP_PC * sizeof(vp_pitch_frame)) % 16 == 0 && offsetof(VPMarkState, beta) % sizeof(double) == 0,
              "carried records are whole 16-byte units");

// prepareToPlay state for every stream; pending per-stream resets are dropped (they are part of it); every stream starts
// with its set lpcPitch
static int reset_state(vp_engine* e) {
    e->histCur = 0;  // (the other history buffer is written in full by the next call before it is read)
    vp_launch_reset_streams(e->st, carried_state(e), nullptr, e->S);
    VP_CUDA_OK(vp_take_launch_error());
    VP_CUDA_OK(cudaStreamSynchronize(e->st));
    for (int s : e->rsList) e->rsMark[s] = 0;
    e->rsList.clear();
    if (e->pordIn != e->pordNext) { e->pordIn = e->pordNext; pitch_orders_changed(e); }
    e->sched.clear();
    e->pgCarryAny = true;
    e->gs.B = e->B; e->gs.z = e->sz;
    e->gs.reset();
    e->failed = false;
    return VP_OK;
}

extern "C" int vp_engine_reset(vp_engine* e) {
    if (!e) return VP_E_ARG;
    if (!e->prepared) return vp_err(e, VP_E_STATE, "vp_engine_prepare has not been called");
    VP_CUDA_OK(cudaSetDevice(e->device));
    VP_CUDA_OK(cudaStreamSynchronize(e->st));
    VP_CUDA_OK(cudaStreamSynchronize(e->st2));
    return reset_state(e);
}

extern "C" int vp_engine_reset_streams(vp_engine* e, const int* streams, int count) {
    if (!e) return VP_E_ARG;
    if (!e->prepared) return vp_err(e, VP_E_STATE, "vp_engine_prepare has not been called");
    if (count < 0 || (count > 0 && !streams)) return vp_err(e, VP_E_ARG, "streams must be non-null and count >= 0");
    for (int i = 0; i < count; ++i)
        if (streams[i] < 0 || streams[i] >= e->S) return vp_err(e, VP_E_ARG, "stream index outside [0, nStreams)");
    bool ordChanged = false;
    for (int i = 0; i < count; ++i) {
        const int s = streams[i];
        if (!e->rsMark[s]) { e->rsMark[s] = 1; e->rsList.push_back(s); }
        // the stream starts at the next call: with its set lpcPitch (PitchProcess::prepare)
        if (e->pordIn[s] != e->pordNext[s]) { e->pordIn[s] = e->pordNext[s]; ordChanged = true; }
    }
    if (ordChanged) pitch_orders_changed(e);
    // the new user of a slot does not inherit the old user's automation
    if (!e->sched.empty() && count > 0) {
        std::vector<uint8_t> listed((size_t)e->S, 0);
        for (int i = 0; i < count; ++i) listed[streams[i]] = 1;
        for (auto it = e->sched.begin(); it != e->sched.end();) {
            if (listed[it->first.second]) it = e->sched.erase(it);
            else ++it;
        }
    }
    return VP_OK;
}

// The pending resets of vp_engine_reset_streams, before the first kernel of a call and before begin_call (rows it moves to
// the orphan store are then already silent): the list goes up through the pinned staging buffer, which is rewritten only
// after the previous upload has read it, and one kernel writes the silent state. Nothing is issued when none is pending.
static int apply_stream_resets(vp_engine* e) {
    if (e->rsList.empty()) return VP_OK;
    const int n = (int)e->rsList.size();
    VP_CUDA_OK(cudaEventSynchronize(e->evRsUp));
    memcpy(e->rsPinned, e->rsList.data(), (size_t)n * sizeof(int));
    VP_CUDA_OK(cudaMemcpyAsync(e->dRsList, e->rsPinned, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, e->st));
    VP_CUDA_OK(cudaEventRecord(e->evRsUp, e->st));
    vp_launch_reset_streams(e->st, carried_state(e), e->dRsList, n);
    e->launches++;
    for (int s : e->rsList) e->rsMark[s] = 0;
    e->rsList.clear();
    return VP_OK;
}

// ---------------------------------------------------------------------------
// Stream snapshots (vp_engine_save_streams / vp_engine_load_streams). A blob is one SnapHeader and `count` records; a
// record is a SnapRecord followed by the stream's raw units of every carried_state() segment, in segment order. The header
// holds the layout key (what must match for the raw units to mean the same thing) and the source's frame grids.
// ---------------------------------------------------------------------------
#define VP_SNAP_MAGIC 0x53535056u  // "VPSS"
#define VP_SNAP_VERSION 1u
struct SnapHeader {
    uint32_t magic, version;
    uint64_t checksum;  // FNV-1a over the header's 64-bit words with this field zero
    // layout key
    double sampleRate;
    int32_t B, H, gateCarry, capV, capS, capP, window, nSeg, unitsPerStream, count, reserved0, reserved1;
    int32_t segUnits[VP_RESET_MAXSEG];
    // the source's GridState
    int64_t blocksDone, nextFrameV, nextChunkP;
    int64_t orphAbs[VP_ORPH], carryAbsP[VP_PC];
    int32_t alignedV, nChunk;
    int32_t alignedOrdV[VP_VC], alignedOrdS[VP_VC], orphOrdV[VP_ORPH], orphOrdS[VP_ORPH], carryLimP[VP_PC];
};
struct SnapRecord {
    uint64_t checksum;  // FNV-1a over the record's 64-bit words (this struct, then the raw units) with this field zero
    vp_stream_params p;
    vp_stream_orders o;
    int32_t lpcPitchIn, lpcPitchNext;
    int32_t rowOrdV[VP_VC], rowOrdS[VP_VC], orphRowOrdV[VP_ORPH], orphRowOrdS[VP_ORPH];  // last non-zero coefficient index
    int32_t reserved;
};
static_assert(sizeof(SnapHeader) == VP_SNAPSHOT_HEADER_BYTES && sizeof(SnapRecord) == VP_SNAPSHOT_RECORD_BYTES,
              "snapshot layout documented in vp_engine.h");
static_assert(sizeof(SnapHeader) % 16 == 0 && sizeof(SnapRecord) % 16 == 0, "raw units stay 16-byte aligned");

static uint64_t snap_hash(uint64_t h, const void* p, size_t bytes) {  // bytes % 8 == 0
    const uint8_t* b = (const uint8_t*)p;
    for (size_t i = 0; i < bytes; i += 8) {
        uint64_t w;
        memcpy(&w, b + i, 8);
        h = (h ^ w) * 1099511628211ull;
    }
    return h;
}
static const uint64_t kSnapHashSeed = 14695981039346656037ull;
static uint64_t snap_header_hash(SnapHeader h) { h.checksum = 0; return snap_hash(kSnapHashSeed, &h, sizeof h); }
static uint64_t snap_record_hash(SnapRecord r, const uint8_t* raw, size_t rawBytes) {
    r.checksum = 0;
    return snap_hash(snap_hash(kSnapHashSeed, &r, sizeof r), raw, rawBytes);
}

static size_t snap_record_bytes(const VPResetSegs& segs) { return sizeof(SnapRecord) + (size_t)segs.unitsPerStream * 16; }

// byte offset of the segment at `base` inside a record's raw units
static size_t seg_offset(const VPResetSegs& segs, const void* base) {
    size_t off = 0;
    for (int j = 0; j < segs.nSeg && segs.seg[j].base != base; ++j) off += (size_t)segs.seg[j].units * 16;
    return off;
}

static void snap_layout(const vp_engine* e, const VPResetSegs& segs, SnapHeader* h) {
    memset(h, 0, sizeof *h);
    h->magic = VP_SNAP_MAGIC; h->version = VP_SNAP_VERSION;
    h->sampleRate = e->fs; h->B = e->B; h->H = e->H; h->gateCarry = e->gateCarry;
    h->capV = e->capV; h->capS = e->capS; h->capP = e->capP; h->window = e->window;
    h->nSeg = segs.nSeg; h->unitsPerStream = segs.unitsPerStream;
    for (int j = 0; j < segs.nSeg; ++j) h->segUnits[j] = segs.seg[j].units;
}
static bool same_layout(const SnapHeader& a, const SnapHeader& b) {
    if (a.sampleRate != b.sampleRate || a.B != b.B || a.H != b.H || a.gateCarry != b.gateCarry || a.capV != b.capV ||
        a.capS != b.capS || a.capP != b.capP || a.window != b.window || a.nSeg != b.nSeg || a.unitsPerStream != b.unitsPerStream)
        return false;
    return memcmp(a.segUnits, b.segUnits, sizeof a.segUnits) == 0;
}

static void snap_put_grid(const GridState& gs, SnapHeader* h) {
    h->blocksDone = gs.blocksDone; h->nextFrameV = gs.nextFrameV; h->nextChunkP = gs.nextChunkP;
    h->alignedV = gs.alignedV; h->nChunk = gs.nChunk;
    for (int j = 0; j < VP_VC; ++j) { h->alignedOrdV[j] = gs.alignedOrdV[j]; h->alignedOrdS[j] = gs.alignedOrdS[j]; }
    for (int j = 0; j < VP_ORPH; ++j) { h->orphAbs[j] = gs.orphAbs[j]; h->orphOrdV[j] = gs.orphOrdV[j]; h->orphOrdS[j] = gs.orphOrdS[j]; }
    for (int j = 0; j < VP_PC; ++j) { h->carryAbsP[j] = gs.carryAbsP[j]; h->carryLimP[j] = gs.carryLimP[j]; }
}
static void snap_get_grid(const SnapHeader& h, GridState* gs) {
    gs->blocksDone = h.blocksDone; gs->nextFrameV = h.nextFrameV; gs->nextChunkP = h.nextChunkP;
    gs->alignedV = h.alignedV; gs->nChunk = h.nChunk;
    for (int j = 0; j < VP_VC; ++j) { gs->alignedOrdV[j] = h.alignedOrdV[j]; gs->alignedOrdS[j] = h.alignedOrdS[j]; }
    for (int j = 0; j < VP_ORPH; ++j) { gs->orphAbs[j] = h.orphAbs[j]; gs->orphOrdV[j] = h.orphOrdV[j]; gs->orphOrdS[j] = h.orphOrdS[j]; }
    for (int j = 0; j < VP_PC; ++j) { gs->carryAbsP[j] = h.carryAbsP[j]; gs->carryLimP[j] = h.carryLimP[j]; }
}

// an orphan slot whose frame still emits at the next call (an expired one is a free slot: grid_begin frees it first)
static bool orph_live(const GridState& gs, int j) {
    return gs.orphAbs[j] >= 0 && gs.orphAbs[j] + gs.z.wlenV > gs.blocksDone * (long long)gs.B;
}

// The grid phase: every absolute position relative to the next call's start, with the counters that go with it (the row
// widths are not part of it). Two engines with the same phase run the same frames at the same call-local positions.
struct GridPhase {
    long long nextV, nextP, orph[VP_ORPH], carry[VP_PC];
    int nChunk, alignedV, lim[VP_PC];
};
static GridPhase grid_phase(const GridState& gs) {
    GridPhase p;
    memset(&p, 0, sizeof p);
    const long long u0 = gs.blocksDone * (long long)gs.B;
    p.nextV = gs.nextFrameV - u0; p.nextP = gs.nextChunkP - u0; p.nChunk = gs.nChunk; p.alignedV = gs.alignedV;
    for (int j = 0; j < VP_ORPH; ++j) p.orph[j] = orph_live(gs, j) ? gs.orphAbs[j] - u0 : -1;
    for (int j = 0; j < VP_PC; ++j) {
        p.carry[j] = gs.carryAbsP[j] >= 0 ? gs.carryAbsP[j] - u0 : 1;
        p.lim[j] = gs.carryAbsP[j] >= 0 ? gs.carryLimP[j] : 0;
    }
    return p;
}

// A grid state a target adopts whole must be one that process calls can produce: the kernels size and index by it.
static bool grid_state_ok(const GridState& gs, int capV, int capS) {
    const vp_sizes& z = gs.z;
    if (gs.blocksDone < 0 || gs.blocksDone > (1LL << 40)) return false;
    const long long u0 = gs.blocksDone * (long long)gs.B;
    if (gs.nextFrameV - u0 < 0 || gs.nextFrameV - u0 >= z.hopV || gs.nextChunkP - u0 < 0 || gs.nextChunkP - u0 >= z.chunk) return false;
    if (gs.alignedV < 0 || gs.alignedV > VP_VC || gs.nChunk < 0 || gs.nChunk > 3) return false;
    for (int j = 0; j < VP_VC; ++j)
        if (gs.alignedOrdV[j] < 0 || gs.alignedOrdV[j] > capV || gs.alignedOrdS[j] < 0 || gs.alignedOrdS[j] > capS) return false;
    for (int j = 0; j < VP_ORPH; ++j) {
        if (gs.orphOrdV[j] < 0 || gs.orphOrdV[j] > capV || gs.orphOrdS[j] < 0 || gs.orphOrdS[j] > capS) return false;
        if (gs.orphAbs[j] < -1 || (gs.orphAbs[j] >= 0 && gs.orphAbs[j] >= u0)) return false;
    }
    for (int j = 0; j < VP_PC; ++j) {
        if (gs.carryAbsP[j] < -1 || (gs.carryAbsP[j] >= 0 && (gs.carryAbsP[j] >= u0 || u0 - gs.carryAbsP[j] > (1LL << 30)))) return false;
        if (gs.carryLimP[j] < 0 || gs.carryLimP[j] > 4) return false;
    }
    return true;
}

// last coefficient index whose bits are not zero (rows are zero padded: truncating there is exact, -0.0 included)
static int row_order(const uint8_t* row, int len) {
    for (int k = len - 1; k > 0; --k) {
        uint64_t w;
        memcpy(&w, row + 8 * (size_t)k, 8);
        if (w) return k;
    }
    return 0;
}
static void snap_row_orders(vp_engine* e, const VPResetSegs& segs, const uint8_t* raw, SnapRecord* r) {
    const size_t oCV = seg_offset(segs, e->cAV), oCS = seg_offset(segs, e->cAS), oOV = seg_offset(segs, e->oAV),
                 oOS = seg_offset(segs, e->oAS);
    const int wV = e->capV + 1, wS = e->capS + 1;
    for (int i = 0; i < VP_VC; ++i) {
        r->rowOrdV[i] = row_order(raw + oCV + (size_t)i * wV * 8, wV);
        r->rowOrdS[i] = row_order(raw + oCS + (size_t)i * wS * 8, wS);
    }
    for (int j = 0; j < VP_ORPH; ++j) {
        r->orphRowOrdV[j] = row_order(raw + oOV + (size_t)j * wV * 8, wV);
        r->orphRowOrdS[j] = row_order(raw + oOS + (size_t)j * wS * 8, wS);
    }
}

// the raw units of a stream that has heard silence since prepare (what k_reset_streams writes)
static void snap_silent(const VPResetSegs& segs, uint8_t* raw) {
    for (int j = 0; j < segs.nSeg; ++j) {
        const VPResetSeg& sg = segs.seg[j];
        double* d = reinterpret_cast<double*>(raw);
        const size_t n = (size_t)sg.units * 2;
        for (size_t k = 0; k < n; ++k) d[k] = (sg.kind == VP_FILL_GATED) ? -1.0 : 0.0;
        if (sg.kind == VP_FILL_ONE_AT) d[sg.oneAt] = 1.0;
        raw += (size_t)sg.units * 16;
    }
}

// Every integer of the raw state that a kernel takes as a bound or an index: mark counts within the storage, periods within
// the lag range (they index the note and Hann tables).
static bool snap_raw_ok(vp_engine* e, const VPResetSegs& segs, const uint8_t* raw) {
    const int tauMax = e->sz.tauMax;
    auto period_ok = [&](int p) { return p >= 0 && p <= tauMax; };
    VPMarkState m;
    memcpy(&m, raw + seg_offset(segs, e->cMarks), sizeof m);
    if (m.nAn < 0 || m.nAn > VP_SLOTS || m.nSt < 0 || m.nSt > VP_SLOTS) return false;
    if (!period_ok(m.period) || !period_ok(m.prevPeriod) || !period_ok(m.prevVoicedPeriod) || !period_ok(m.periodNew)) return false;
    const size_t oF = seg_offset(segs, e->cFrames);
    for (int j = 0; j < VP_PC; ++j) {
        vp_pitch_frame f;
        memcpy(&f, raw + oF + j * sizeof f, sizeof f);
        if (f.nAn < 0 || f.nAn > VP_MAX_MARKS || f.nSt < 0 || f.nSt > VP_MAX_MARKS || f.nAnOv < 0 || f.nAnOv > VP_MAX_MARKS) return false;
        if (!period_ok(f.period) || !period_ok(f.periodPsola) || !period_ok(f.periodNew)) return false;
    }
    return true;
}

// pinned + device staging for `count` records (raw units, then the stream list); VP_E_NOMEM before anything is issued
static int snap_staging(vp_engine* e, int count, size_t rawBytes) {
    const size_t need = (size_t)count * rawBytes + ((size_t)count * sizeof(int) + 15) / 16 * 16;
    if (need <= e->snapCap) return VP_OK;
    VP_CUDA_OK(cudaEventSynchronize(e->evSnapUp));  // the last upload has read the old pinned buffer
    if (e->snapPinned) cudaFreeHost(e->snapPinned);
    if (e->dSnap) cudaFree(e->dSnap);  // (cudaFree waits for the device: only when a larger list comes)
    e->snapPinned = nullptr; e->dSnap = nullptr; e->snapCap = 0;
    if (cudaHostAlloc((void**)&e->snapPinned, need, cudaHostAllocDefault) != cudaSuccess ||
        cudaMalloc((void**)&e->dSnap, need) != cudaSuccess) {
        cudaGetLastError();
        if (e->snapPinned) cudaFreeHost(e->snapPinned);
        e->snapPinned = nullptr; e->dSnap = nullptr;
        return vp_err(e, VP_E_NOMEM, "no pinned host or device memory for the snapshot staging buffers");
    }
    e->snapCap = need;
    return VP_OK;
}

// the checks save and load share: state, list (in range; a load also refuses duplicates), buffer
static int snap_check_list(vp_engine* e, const int* streams, int count, const void* buf, bool unique) {
    if (!e->prepared) return vp_err(e, VP_E_STATE, "vp_engine_prepare has not been called");
    if (e->failed) return vp_err(e, VP_E_STATE, "an earlier process call failed half way: the carried stream state is undefined, call vp_engine_reset");
    if (count < 0 || (count > 0 && !streams) || !buf) return vp_err(e, VP_E_ARG, "streams and buf must be non-null and count >= 0");
    std::vector<uint8_t> seen(unique ? (size_t)e->S : 0, 0);
    for (int i = 0; i < count; ++i) {
        if (streams[i] < 0 || streams[i] >= e->S) return vp_err(e, VP_E_ARG, "stream index outside [0, nStreams)");
        if (unique && seen[streams[i]]++) return vp_err(e, VP_E_ARG, "a stream is listed twice");
    }
    return VP_OK;
}

extern "C" int vp_engine_snapshot_size(const vp_engine* e, int count, size_t* bytes) {
    if (!e || !bytes || count < 0) return VP_E_ARG;
    if (!e->prepared) return VP_E_STATE;
    *bytes = sizeof(SnapHeader) + (size_t)count * snap_record_bytes(carried_state(const_cast<vp_engine*>(e)));
    return VP_OK;
}

extern "C" int vp_engine_save_streams(vp_engine* e, const int* streams, int count, void* buf, size_t bytes) {
    if (!e) return VP_E_ARG;
    int rc = snap_check_list(e, streams, count, buf, false);
    if (rc) return rc;
    const VPResetSegs segs = carried_state(e);
    const size_t rawB = (size_t)segs.unitsPerStream * 16, recB = snap_record_bytes(segs);
    if (bytes < sizeof(SnapHeader) + (size_t)count * recB) return vp_err(e, VP_E_ARG, "buffer smaller than vp_engine_snapshot_size");
    VP_CUDA_OK(cudaSetDevice(e->device));
    if ((rc = snap_staging(e, count, rawB))) return rc;
    if (count > 0) {
        // behind every call already issued, the side stream's mark chain included: one gather, one copy back
        int* list = reinterpret_cast<int*>(e->snapPinned + (size_t)count * rawB);
        VP_CUDA_OK(cudaEventSynchronize(e->evSnapUp));
        memcpy(list, streams, (size_t)count * sizeof(int));
        VP_CUDA_OK(cudaEventRecord(e->evSnapSide, e->st2));
        VP_CUDA_OK(cudaStreamWaitEvent(e->st, e->evSnapSide, 0));
        VP_CUDA_OK(cudaMemcpyAsync(e->dSnap + (size_t)count * rawB, list, (size_t)count * sizeof(int), cudaMemcpyHostToDevice, e->st));
        vp_launch_snapshot_streams(e->st, segs, reinterpret_cast<const int*>(e->dSnap + (size_t)count * rawB), count, e->dSnap, true);
        VP_CUDA_OK(vp_take_launch_error());
        VP_CUDA_OK(cudaMemcpyAsync(e->snapPinned, e->dSnap, (size_t)count * rawB, cudaMemcpyDeviceToHost, e->st));
        VP_CUDA_OK(cudaEventRecord(e->evSnapUp, e->st));
        VP_CUDA_OK(cudaStreamSynchronize(e->st));
    }
    SnapHeader h;
    snap_layout(e, segs, &h);
    snap_put_grid(e->gs, &h);
    h.count = count;
    h.checksum = snap_header_hash(h);
    uint8_t* out = (uint8_t*)buf;
    memcpy(out, &h, sizeof h);
    for (int i = 0; i < count; ++i) {
        const int s = streams[i];
        uint8_t* rec = out + sizeof h + (size_t)i * recB;
        uint8_t* raw = rec + sizeof(SnapRecord);
        if (e->rsMark[s]) snap_silent(segs, raw);  // a reset of it is pending: the state that reset gives
        else memcpy(raw, e->snapPinned + (size_t)i * rawB, rawB);
        SnapRecord r;
        memset(&r, 0, sizeof r);
        r.p = e->sprm[s]; r.o = e->sord[s]; r.lpcPitchIn = e->pordIn[s]; r.lpcPitchNext = e->pordNext[s];
        snap_row_orders(e, segs, raw, &r);
        r.checksum = snap_record_hash(r, raw, rawB);
        memcpy(rec, &r, sizeof r);
    }
    return VP_OK;
}

extern "C" int vp_engine_load_streams(vp_engine* e, const int* streams, int count, const void* buf, size_t bytes) {
    if (!e) return VP_E_ARG;
    int rc = snap_check_list(e, streams, count, buf, true);
    if (rc) return rc;
    const VPResetSegs segs = carried_state(e);
    const size_t rawB = (size_t)segs.unitsPerStream * 16, recB = snap_record_bytes(segs);
    // ---- everything is validated on the host before anything is issued
    SnapHeader h, mine;
    if (bytes < sizeof h) return vp_err(e, VP_E_ARG, "buffer smaller than a snapshot header");
    memcpy(&h, buf, sizeof h);
    if (h.magic != VP_SNAP_MAGIC || h.version != VP_SNAP_VERSION) return vp_err(e, VP_E_ARG, "not a stream snapshot of this format version");
    if (h.checksum != snap_header_hash(h)) return vp_err(e, VP_E_ARG, "snapshot header checksum mismatch");
    snap_layout(e, segs, &mine);
    if (!same_layout(h, mine))
        return vp_err(e, VP_E_STATE, "snapshot of an engine with another layout (sample rate, block size, reserved orders or window)");
    if (h.count != count) return vp_err(e, VP_E_ARG, "count differs from the number of records in the snapshot");
    if (bytes < sizeof h + (size_t)count * recB) return vp_err(e, VP_E_ARG, "buffer shorter than the snapshot it holds");
    if (count == 0) return VP_OK;
    GridState src = e->gs;
    snap_get_grid(h, &src);
    const bool adopt = e->gs.blocksDone == 0;  // a target that has processed no block takes the source's grids
    if (adopt) {
        if (!grid_state_ok(src, e->capV, e->capS)) return vp_err(e, VP_E_ARG, "snapshot grid state out of range");
    } else {
        const GridPhase a = grid_phase(src), b = grid_phase(e->gs);
        if (memcmp(&a, &b, sizeof a) != 0)
            return vp_err(e, VP_E_STATE, "snapshot grid phase differs from this engine's (another block sequence or bypass history)");
    }
    const uint8_t* in = (const uint8_t*)buf + sizeof h;
    std::vector<SnapRecord> recs((size_t)count);
    for (int i = 0; i < count; ++i) {
        const uint8_t* rec = in + (size_t)i * recB;
        const uint8_t* raw = rec + sizeof(SnapRecord);
        SnapRecord& r = recs[i];
        memcpy(&r, rec, sizeof r);
        if (r.checksum != snap_record_hash(r, raw, rawB)) return vp_err(e, VP_E_ARG, "snapshot record checksum mismatch");
        if (!stream_params_ok(r.p)) return vp_err(e, VP_E_RANGE, "snapshot record: parameter outside the plug-in's range");
        if ((rc = check_orders(e, &r.o, 1, 1))) return rc;
        if (r.lpcPitchIn < 2 || r.lpcPitchIn > 100 || r.lpcPitchNext < 2 || r.lpcPitchNext > 100)
            return vp_err(e, VP_E_RANGE, "snapshot record: lpcPitch outside the plug-in's range");
        if (r.lpcPitchIn > e->capP || r.lpcPitchNext > e->capP) return vp_err(e, VP_E_STATE, "snapshot record: lpcPitch beyond the reservation");
        if (!snap_raw_ok(e, segs, raw)) return vp_err(e, VP_E_RANGE, "snapshot record: mark count or period outside its range");
        SnapRecord chk = r;
        snap_row_orders(e, segs, raw, &chk);
        if (memcmp(&chk, &r, sizeof r) != 0) return vp_err(e, VP_E_ARG, "snapshot record: row orders do not match its rows");
    }
    VP_CUDA_OK(cudaSetDevice(e->device));
    if ((rc = snap_staging(e, count, rawB))) return rc;
    // ---- issued behind every call already issued: one upload (the pinned buffer is rewritten only after the last upload has
    // read it), one scatter
    VP_CUDA_OK(cudaEventSynchronize(e->evSnapUp));
    int* list = reinterpret_cast<int*>(e->snapPinned + (size_t)count * rawB);
    for (int i = 0; i < count; ++i) memcpy(e->snapPinned + (size_t)i * rawB, in + (size_t)i * recB + sizeof(SnapRecord), rawB);
    memcpy(list, streams, (size_t)count * sizeof(int));
    const size_t upB = (size_t)count * rawB + (size_t)count * sizeof(int);
    VP_CUDA_OK(cudaMemcpyAsync(e->dSnap, e->snapPinned, upB, cudaMemcpyHostToDevice, e->st));
    VP_CUDA_OK(cudaEventRecord(e->evSnapUp, e->st));
    vp_launch_snapshot_streams(e->st, segs, reinterpret_cast<const int*>(e->dSnap + (size_t)count * rawB), count, e->dSnap, false);
    VP_CUDA_OK(vp_take_launch_error());
    e->launches++;
    // ---- host bookkeeping
    std::vector<uint8_t> loaded((size_t)e->S, 0);
    for (int i = 0; i < count; ++i) loaded[streams[i]] = 1;
    if (adopt) {
        snap_get_grid(h, &e->gs);
        // events before the adopted block would have applied already: the values in force from them on
        bool changed = false;
        for (auto it = e->sched.begin(); it != e->sched.end() && it->first.first < e->gs.blocksDone;) {
            const int s = it->first.second;
            const vp_engine::Pending& q = it->second;
            changed = put_one_stream(e, s, q.hasP ? q.p : e->sprm[s], q.hasO ? q.o : e->sord[s]) || changed;
            it = e->sched.erase(it);
        }
        if (changed) stream_table_changed(e);
    }
    // the row widths cover each loaded row's own order (not the source's batch-wide widest)
    for (const SnapRecord& r : recs) {
        for (int i = VP_VC - e->gs.alignedV; i < VP_VC; ++i) {
            e->gs.alignedOrdV[i] = std::max(e->gs.alignedOrdV[i], r.rowOrdV[i]);
            e->gs.alignedOrdS[i] = std::max(e->gs.alignedOrdS[i], r.rowOrdS[i]);
        }
        for (int j = 0; j < VP_ORPH; ++j) {
            if (!orph_live(e->gs, j)) continue;
            e->gs.orphOrdV[j] = std::max(e->gs.orphOrdV[j], r.orphRowOrdV[j]);
            e->gs.orphOrdS[j] = std::max(e->gs.orphOrdS[j], r.orphRowOrdS[j]);
        }
    }
    {   // the carried chunk gains stay uniform only if every loaded one is the batch's
        const size_t oPG = seg_offset(segs, e->cPG[e->histCur]);
        float g0;
        memcpy(&g0, in + sizeof(SnapRecord) + oPG, sizeof g0);
        bool same = e->pgCarryAny || e->pgCarry == g0;
        for (int i = 0; i < count && same; ++i) {
            float pg[VP_PC * 4];
            memcpy(pg, in + (size_t)i * recB + sizeof(SnapRecord) + oPG, sizeof pg);
            for (float g : pg) same = same && g == g0;
        }
        e->pgCarry = same ? g0 : -1.0f;
        e->pgCarryAny = false;
    }
    bool changed = false, ordChanged = false;
    for (int i = 0; i < count; ++i) {
        const int s = streams[i];
        changed = put_one_stream(e, s, recs[i].p, recs[i].o) || changed;
        if (e->pordIn[s] != recs[i].lpcPitchIn) { e->pordIn[s] = recs[i].lpcPitchIn; ordChanged = true; }
        e->pordNext[s] = recs[i].lpcPitchNext;
        e->rsMark[s] = 0;
    }
    if (changed) stream_table_changed(e);
    if (ordChanged) pitch_orders_changed(e);
    // a loaded slot drops its pending reset and its pending scheduled events
    e->rsList.erase(std::remove_if(e->rsList.begin(), e->rsList.end(), [&](int s) { return loaded[s] != 0; }), e->rsList.end());
    for (auto it = e->sched.begin(); it != e->sched.end();) {
        if (loaded[it->first.second]) it = e->sched.erase(it);
        else ++it;
    }
    return VP_OK;
}

// Host part of a call's scheduled changes (nothing is issued; what the call needs is allocated here, so that VP_E_NOMEM comes
// before its first kernel). Events at the call's first block b0 go into the [S] table now: exactly vp_engine_set_stream_params
// before the call. Events after b0 inside the call are listed in callEv (ascending block, then stream); they make the call
// read the block-indexed table. The call's flags (dry paths, uniform pitch gain) cover all of its blocks.
static int plan_schedule(vp_engine* e, int nBlocks) {
    const long long b0 = e->gs.blocksDone;
    bool changed = false;
    for (auto it = e->sched.begin(); it != e->sched.end() && it->first.first == b0;) {  // (no earlier block can be pending)
        const int s = it->first.second;
        const vp_engine::Pending& q = it->second;
        changed = put_one_stream(e, s, q.hasP ? q.p : e->sprm[s], q.hasO ? q.o : e->sord[s]) || changed;
        it = e->sched.erase(it);
    }
    if (changed) stream_table_changed(e);
    e->callEv.clear();
    const auto end = e->sched.lower_bound({b0 + nBlocks, INT_MIN});
    {   // each event carries the full values in force from its block on: a parameter event keeps the stream's orders at that
        // block, an order event its parameters (ascending blocks: the stream's previous event in the list is the one before)
        std::map<int, size_t> lastOf;
        for (auto it = e->sched.begin(); it != end; ++it) {
            const int s = it->first.second;
            const vp_engine::Pending& q = it->second;
            const auto prev = lastOf.find(s);
            vp_stream_params p = prev != lastOf.end() ? e->callEv[prev->second].p : e->sprm[s];
            vp_stream_orders o = prev != lastOf.end() ? e->callEv[prev->second].o : e->sord[s];
            if (q.hasP) p = q.p;
            if (q.hasO) o = q.o;
            lastOf[s] = e->callEv.size();
            e->callEv.push_back({(int)(it->first.first - b0), s, p, o, stream_table_entry(p, o)});
        }
    }
    e->callAnyDry = e->anyDry; e->callAnySynth = e->anySynth;
    e->callPg = e->spTab[0].gainPitchF; e->callPgUniform = e->pitchGainUniform;
    e->callOrdV = e->spTab[0].ordV; e->callOrdS = e->spTab[0].ordS;
    bool ordUniform = e->ordUniform;
    int maxV = e->ordMaxV, maxS = e->ordMaxS;
    for (const auto& c : e->callEv) {
        e->callAnyDry = e->callAnyDry || c.v.dryOn || c.v.synthOn;
        e->callAnySynth = e->callAnySynth || c.v.synthOn;
        e->callPgUniform = e->callPgUniform && c.v.gainPitchF == e->callPg;
        ordUniform = ordUniform && c.v.ordV == e->callOrdV && c.v.ordS == e->callOrdS;
        maxV = std::max(maxV, (int)c.v.ordV); maxS = std::max(maxS, (int)c.v.ordS);
    }
    // orders that differ between streams or blocks: rows as wide as the widest (at least the tuned kernels' 40 / 5), each
    // frame solved at its own orders
    e->callOrdTab = !ordUniform;
    if (e->callOrdTab) { e->callOrdV = std::max(maxV, 40); e->callOrdS = std::max(maxS, 5); }
    e->callSP = e->dSP; e->callStride = 0;
    if (e->callEv.empty()) return VP_OK;
    if (!e->dSPB) {
        if (cudaMalloc((void**)&e->dSPB, (size_t)e->S * e->maxBlocks * sizeof(VPStreamParam)) != cudaSuccess) {
            cudaGetLastError();
            e->dSPB = nullptr;
            return vp_err(e, VP_E_NOMEM, "no device memory for the per-block parameter table of a scheduled call");
        }
    }
    const size_t nEv = e->callEv.size();
    const size_t bytes = (((size_t)(e->S + 1) * 4 + 15) & ~(size_t)15) + ((nEv * 4 + 15) & ~(size_t)15) + nEv * sizeof(VPStreamParam);
    if (bytes > e->schPinnedCap) {
        VP_CUDA_OK(cudaEventSynchronize(e->evSchUp));  // the previous upload has read the old buffer
        if (e->schPinned) cudaFreeHost(e->schPinned);
        e->schPinned = nullptr; e->schPinnedCap = 0;
        if (cudaHostAlloc((void**)&e->schPinned, bytes, cudaHostAllocDefault) != cudaSuccess) {
            cudaGetLastError();
            e->schPinned = nullptr;
            return vp_err(e, VP_E_NOMEM, "no pinned host memory for the scheduled events");
        }
        e->schPinnedCap = bytes;
    }
    if (bytes > e->dSchCap) {
        if (e->dSch) cudaFree(e->dSch);  // (cudaFree waits for the device: only when the list outgrows the buffer)
        e->dSch = nullptr; e->dSchCap = 0;
        if (cudaMalloc((void**)&e->dSch, bytes) != cudaSuccess) {
            cudaGetLastError();
            e->dSch = nullptr;
            return vp_err(e, VP_E_NOMEM, "no device memory for the scheduled events");
        }
        e->dSchCap = bytes;
    }
    e->callSP = e->dSPB; e->callStride = e->S;
    return VP_OK;
}

// Device part, after the [S] table of the call's start is on its way: the events go up through the pinned staging buffer
// (rewritten only after the previous upload has read it) as per-stream lists, and one kernel builds the [nBlocks][S] table.
// The host then holds the values in force at the call's last block; they reach dSP with the next call's upload.
static int issue_schedule(vp_engine* e, int nBlocks) {
    if (e->callEv.empty()) return VP_OK;
    const int S = e->S;
    const size_t nEv = e->callEv.size();
    const size_t offB = ((size_t)(S + 1) * 4 + 15) & ~(size_t)15, blkB = (nEv * 4 + 15) & ~(size_t)15;
    const size_t bytes = offB + blkB + nEv * sizeof(VPStreamParam);
    VP_CUDA_OK(cudaEventSynchronize(e->evSchUp));
    int* off = reinterpret_cast<int*>(e->schPinned);
    int* blk = reinterpret_cast<int*>(e->schPinned + offB);
    VPStreamParam* val = reinterpret_cast<VPStreamParam*>(e->schPinned + offB + blkB);
    for (int i = 0; i <= S; ++i) off[i] = 0;
    for (const auto& c : e->callEv) off[c.stream + 1]++;
    for (int i = 0; i < S; ++i) off[i + 1] += off[i];
    {   // stable counting sort by stream: each stream's events keep their ascending blocks
        std::vector<int> pos(off, off + S);
        for (const auto& c : e->callEv) { const int k = pos[c.stream]++; blk[k] = c.blk; val[k] = c.v; }
    }
    VP_CUDA_OK(cudaMemcpyAsync(e->dSch, e->schPinned, bytes, cudaMemcpyHostToDevice, e->st));
    VP_CUDA_OK(cudaEventRecord(e->evSchUp, e->st));
    vp_launch_expand_stream_params(e->st, e->dSP, reinterpret_cast<const int*>(e->dSch), reinterpret_cast<const int*>(e->dSch + offB),
                                   reinterpret_cast<const VPStreamParam*>(e->dSch + offB + blkB), e->dSPB, S, nBlocks);
    e->launches++;
    bool changed = false;
    for (const auto& c : e->callEv) changed = put_one_stream(e, c.stream, c.p, c.o) || changed;  // ascending blocks: the last one stays
    if (changed) stream_table_changed(e);
    const long long b0 = e->gs.blocksDone;
    e->sched.erase(e->sched.begin(), e->sched.lower_bound({b0 + nBlocks, INT_MIN}));
    return VP_OK;
}

extern "C" int vp_engine_prepare(vp_engine* e, double fs, int B, int S, int maxBlocks, size_t workspaceBytes) {
    if (!e) return VP_E_ARG;
    if (S <= 0 || maxBlocks <= 0 || B <= 0) return vp_err(e, VP_E_ARG, "nStreams, maxBlocks, samplesPerBlock must be > 0");
    vp_sizes z;
    if (vp_sizes_for(fs, B, e->prm.keyPitch, &z) != VP_OK) return vp_err(e, VP_E_ARG, "unsupported sample rate / block size");
    if (z.anCap > VP_MAX_MARKS - 1 || z.tauMin < 2) return vp_err(e, VP_E_ARG, "sample rate outside the supported range");
    // what the kernels can serve: the FP64 YIN re-decision tiles lags as 128 x 15 (tauMax <= 1920), the pitch kernels stage a
    // frame (+ look-back) in shared memory: 192 kHz is the top of the range (8 kHz the bottom, vp_sizes_for)
    if (z.tauMax > 1920) return vp_err(e, VP_E_ARG, "sample rate above 192 kHz is not supported");
    VP_CUDA_OK(cudaSetDevice(e->device));
    VP_CUDA_OK(cudaDeviceSynchronize());
    free_workspace(e);
    e->prepared = false;
    e->fs = fs; e->B = B; e->S = S; e->maxBlocks = maxBlocks; e->sz = z;
    int rc = build_tables(e);
    if (rc) return rc;
    const long long n = (long long)maxBlocks * B;
    int nV, nP;
    frame_counts(z, n, &nV, &nP);
    nV += 1; nP += 1;  // a frame grid that a vocBool / pitchBool-off stretch has shifted can put one more frame into a call
    const int capV = std::max(std::max(e->prm.lpcVoice, e->reserveV), 40), capS = std::max(std::max(e->prm.lpcSynth, e->reserveS), 5);
    const int capP = std::max(e->prm.lpcPitch, e->reserveP);
    {
        const char* ym = getenv("VP_YIN_MODE");
        e->yinDirect = (ym && strcmp(ym, "direct") == 0) ? 1 : 0;
    }
    VPGeom gy;
    memset(&gy, 0, sizeof gy);
    gy.tauMax = z.tauMax; gy.nFramesP = nP;
    const size_t yinP = e->yinDirect ? 0 : (size_t)vp_yin_corr_chunks(gy) * (size_t)vp_yin_corr_lagpad(gy);
    // bytes of intermediates per stream
    const size_t perStream = (size_t)maxBlocks * 33 + (size_t)nV * 8 * (size_t)(3 * (capV + 1) + 3 * (capS + 1) + 3) +
                             (size_t)nP * (12 + sizeof(vp_pitch_frame) + 16 * (size_t)(capP + 1) + 4 * (size_t)z.frameLenP) +
                             (size_t)n * 8 + yinP * 4 + (size_t)(3 * nP + 1) * 8;
    if (workspaceBytes == 0) {
        // default: up to 64 GiB, never more than 40 % of what is free now (the caller's I/O arrays come on top)
        size_t freeB = 0, totalB = 0;
        VP_CUDA_OK(cudaMemGetInfo(&freeB, &totalB));
        workspaceBytes = std::min<size_t>((size_t)64 << 30, (size_t)(0.40 * (double)freeB));
        if (const char* ws = getenv("VP_WORKSPACE_GB")) workspaceBytes = (size_t)(atof(ws) * 1073741824.0);
    }
    long long Sc = (long long)(workspaceBytes / perStream);
    if (Sc < 1) Sc = 1;
    if (Sc > S) Sc = S;
    if (Sc > 32) Sc &= ~31LL;
    if (Sc > 65535) Sc = 65535 & ~31;
    // frame, chunk and tile indices of a pass are 32-bit in the kernels (re-check / pending / tile lists)
    while (Sc > 1 && (long long)Sc * (long long)std::max((long long)nV + VP_VC, (long long)3 * nP + 1 + VP_PC) >= (1LL << 30)) Sc = (Sc / 2 > 32) ? ((Sc / 2) & ~31LL) : Sc / 2;
    e->Sc = (int)Sc;
    e->workspace = perStream * (size_t)Sc;
    const size_t fV = (size_t)Sc * nV, fP = (size_t)Sc * nP;
    const size_t fVc = (size_t)Sc * (nV + VP_VC), fPc = (size_t)Sc * (nP + VP_PC);  // with the carry rows in front
    e->gateCarry = z.inSize / B + 1;
    e->H = (z.latency + z.frameLenP + 3 * z.chunk + VP_ORDER_MAX + 3) & ~3;
    if ((rc = wsalloc(e, &e->dGate, (size_t)Sc * maxBlocks))) return rc;
    if ((rc = wsalloc(e, &e->dGatePart, (size_t)Sc * (maxBlocks + e->gateCarry) * 4))) return rc;
    if ((rc = wsalloc(e, &e->dRV, fV * vp_rowlen(capV)))) return rc;
    if ((rc = wsalloc(e, &e->dRS, fV * vp_rowlen(capS)))) return rc;
    if ((rc = wsalloc(e, &e->dAV, fVc * (capV + 1)))) return rc;
    if ((rc = wsalloc(e, &e->dAS, fVc * (capS + 1)))) return rc;
    if ((rc = wsalloc(e, &e->dEeV, fVc))) return rc;
    if ((rc = wsalloc(e, &e->dEeS, fVc))) return rc;
    if ((rc = wsalloc(e, &e->dG, fVc))) return rc;
    if ((rc = wsalloc(e, &e->dGs, fVc))) return rc;
    if ((rc = wsalloc(e, &e->dPeriod, fP))) return rc;
    if ((rc = wsalloc(e, &e->dYFlags, fP))) return rc;
    e->maxList = (int)std::max<size_t>(fP, 1);  // every frame of a pass can be listed (once): the list cannot overflow
    if ((rc = wsalloc(e, &e->dList, (size_t)e->maxList))) return rc;
    if ((rc = wsalloc(e, &e->dListCount, 1024))) return rc;
    VP_CUDA_OK(cudaMemset(e->dListCount, 0, 1024 * sizeof(int)));
    if ((rc = wsalloc(e, &e->dFrames, fPc))) return rc;
    if ((rc = wsalloc(e, &e->dAP, fPc * (capP + 1)))) return rc;
    if ((rc = wsalloc(e, &e->dRP, fPc * (capP + 1)))) return rc;
    if ((rc = wsalloc(e, &e->dOutE, fPc * (size_t)z.frameLenP))) return rc;
    if ((rc = wsalloc(e, &e->dYinP, (size_t)Sc * yinP))) return rc;
    if ((rc = wsalloc(e, &e->dYinE, e->yinDirect ? 1 : (size_t)Sc * vp_yin_corr_chunks(gy)))) return rc;
    e->yinTilesPerStreamCap = e->yinDirect ? 0 : (size_t)vp_yin_corr_tiles(gy);
    if ((rc = wsalloc(e, &e->dYinTiles, 4 + 2 * (size_t)Sc * e->yinTilesPerStreamCap))) return rc;
    if ((rc = wsalloc(e, &e->dYinPending, (size_t)Sc * (size_t)std::max(nP, 1)))) return rc;
    if ((rc = wsalloc(e, &e->dOutV, (size_t)Sc * n))) return rc;
    if ((rc = wsalloc(e, &e->dOutP, (size_t)Sc * n))) return rc;
    // decisions for all streams (small): frames, gates, energies
    const char* kd = getenv("VP_KEEP_DECISIONS");
    e->keepDecisions = !(kd && kd[0] == '0');
    if (e->keepDecisions) {
        if ((rc = wsalloc(e, &e->dFramesAll, (size_t)S * nP))) return rc;
        if ((rc = wsalloc(e, &e->dGateAll, (size_t)S * maxBlocks))) return rc;
        if ((rc = wsalloc(e, &e->dEeVAll, (size_t)S * nV))) return rc;
        if ((rc = wsalloc(e, &e->dEeSAll, (size_t)S * nV))) return rc;
        if ((rc = wsalloc(e, &e->dGAll, (size_t)S * nV))) return rc;
    }
    // carried state, all S streams
    for (int i = 0; i < 2; ++i) for (int j = 0; j < 3; ++j) if ((rc = wsalloc(e, &e->cHist[i][j], (size_t)S * e->H))) return rc;
    if ((rc = wsalloc(e, &e->cGate, (size_t)S * e->gateCarry * 4))) return rc;
    if ((rc = wsalloc(e, &e->cAV, (size_t)S * VP_VC * (capV + 1)))) return rc;
    if ((rc = wsalloc(e, &e->cAS, (size_t)S * VP_VC * (capS + 1)))) return rc;
    if ((rc = wsalloc(e, &e->oAV, (size_t)S * VP_ORPH * (capV + 1)))) return rc;
    if ((rc = wsalloc(e, &e->oAS, (size_t)S * VP_ORPH * (capS + 1)))) return rc;
    if ((rc = wsalloc(e, &e->oEeS, (size_t)S * VP_ORPH))) return rc;
    if ((rc = wsalloc(e, &e->oG, (size_t)S * VP_ORPH))) return rc;
    if ((rc = wsalloc(e, &e->cEeS, (size_t)S * VP_VC))) return rc;
    if ((rc = wsalloc(e, &e->cG, (size_t)S * VP_VC))) return rc;
    if ((rc = wsalloc(e, &e->cGainHist, (size_t)S * 20))) return rc;
    if ((rc = wsalloc(e, &e->cFrames, (size_t)S * VP_PC))) return rc;
    if ((rc = wsalloc(e, &e->cMarks, (size_t)S))) return rc;
    for (int i = 0; i < 2; ++i) {
        if ((rc = wsalloc(e, &e->cPG[i], (size_t)S * VP_PC * 4))) return rc;
        VP_CUDA_OK(cudaMemset(e->cPG[i], 0, (size_t)S * VP_PC * 4 * sizeof(float)));
    }
    // every stream starts from the engine's parameters
    if ((rc = wsalloc(e, &e->dSP, (size_t)S))) return rc;
    VP_CUDA_OK(cudaHostAlloc((void**)&e->spPinned, (size_t)S * sizeof(VPStreamParam), cudaHostAllocDefault));
    if ((rc = wsalloc(e, &e->dRsList, (size_t)S))) return rc;
    VP_CUDA_OK(cudaHostAlloc((void**)&e->rsPinned, (size_t)S * sizeof(int), cudaHostAllocDefault));
    e->rsMark.assign((size_t)S, 0);
    e->rsList.clear();
    e->sprm.assign((size_t)S, stream_part(e->prm));
    e->sord.assign((size_t)S, order_part(e->prm));
    e->spTab.assign((size_t)S, stream_table_entry(e->sprm[0], e->sord[0]));
    stream_table_changed(e);
    // every stream starts with the engine's lpcPitch; dOrdP is read only once the orders differ, and any change uploads it whole
    if ((rc = wsalloc(e, &e->dOrdP, (size_t)S))) return rc;
    VP_CUDA_OK(cudaHostAlloc((void**)&e->pordPinned, (size_t)S * sizeof(int16_t), cudaHostAllocDefault));
    e->pordIn.assign((size_t)S, e->prm.lpcPitch);
    e->pordNext = e->pordIn;
    pitch_orders_changed(e);
    e->pordDirty = false;
    e->capV = capV; e->capS = capS; e->capP = capP;
    if ((rc = reset_state(e))) return rc;
    e->launches = e->yinRechecked = e->yinFrames = 0;
    e->prepared = true;
    e->lastBlocks = 0;
    return VP_OK;
}

extern "C" int vp_engine_get_sizes(const vp_engine* e, vp_sizes* out) {
    if (!e || !out) return VP_E_ARG;
    if (!e->prepared) return VP_E_STATE;
    *out = e->sz;
    return VP_OK;
}

static void stage_mark(vp_engine* e, int stage) {
    if (!e->stageTiming) return;
    if (e->evUsed >= e->ev.size()) {
        cudaEvent_t ev;
        cudaEventCreate(&ev);
        e->ev.push_back(ev);
        e->evStage.push_back(0);
    }
    e->evStage[e->evUsed] = stage;
    cudaEventRecord(e->ev[e->evUsed++], e->st);
}

static void side_mark(vp_engine* e, int stage = ST_MARKS) {
    if (!e->stageTiming) return;
    if (e->evSideUsed >= e->evSide.size()) {
        cudaEvent_t ev;
        cudaEventCreate(&ev);
        e->evSide.push_back(ev);
        e->evSideStage.push_back(stage);
    }
    e->evSideStage[e->evSideUsed] = stage;
    cudaEventRecord(e->evSide[e->evSideUsed++], e->st2);
}

static void grid_geom(const GridState& gs, VPGeom* g);

static int make_geom(vp_engine* e, int nBlocks, size_t stride, VPGeom* g) {
    const vp_sizes& z = e->sz;
    memset(g, 0, sizeof *g);
    g->fs = e->fs; g->B = e->B; g->hopV = z.hopV; g->wlenV = z.wlenV; g->hopP = z.hopP; g->L = z.frameLenP; g->c = z.chunk;
    g->tauMin = z.tauMin; g->tauMax = z.tauMax; g->lat = z.latency; g->keep = z.keep; g->inSize = z.inSize; g->anCap = z.anCap;
    g->nBlocks = nBlocks; g->n = (long long)nBlocks * e->B; g->stride = (long long)stride;
    g->wstride = (long long)e->maxBlocks * e->B;
    g->vstride = g->pstride = g->wstride;
    g->vocOn = e->prm.vocBool != 0; g->pitchOn = e->prm.pitchBool != 0;
    g->ordV = e->callOrdV; g->ordS = e->callOrdS;  // (plan_schedule: the streams' orders in this call)
    g->ordTab = e->callOrdTab;
    // pitch: every stream at one order -- exactly the kernels of an engine prepared with it; else rows as wide as the widest
    // order, at least 16 doubles when the workspace holds them (the P = 15 residual path then serves every order <= 15)
    g->ordTabP = !e->pordUniform;
    g->ordP = e->pordUniform ? e->pordIn[0] : std::max(e->pordMax, std::min(15, e->capP));
    g->H = e->H;
    g->defined = e->mode == VP_MODE_DEFINED;
    grid_geom(e->gs, g);
    g->yinEps = 1e-4;
    if (const char* ye = getenv("VP_YIN_EPS")) g->yinEps = atof(ye);
    return VP_OK;
}

// ---------------------------------------------------------------------------
// One pass = Sc' <= Sc streams whose I/O rows start at the given pointers; streamBase = index of the pass's first stream in
// the engine's batch (selects its carried state). Phases:
//   A (main)  gate, YIN correlation + decision + FP64 re-decision                       -> evYin
//   S (side)  pitch-mark chain (sequential per stream: one warp per stream)             -> evSideDone   (needs evYin, re-recorded
//             behind the autocorrelation: the chain runs next to the Levinson and synthesis kernels)
//   V (main)  vocoder: autocorrelation | Levinson, gain, synthesis (S is forked between the two parts)
//   P (main)  pitch LPC, PSOLA, all-pole resynthesis + overlap-add                      (needs evSideDone)
//   M (main)  mix + egress, carried state, decisions kept for the getters
// The mark chain has one warp per stream and cannot fill the GPU, so it runs on the side stream next to the vocoder
// kernels. Measured and NOT adopted (profiles/README.md, round 2): the whole pitch synthesis on the side stream, and passes
// software-pipelined across each other so that it has more to hide under -- the step time did not move (556.1 vs 555.6 ms):
// the kernels slow each other down by what they overlap, the step is bound by instruction issue as a whole
// (roofline.mix), not by latency.
// ---------------------------------------------------------------------------
struct PassCtx {
    VPGeom g;
    VPTables tb;
    int Sp = 0;
    size_t sb = 0;
    const float *voice = nullptr, *synthL = nullptr, *synthR = nullptr;
    float *outL = nullptr, *outR = nullptr;
    int* listCount = nullptr;
    int slot = 0;        // event set (pass parity)
    bool sideUsed = false;
};

static void pass_init(vp_engine* e, PassCtx& c, const VPGeom& gIO, int Sp, int streamBase, const float* voice, const float* synthL,
                      const float* synthR, float* outL, float* outR) {
    c.g = gIO;
    c.tb = VPTables{e->dWV, e->dWS ? e->dWS : e->dWV, e->dStP, e->dHann, e->dHannOff, e->dLutBeta, e->dLutPeriodNew, e->dLutNote,
                    e->callSP + streamBase, e->callStride, e->dOrdP + streamBase};
    c.Sp = Sp;
    c.sb = (size_t)streamBase;
    const int hc = e->histCur;
    c.g.histV = e->cHist[hc][0] + c.sb * e->H;
    c.g.histS = e->cHist[hc][1] + c.sb * e->H;
    c.g.histR = e->cHist[hc][2] + c.sb * e->H;
    c.voice = voice; c.synthL = synthL; c.synthR = synthR; c.outL = outL; c.outR = outR;
    c.listCount = e->dListCount + (e->passCount % 1024);
    c.slot = e->passCount & 1;
    e->passCount++;
    c.sideUsed = false;
}

// phase A (main stream)
static int pass_A(vp_engine* e, PassCtx& c) {
    cudaStream_t st = e->st;
    const VPGeom& g = c.g;
    const int Sp = c.Sp;
    const size_t sb = c.sb;
    const long long rowsG = g.nBlocks + e->gateCarry;
    stage_mark(e, ST_OTHER);
    // the previous pass's mark chain reads the gate flags and the YIN decisions this phase is about to overwrite
    if (e->sidePending) VP_CUDA_OK(cudaStreamWaitEvent(st, e->evMarks[c.slot ^ 1], 0));
    vp_launch_carry_in(st, e->dGatePart, e->cGate + sb * e->gateCarry * 4, Sp, 32, 32, e->gateCarry, rowsG);
    vp_launch_gate(st, g, Sp, c.voice, c.synthL, e->dGate, e->dGatePart, (int)rowsG);
    vp_launch_carry_out(st, e->cGate + sb * e->gateCarry * 4, e->dGatePart, Sp, 32, 32, e->gateCarry, g.nBlocks, rowsG);
    if (e->keepDecisions) VP_CUDA_OK(cudaMemcpyAsync(e->dGateAll + sb * g.nBlocks, e->dGate, (size_t)Sp * g.nBlocks, cudaMemcpyDeviceToDevice, st));
    e->launches += 2;
    stage_mark(e, ST_GATE);
    if (g.pitchMix) {
        VP_CUDA_OK(cudaMemsetAsync(c.listCount, 0, sizeof(int), st));
        stage_mark(e, ST_CLEAR);
    }
    if (g.pitchOn && g.nFramesP > 0) {
        if (e->yinDirect) {
            vp_launch_yin(st, g, Sp, c.voice, e->dGate, e->dPeriod, e->dYFlags, e->dList, c.listCount, e->maxList);
            stage_mark(e, ST_YIN);
        } else {
            // (batch calls only: a streaming block has at most one pitch frame per stream and pays per launch)
            const int k1 = (e->yinTwoPhase && g.nFramesP >= 16) ? vp_yin_phase_split(g) : 0;
            if (k1 > 0) {
                // two lag phases: the decision of most voiced frames ends below k1, and the lags above it are then
                // never correlated for their chunks (exact: see k_yin_decide_reg)
                const size_t nT = (size_t)Sp * (size_t)vp_yin_corr_tiles(g);
                int* tCount = e->dYinTiles;
                int* tFlag = e->dYinTiles + 4;
                int* tList = tFlag + (size_t)e->Sc * e->yinTilesPerStreamCap;
                VP_CUDA_OK(cudaMemsetAsync(e->dYinTiles, 0, (4 + nT) * sizeof(int), st));
                vp_launch_yin_corr(st, g, Sp, c.voice, e->dYinP, e->dYinE, 0, k1, nullptr, nullptr);
                stage_mark(e, ST_YIN);
                vp_launch_yin_decide(st, g, Sp, c.voice, e->dGate, e->dYinP, e->dYinE, e->dPeriod, e->dYFlags, e->dList, c.listCount,
                                     e->maxList, k1, 1, e->dYinPending, tCount + 1, tFlag, tList, tCount);
                stage_mark(e, ST_YIN_DECIDE);
                vp_launch_yin_corr(st, g, Sp, c.voice, e->dYinP, e->dYinE, k1, 0, tList, tCount);
                stage_mark(e, ST_YIN);
                vp_launch_yin_decide(st, g, Sp, c.voice, e->dGate, e->dYinP, e->dYinE, e->dPeriod, e->dYFlags, e->dList, c.listCount,
                                     e->maxList, 0, 2, e->dYinPending, tCount + 1, tFlag, tList, tCount);
                stage_mark(e, ST_YIN_DECIDE);
                e->launches += 3;
            } else {
                vp_launch_yin_corr(st, g, Sp, c.voice, e->dYinP, e->dYinE, 0, 0, nullptr, nullptr);
                stage_mark(e, ST_YIN);
                vp_launch_yin_decide(st, g, Sp, c.voice, e->dGate, e->dYinP, e->dYinE, e->dPeriod, e->dYFlags, e->dList, c.listCount,
                                     e->maxList, 0, 0, nullptr, nullptr, nullptr, nullptr, nullptr);
                stage_mark(e, ST_YIN_DECIDE);
                e->launches++;
            }
        }
        vp_launch_yin_recheck(st, g, Sp, c.voice, e->dGate, e->dPeriod, e->dYFlags, e->dList, c.listCount, e->maxList);
        stage_mark(e, ST_YIN64);
        e->launches += 2;
    }
    VP_CUDA_OK(cudaEventRecord(e->evYin[c.slot], st));
    return VP_OK;
}

// phase S: everything of the pitch corrector after the YIN decision. On the side stream when the vocoder runs in this pass
// (it then hides under the vocoder kernels), else on the main stream.
static int pass_S(vp_engine* e, PassCtx& c) {
    const VPGeom& g = c.g;
    const int Sp = c.Sp;
    const size_t sb = c.sb;
    const long long rowsP = g.nFramesP + VP_PC;
    const bool side = e->overlapMarks && g.vocOn && g.pitchOn && g.nFramesP > 0;
    cudaStream_t q = side ? e->st2 : e->st;
    c.sideUsed = side;
    auto mark = [&](int stage) { if (side) side_mark(e, stage); else stage_mark(e, stage); };
    if (side) {
        VP_CUDA_OK(cudaStreamWaitEvent(q, e->evYin[c.slot], 0));
        // the pitch workspace (frame records, LPC rows, PSOLA output, pitch plane) is single: the previous pass's phase M
        // must have read it (mix, carried records, kept decisions)
        if (e->mixPending) VP_CUDA_OK(cudaStreamWaitEvent(q, e->evMix[c.slot ^ 1], 0));
    }
    if (!g.pitchOn) {
        // pitchBool off for these blocks: PitchProcess::silence() (PluginProcessor.cpp:218-221)
        vp_launch_marks_silence(q, e->cMarks + sb, Sp);
        e->launches++;
    }
    // (the chain first: it is the long, latency-bound part of this phase and starts the moment the fork allows; the carried
    // records occupy the rows in front of the ones it writes, and the cleared plane is only needed by phase P)
    if (g.pitchOn && g.nFramesP > 0) {
        if (side) side_mark(e, ST_MARKS);
        vp_launch_marks(q, g, c.tb, Sp, c.voice, e->dGate, e->dPeriod, e->dYFlags, e->dFrames, e->cMarks + sb);
        mark(ST_MARKS);
        e->launches++;
    }
    if (g.pitchMix) {
        if (side) side_mark(e, ST_CLEAR);
        vp_launch_carry_in(q, e->dFrames, e->cFrames + sb * VP_PC, Sp, (int)sizeof(vp_pitch_frame), (int)sizeof(vp_pitch_frame), VP_PC, rowsP);
        VP_CUDA_OK(cudaMemsetAsync(e->dOutP, 0, (size_t)Sp * g.wstride * sizeof(float), q));
        mark(ST_CLEAR);
    }
    if (side) {
        VP_CUDA_OK(cudaEventRecord(e->evMarks[c.slot], q));
        VP_CUDA_OK(cudaEventRecord(e->evSideDone[c.slot], q));
        e->sidePending = true;
    }
    return VP_OK;
}

// phase P (main stream): pitch synthesis
static int pass_P(vp_engine* e, PassCtx& c) {
    cudaStream_t st = e->st;
    const VPGeom& g = c.g;
    const int Sp = c.Sp;
    if (c.sideUsed) {
        VP_CUDA_OK(cudaStreamWaitEvent(st, e->evSideDone[c.slot], 0));
        stage_mark(e, ST_OTHER);  // whatever of the mark chain was not hidden under the vocoder kernels
    }
    if (g.pitchMix) {
        vp_launch_pitch_lpc(st, g, c.tb, Sp, c.voice, e->dFrames, e->dRP, e->dAP);
        stage_mark(e, ST_PLPC);
        vp_launch_pitch_psola(st, g, c.tb, Sp, c.voice, e->dFrames, e->dAP, e->dOutE);
        stage_mark(e, ST_PFRAME);
        // one gain for every chunk of the call: every stream has it in every block, and the carried chunks went out with it
        // (a captured graph reads the table: a gain change between blocks must not need a new capture)
        const bool uniform = e->callPgUniform && (e->pgCarryAny || e->pgCarry == e->callPg) && !e->capturing;
        const int hc = e->histCur;
        vp_launch_pitch_iir(st, g, c.tb, Sp, e->dFrames, e->dAP, e->dOutE, e->dOutP, uniform ? &e->callPg : nullptr,
                            e->cPG[hc] + c.sb * VP_PC * 4, e->cPG[hc ^ 1] + c.sb * VP_PC * 4);
        stage_mark(e, ST_PIIR);
        e->launches += 4;
        e->yinFrames += (size_t)Sp * g.nFramesP;
    }
    return VP_OK;
}

// phase V (main stream): the vocoder. part = 1: up to and including the autocorrelation, 2: the rest, 0: everything
static int pass_V(vp_engine* e, PassCtx& c, int part) {
    cudaStream_t st = e->st;
    const VPGeom& g = c.g;
    const int Sp = c.Sp;
    const size_t sb = c.sb;
    const int synV1 = g.synV + 1, synS1 = g.synS + 1, capV1 = e->capV + 1, capS1 = e->capS + 1;
    const long long rowsV = g.nFramesV + VP_VC;
    float* vDst = e->dOutV;
    if (g.vocOn && part != 2) {
        // carried rows of the previous call in front of this call's rows (coefficient rows: from the store's width to the
        // call's row width; rows of narrower orders are zero padded)
        vp_launch_carry_in(st, e->dAV, e->cAV + sb * VP_VC * capV1, Sp, 8 * synV1, 8 * capV1, VP_VC, rowsV);
        vp_launch_carry_in(st, e->dAS, e->cAS + sb * VP_VC * capS1, Sp, 8 * synS1, 8 * capS1, VP_VC, rowsV);
        vp_launch_carry_in(st, e->dEeS, e->cEeS + sb * VP_VC, Sp, 8, 8, VP_VC, rowsV);
        vp_launch_carry_in(st, e->dGs, e->cG + sb * VP_VC, Sp, 8, 8, VP_VC, rowsV);
        if (vp_voc_synth_needs_clear(g)) {
            VP_CUDA_OK(cudaMemsetAsync(e->dOutV, 0, (size_t)Sp * g.wstride * sizeof(float), st));
            stage_mark(e, ST_CLEAR);
        }
        if (g.nFramesV > 0) {
            vp_launch_voc_autocorr(st, g, c.tb, Sp, c.voice, c.synthL, e->dGate, e->dRV, e->dRS);
            stage_mark(e, ST_VOC_AC);
            e->launches += 1;
        }
    }
    if (part == 1) return VP_OK;
    if (g.vocOn) {
        if (g.nFramesV > 0) {
            vp_launch_voc_levinson(st, g, c.tb, Sp, c.voice, c.synthL, e->dGate, e->dRV, e->dRS, e->dAV, e->dAS, e->dEeV, e->dEeS);
            vp_launch_voc_gain(st, g, c.tb, Sp, e->dEeV, e->dEeS, e->dG, e->dGs, e->cGainHist + sb * 20);
            stage_mark(e, ST_VOC_LEV);
            e->launches += 2;
        }
        vp_launch_voc_synth(st, g, c.tb, Sp, c.synthL, e->dAV, e->dAS, e->dEeS, e->dGs, vDst);
        stage_mark(e, ST_VOC_SYN);
        e->launches += 1;
    } else if (g.vocMix) {
        VP_CUDA_OK(cudaMemsetAsync(e->dOutV, 0, (size_t)Sp * g.wstride * sizeof(float), st));
        stage_mark(e, ST_CLEAR);
    }
    if (g.vocMix) {
        bool any = false;
        for (int j = 0; j < VP_ORPH; ++j) any = any || g.orphPos[j] != VP_NOFRAME;
        if (any) {  // frames of earlier calls that a vocBool-off stretch left off this call's grid
            vp_launch_voc_orphans(st, g, c.tb, Sp, c.synthL, e->oAV + sb * VP_ORPH * capV1, e->oAS + sb * VP_ORPH * capS1, e->oEeS + sb * VP_ORPH,
                                  e->oG + sb * VP_ORPH, vDst, e->capV, e->capS);
            stage_mark(e, ST_VOC_SYN);
            e->launches += 1;
        }
    }
    if (g.vocOn) {  // the vocoder's carried state: last rows of (carry ++ new); kept decisions
        vp_launch_carry_out(st, e->cAV + sb * VP_VC * capV1, e->dAV, Sp, 8 * synV1, 8 * capV1, VP_VC, g.nFramesV, rowsV);
        vp_launch_carry_out(st, e->cAS + sb * VP_VC * capS1, e->dAS, Sp, 8 * synS1, 8 * capS1, VP_VC, g.nFramesV, rowsV);
        vp_launch_carry_out(st, e->cEeS + sb * VP_VC, e->dEeS, Sp, 8, 8, VP_VC, g.nFramesV, rowsV);
        vp_launch_carry_out(st, e->cG + sb * VP_VC, e->dGs, Sp, 8, 8, VP_VC, g.nFramesV, rowsV);
        if (e->keepDecisions && g.nFramesV > 0) {
            const size_t w = (size_t)g.nFramesV * 8, sp = (size_t)rowsV * 8;
            VP_CUDA_OK(cudaMemcpy2DAsync(e->dEeVAll + sb * g.nFramesV, w, e->dEeV + VP_VC, sp, w, Sp, cudaMemcpyDeviceToDevice, st));
            VP_CUDA_OK(cudaMemcpy2DAsync(e->dEeSAll + sb * g.nFramesV, w, e->dEeS + VP_VC, sp, w, Sp, cudaMemcpyDeviceToDevice, st));
            VP_CUDA_OK(cudaMemcpy2DAsync(e->dGAll + sb * g.nFramesV, w, e->dG + VP_VC, sp, w, Sp, cudaMemcpyDeviceToDevice, st));
        }
        stage_mark(e, ST_OTHER);
    }
    return VP_OK;
}

// phase M (main stream): mix + egress and what the next call needs
static int pass_M(vp_engine* e, PassCtx& c) {
    cudaStream_t st = e->st;
    const VPGeom& g = c.g;
    const int Sp = c.Sp;
    const size_t sb = c.sb;
    const int hc = e->histCur;
    const long long rowsP = g.nFramesP + VP_PC;
    vp_launch_mix(st, g, c.tb, e->callAnyDry, Sp, c.voice, c.synthL, c.synthR, e->dOutV, e->dOutP, c.outL, c.outR);
    e->launches++;
    stage_mark(e, ST_MIX);
    if (g.pitchMix) vp_launch_carry_out(st, e->cFrames + sb * VP_PC, e->dFrames, Sp, (int)sizeof(vp_pitch_frame), (int)sizeof(vp_pitch_frame), VP_PC, g.nFramesP, rowsP);
    vp_launch_hist_update(st, e->cHist[hc ^ 1][0] + sb * e->H, g.histV, c.voice, Sp, e->H, g.n, g.stride);
    vp_launch_hist_update(st, e->cHist[hc ^ 1][1] + sb * e->H, g.histS, c.synthL, Sp, e->H, g.n, g.stride);
    // channel 1 of the side-chain ring is filled on every block whatever gainSynth is (MyBuffer.cpp:69-92): the history
    // follows the caller's right channel when there is one, else channel 0 (R == L), so that gainSynth can be automated on
    vp_launch_hist_update(st, e->cHist[hc ^ 1][2] + sb * e->H, g.histR, c.synthR ? c.synthR : c.synthL, Sp, e->H, g.n, g.stride);
    if (e->keepDecisions && g.pitchOn && g.nFramesP > 0)
        VP_CUDA_OK(cudaMemcpy2DAsync(e->dFramesAll + sb * g.nFramesP, (size_t)g.nFramesP * sizeof(vp_pitch_frame),
                                     e->dFrames + VP_PC, (size_t)rowsP * sizeof(vp_pitch_frame),
                                     (size_t)g.nFramesP * sizeof(vp_pitch_frame), Sp, cudaMemcpyDeviceToDevice, st));
    stage_mark(e, ST_OTHER);
    VP_CUDA_OK(cudaEventRecord(e->evMix[c.slot], st));
    e->mixPending = true;
    VP_CUDA_OK(vp_take_launch_error());
    VP_CUDA_OK(cudaGetLastError());
    return VP_OK;
}

// the phases of one pass
static int run_pass(vp_engine* e, const VPGeom& gIO, int Sp, int streamBase, const float* voice, const float* synthL,
                    const float* synthR, float* outL, float* outR) {
    PassCtx c;
    pass_init(e, c, gIO, Sp, streamBase, voice, synthL, synthR, outL, outR);
    int rc;
    // The mark chain is forked after the autocorrelation: it then runs next to the Levinson and synthesis kernels (long
    // enough to hide it), and the autocorrelation -- the step's largest kernel, the one the roofline line is about -- is
    // timed without a co-runner. The step time is the same wherever the chain overlaps (it costs its ~25 ms of issue slots).
    if ((rc = pass_A(e, c))) return rc;
    if (e->forkEarly) {  // developer A/B (VP_OVERLAP=y): chain forked right after YIN, next to the autocorrelation
        if ((rc = pass_S(e, c))) return rc;
        if ((rc = pass_V(e, c, 0))) return rc;
    } else {
        if ((rc = pass_V(e, c, 1))) return rc;
        VP_CUDA_OK(cudaEventRecord(e->evYin[c.slot], e->st));  // the fork point of phase S: now behind the autocorrelation
        if ((rc = pass_S(e, c))) return rc;
        if ((rc = pass_V(e, c, 2))) return rc;
    }
    if ((rc = pass_P(e, c))) return rc;
    return pass_M(e, c);
}

// Before the first pass of a call: what a block with vocBool / pitchBool off does to the state every stream shares.
// Returns the carry rows that have to move to the orphan store (the caller moves the device rows).
static int grid_begin(GridState& gs, int vocBool, int pitchBool, GridMove* moves) {
    const vp_sizes& z = gs.z;
    const long long u0 = gs.blocksDone * (long long)gs.B;
    int nMoves = 0;
    for (int j = 0; j < VP_ORPH; ++j)  // frames that have emitted everything
        if (gs.orphAbs[j] >= 0 && gs.orphAbs[j] + z.wlenV <= u0) gs.orphAbs[j] = -1;
    if (!vocBool && gs.alignedV > 0) {
        // VocoderProcess::process is skipped (PluginProcessor.cpp:214-215): its startSample freezes, so the frames carried
        // from the previous call are no longer on the grid of whatever call runs the vocoder next. Their rows move to the
        // orphan store (those that still reach into this call), where k_voc_orphans finishes them.
        for (int i = VP_VC - gs.alignedV; i < VP_VC; ++i) {
            const long long pos = gs.nextFrameV - (long long)(VP_VC - i) * z.hopV;
            if (pos + z.wlenV <= u0) continue;
            int slot = -1;
            for (int j = 0; j < VP_ORPH && slot < 0; ++j) if (gs.orphAbs[j] < 0) slot = j;
            if (slot < 0) continue;  // cannot happen: frames are at least a hop apart, at most 4 reach any position
            moves[nMoves].srcRow = i; moves[nMoves].dstSlot = slot; ++nMoves;
            gs.orphAbs[slot] = pos;
            gs.orphOrdV[slot] = gs.alignedOrdV[i];
            gs.orphOrdS[slot] = gs.alignedOrdS[i];
        }
        gs.alignedV = 0;
    }
    if (!pitchBool) {
        // PitchProcess::silence() (PitchProcess.cpp:146-158): the chunks of a frame in flight that have not been handled yet
        // find anMarks empty and do nothing (:253-271); the chunks handled before this block keep their output
        for (int j = 0; j < VP_PC; ++j) {
            if (gs.carryAbsP[j] < 0) continue;
            int done = 0;
            for (int n = 0; n < 4; ++n) if (gs.carryAbsP[j] + (long long)n * z.chunk < u0) ++done;
            gs.carryLimP[j] = std::min(gs.carryLimP[j], done);
        }
    }
    return nMoves;
}

// call-local frame grids of a call of n samples from the grid state (the timeline continues where the previous call ended)
static void grid_geom(const GridState& gs, VPGeom* g) {
    const vp_sizes& z = gs.z;
    const long long u0 = gs.blocksDone * (long long)gs.B;
    g->hasPrev = gs.blocksDone > 0;
    // vocoder (VocoderProcess::process, :173-183): frames at nextFrameV + k hop while they start inside the call
    g->synV = g->ordV; g->synS = g->ordS;
    if (g->vocOn) {
        g->offV = (int)(gs.nextFrameV - u0);
        g->nFramesV = (g->n > g->offV) ? (int)((g->n - g->offV + z.hopV - 1) / z.hopV) : 0;
        g->kV0 = gs.alignedV;  // carried rows -kV0 .. -1 are frames on this grid
        for (int i = VP_VC - gs.alignedV; i < VP_VC; ++i) {
            g->synV = std::max(g->synV, gs.alignedOrdV[i]);
            g->synS = std::max(g->synS, gs.alignedOrdS[i]);
        }
    } else {
        g->offV = 0; g->nFramesV = 0; g->kV0 = 0;
    }
    // Rows are at least as wide as the tuned kernels' orders (40 / 5): a narrower order rides along zero padded, and the
    // register-resident synthesis kernel serves every lpcVoice <= 40, lpcSynth <= 5 (the taps beyond the order are exact zeros)
    if (g->synV < 40) g->synV = 40;
    if (g->synS < 5) g->synS = 5;
    bool orphLive = false;
    for (int j = 0; j < VP_ORPH; ++j) {
        const bool live = gs.orphAbs[j] >= 0 && gs.orphAbs[j] + z.wlenV > u0;
        g->orphPos[j] = live ? (int)(gs.orphAbs[j] - u0) : VP_NOFRAME;
        g->orphOrdV[j] = gs.orphOrdV[j]; g->orphOrdS[j] = gs.orphOrdS[j];
        orphLive = orphLive || live;
    }
    g->vocMix = g->vocOn || orphLive;
    // pitch (PitchProcess::process, :166-196): a frame starts at the chunk for which nChunk is 0 or 3
    if (g->pitchOn) {
        const int j0 = (gs.nChunk == 0 || gs.nChunk == 3) ? 0 : 3 - gs.nChunk;
        g->offP = (int)(gs.nextChunkP + (long long)j0 * z.chunk - u0);
        g->nFramesP = (g->n > g->offP) ? (int)((g->n - g->offP + z.hopP - 1) / z.hopP) : 0;
    } else {
        g->offP = 0; g->nFramesP = 0;
    }
    g->fP0 = 0;
    bool carryLive = false;
    for (int j = 0; j < VP_PC; ++j) {
        const bool have = gs.carryAbsP[j] >= 0;
        g->carryPosP[j] = have ? (int)(gs.carryAbsP[j] - u0) : VP_NOFRAME;
        g->carryLimP[j] = have ? gs.carryLimP[j] : 0;
        // chunks are added to the output when they are handled, also beyond the block (MyBuffer::addOutSample): a carried
        // frame still owns positions of this call while one of its processed chunks reaches past the call's start
        if (have && g->carryLimP[j] > 0 && g->carryPosP[j] + (long long)std::min(g->carryLimP[j], 4) * z.chunk > 0) carryLive = true;
    }
    g->pitchMix = g->pitchOn || carryLive;
}

// after the last pass of a call: the timeline and the frame grids have advanced
static void grid_finish(GridState& gs, const VPGeom& g) {
    const vp_sizes& z = gs.z;
    const long long u0 = gs.blocksDone * (long long)gs.B;
    if (g.vocOn) {
        // orders of the rows the device carried out: the last VP_VC of (carried ++ new)
        int ov[2 * VP_VC], os[2 * VP_VC], cnt = 0;
        for (int i = VP_VC - gs.alignedV; i < VP_VC; ++i) { ov[cnt] = gs.alignedOrdV[i]; os[cnt] = gs.alignedOrdS[i]; ++cnt; }
        const int add = std::min(g.nFramesV, VP_VC);
        for (int i = 0; i < add; ++i) { ov[cnt] = g.ordV; os[cnt] = g.ordS; ++cnt; }
        const int keep = std::min(cnt, VP_VC);
        for (int i = 0; i < keep; ++i) { gs.alignedOrdV[VP_VC - keep + i] = ov[cnt - keep + i]; gs.alignedOrdS[VP_VC - keep + i] = os[cnt - keep + i]; }
        gs.alignedV = std::min(VP_VC, gs.alignedV + g.nFramesV);
        gs.nextFrameV = u0 + g.offV + (long long)g.nFramesV * z.hopV;
    } else {
        gs.nextFrameV += g.n;  // startSample is relative to the block: it does not move while process() is skipped
    }
    if (g.pitchOn) {
        // chunks that started inside the call (PitchProcess::process, :169-192), and nChunk after them
        const long long K = (gs.nextChunkP < u0 + g.n) ? (u0 + g.n - gs.nextChunkP + z.chunk - 1) / z.chunk : 0;
        gs.nextChunkP += K * z.chunk;
        if (K > 0) {  // nChunk: 0 -> 1 -> 2 -> 3 -> 1 -> 2 -> 3 ...
            int nc = gs.nChunk;
            const long long steps = (K > 6) ? 6 + (K - 6) % 3 : K;
            for (long long i = 0; i < steps; ++i) nc = (nc == 0 || nc == 3) ? 1 : nc + 1;
            gs.nChunk = nc;
        }
        // the records the device carried out: the last VP_PC of (carried ++ new)
        for (int f = std::max(0, g.nFramesP - VP_PC); f < g.nFramesP; ++f) {
            for (int j = 0; j + 1 < VP_PC; ++j) { gs.carryAbsP[j] = gs.carryAbsP[j + 1]; gs.carryLimP[j] = gs.carryLimP[j + 1]; }
            gs.carryAbsP[VP_PC - 1] = u0 + g.offP + (long long)f * z.hopP;
            gs.carryLimP[VP_PC - 1] = 4;
        }
    } else {
        gs.nextChunkP += g.n;
    }
    gs.blocksDone += g.nBlocks;
}

extern "C" int vp_grid_plan(double sampleRate, int samplesPerBlock, int nCalls, const int* nBlocks, const vp_params* params,
                           vp_call_plan* out) {
    if (nCalls < 0 || (nCalls > 0 && (!nBlocks || !params || !out))) return VP_E_ARG;
    GridState gs;
    if (vp_sizes_for(sampleRate, samplesPerBlock, 12, &gs.z) != VP_OK) return VP_E_ARG;
    gs.B = samplesPerBlock;
    gs.reset();
    for (int c = 0; c < nCalls; ++c) {
        if (nBlocks[c] <= 0) return VP_E_ARG;
        GridMove mv[VP_VC];
        const int nm = grid_begin(gs, params[c].vocBool, params[c].pitchBool, mv);
        VPGeom g;
        memset(&g, 0, sizeof g);
        g.B = gs.B; g.hopV = gs.z.hopV; g.wlenV = gs.z.wlenV; g.hopP = gs.z.hopP; g.L = gs.z.frameLenP; g.c = gs.z.chunk;
        g.nBlocks = nBlocks[c]; g.n = (long long)nBlocks[c] * gs.B;
        g.vocOn = params[c].vocBool != 0; g.pitchOn = params[c].pitchBool != 0;
        g.ordV = params[c].lpcVoice; g.ordS = params[c].lpcSynth;
        grid_geom(gs, &g);
        vp_call_plan& o = out[c];
        memset(&o, 0, sizeof o);
        o.firstBlock = gs.blocksDone; o.offV = g.offV; o.nFramesV = g.nFramesV; o.carriedV = g.kV0; o.rowOrderV = g.synV; o.rowOrderS = g.synS;
        o.offP = g.offP; o.nFramesP = g.nFramesP; o.vocMix = g.vocMix; o.pitchMix = g.pitchMix; o.rowsOrphaned = nm;
        for (int j = 0; j < VP_ORPH; ++j) if (g.orphPos[j] != VP_NOFRAME) o.orphansLive++;
        for (int j = 0; j < 2; ++j) { o.carryPosP[j] = g.carryPosP[j]; o.carryChunksP[j] = g.carryLimP[j]; }
        grid_finish(gs, g);
    }
    return VP_OK;
}

static void begin_call(vp_engine* e) {
    GridMove mv[VP_VC];
    const int nm = grid_begin(e->gs, e->prm.vocBool, e->prm.pitchBool, mv);
    const int capV1 = e->capV + 1, capS1 = e->capS + 1;
    for (int i = 0; i < nm; ++i) {
        vp_launch_row_move(e->st, e->oAV, e->cAV, e->S, 8 * capV1, VP_VC, mv[i].srcRow, VP_ORPH, mv[i].dstSlot);
        vp_launch_row_move(e->st, e->oAS, e->cAS, e->S, 8 * capS1, VP_VC, mv[i].srcRow, VP_ORPH, mv[i].dstSlot);
        vp_launch_row_move(e->st, e->oEeS, e->cEeS, e->S, 8, VP_VC, mv[i].srcRow, VP_ORPH, mv[i].dstSlot);
        vp_launch_row_move(e->st, e->oG, e->cG, e->S, 8, VP_VC, mv[i].srcRow, VP_ORPH, mv[i].dstSlot);
        e->launches += 4;
    }
}

static void finish_call(vp_engine* e, const VPGeom& g) {
    grid_finish(e->gs, g);
    e->histCur ^= 1;
    // the frames carried out: all their emitted chunks went out with callPg if the call had it throughout and they start in
    // the call (or the chunks before it had it as well)
    const bool same = e->callPgUniform && (e->pgCarryAny || e->pgCarry == e->callPg || g.nFramesP >= VP_PC);
    e->pgCarry = same ? e->callPg : -1.0f;
    e->pgCarryAny = false;
}

static int check_process_args(vp_engine* e, int nBlocks, const float* voice, const float* synthL, const float* synthR,
                              float* outL, size_t stride) {
    if (!e) return VP_E_ARG;
    if (!e->prepared) return vp_err(e, VP_E_STATE, "vp_engine_prepare has not been called");
    if (e->failed) return vp_err(e, VP_E_STATE, "an earlier process call failed half way: the carried stream state is undefined, call vp_engine_reset");
    if (nBlocks <= 0 || nBlocks > e->maxBlocks) return vp_err(e, VP_E_ARG, "nBlocks outside (0, maxBlocks]");
    if (!voice || !synthL || !outL) return vp_err(e, VP_E_ARG, "voice, synthL and outL must be non-null");
    if (stride < (size_t)nBlocks * e->B) return vp_err(e, VP_E_ARG, "strideSamples < nBlocks * samplesPerBlock");
    (void)synthR;  // optional: without it the right side-chain channel equals the left one
    return VP_OK;
}

// [a, a + na) and [b, b + nb) floats overlap?
static bool ranges_overlap(const float* a, size_t na, const float* b, size_t nb) {
    if (!a || !b) return false;
    const uintptr_t a0 = (uintptr_t)a, a1 = a0 + na * sizeof(float), b0 = (uintptr_t)b, b1 = b0 + nb * sizeof(float);
    return a0 < b1 && b0 < a1;
}

extern "C" int vp_engine_process_device(vp_engine* e, int nBlocks, const float* voice, const float* synthL,
                                        const float* synthR, float* outL, float* outR, size_t stride) {
    int rc = check_process_args(e, nBlocks, voice, synthL, synthR, outL, stride);
    if (rc) return rc;
    {   // the mix kernel reads the delayed inputs while other threads already write the outputs: no in-place use
        const size_t span = (size_t)(e->S - 1) * stride + (size_t)nBlocks * e->B;
        const float* ins[3] = {voice, synthL, synthR};
        float* outs[2] = {outL, outR};
        for (const float* in : ins) for (float* out : outs)
            if (ranges_overlap(in, span, out, span)) return vp_err(e, VP_E_ARG, "output arrays must not overlap the input arrays");
        if (ranges_overlap(outL, span, outR, span)) return vp_err(e, VP_E_ARG, "outL and outR must not overlap");
    }
    VP_CUDA_OK(cudaSetDevice(e->device));
    if ((rc = plan_schedule(e, nBlocks))) return rc;
    if ((rc = upload_stream_params(e))) return rc;
    if ((rc = issue_schedule(e, nBlocks))) return rc;
    if ((rc = apply_stream_resets(e))) return rc;
    begin_call(e);
    VPGeom g;
    make_geom(e, nBlocks, stride, &g);
    e->lastBlocks = nBlocks;
    e->lastG = g;
    e->passCount = 0;
    if (!e->timingOpen) { e->evUsed = 0; e->evSideUsed = 0; VP_CUDA_OK(cudaEventRecord(e->evT0, e->st)); e->timingOpen = e->timingAccumulate; }
    e->sidePending = e->mixPending = false;
    for (int s0 = 0; s0 < e->S; s0 += e->Sc) {
        const int Sp = std::min(e->Sc, e->S - s0);
        const size_t off = (size_t)s0 * stride;
        rc = run_pass(e, g, Sp, s0, voice + off, synthL + off, synthR ? synthR + off : nullptr, outL + off, outR ? outR + off : nullptr);
        if (rc) { e->failed = true; return rc; }  // some streams' carried state has advanced, others' has not
    }
    finish_call(e, g);
    VP_CUDA_OK(cudaEventRecord(e->evT1, e->st));
    return VP_OK;
}

extern "C" int vp_engine_sync(vp_engine* e) {
    if (!e) return VP_E_ARG;
    VP_CUDA_OK(cudaSetDevice(e->device));
    VP_CUDA_OK(cudaStreamSynchronize(e->st));
    VP_CUDA_OK(cudaStreamSynchronize(e->st2));
    VP_CUDA_OK(cudaStreamSynchronize(e->stIn));
    VP_CUDA_OK(cudaStreamSynchronize(e->stOut));
    // guard: the FP64 re-decision list holds every frame of a pass, so it cannot overflow; should a count ever exceed it
    // (a frame listed twice), frames would have kept their unverified FP32 decision -- that is an error, not a truncation
    if (e->prepared && e->dListCount && e->passCount > 0 && e->prm.pitchBool) {
        int h[1024];
        const int np = e->passCount < 1024 ? e->passCount : 1024;
        VP_CUDA_OK(cudaMemcpy(h, e->dListCount, sizeof(int) * (size_t)np, cudaMemcpyDeviceToHost));
        for (int i = 0; i < np; ++i)
            if (h[i] > e->maxList) { e->failed = true; return vp_err(e, VP_E_STATE, "YIN re-decision list overflow: results of this call are not verified"); }
    }
    return VP_OK;
}

extern "C" int vp_engine_get_info(const vp_engine* e, int* streamsPerPass, int* historySamples, size_t* workspaceBytes) {
    if (!e) return VP_E_ARG;
    if (!e->prepared) return VP_E_STATE;
    if (streamsPerPass) *streamsPerPass = e->Sc;
    if (historySamples) *historySamples = e->H;
    if (workspaceBytes) *workspaceBytes = e->workspace;
    return VP_OK;
}

// Host path: slices of Sh streams, H2D on stIn, compute on st, D2H on stOut, three slice buffers in rotation.
// pcm16: the host arrays are 16-bit PCM; they cross the link as such (6 instead of 12 bytes per sample for the default
// mono-voice + one side-chain channel in, one channel out) and are converted on the device.
static int process_host_impl(vp_engine* e, int nBlocks, const void* voiceV, const void* synthLV, const void* synthRV, void* outLV,
                             void* outRV, size_t stride, bool pcm16) {
    int rc = check_process_args(e, nBlocks, (const float*)voiceV, (const float*)synthLV, (const float*)synthRV, (float*)outLV, stride);
    if (rc) return rc;
    VP_CUDA_OK(cudaSetDevice(e->device));
    if ((rc = plan_schedule(e, nBlocks))) return rc;
    const long long n = (long long)nBlocks * e->B;
    const bool synthOn = e->callAnySynth;  // (some block of some stream has the dry side-chain on)
    const size_t esz = pcm16 ? sizeof(int16_t) : sizeof(float);
    const char *voice = (const char*)voiceV, *synthL = (const char*)synthLV, *synthR = (const char*)synthRV;
    char *outL = (char*)outLV, *outR = (char*)outRV;
    if (e->Sh == 0) {
        // slice = at most Sc streams and at most ~3 GiB per array: large enough that a slice's vocoder kernels outlast
        // its (latency-bound, side-stream) pitch-mark chain, small enough that pipeline fill / drain stay short
        long long Sh = std::max<long long>(1, ((long long)3 << 28) / ((long long)e->maxBlocks * e->B));
        if (Sh > 32) Sh &= ~31LL;
        Sh = std::min<long long>(Sh, e->Sc);
        Sh = std::min<long long>(Sh, (e->S + 2) / 3 > 0 ? (e->S + 2) / 3 : 1);
        if (Sh < 1) Sh = 1;
        const size_t cnt = (size_t)Sh * (size_t)e->maxBlocks * e->B;
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 2; ++j) if ((rc = wsalloc(e, &e->hIn[i][j], cnt))) return rc;
            if ((rc = wsalloc(e, &e->hOut[i][0], cnt))) return rc;
        }
        e->Sh = (int)Sh;
    }
    // the right side-chain travels whenever the caller has one (its ring is filled whatever gainSynth is); the right
    // output only when some stream mixes the dry side-chain in (otherwise L == R; streams without it keep L == R)
    const bool haveR = synthR != nullptr;
    const size_t cnt = (size_t)e->Sh * (size_t)e->maxBlocks * e->B;
    if (haveR && !e->hIn[0][2])
        for (int i = 0; i < 3; ++i) if ((rc = wsalloc(e, &e->hIn[i][2], cnt))) return rc;
    if (synthOn && outR && !e->hOut[0][1])
        for (int i = 0; i < 3; ++i) if ((rc = wsalloc(e, &e->hOut[i][1], cnt))) return rc;
    if (pcm16) {  // 16-bit landing / take-off buffers beside the float ones
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < (haveR ? 3 : 2); ++j) if (!e->pIn[i][j] && (rc = wsalloc(e, &e->pIn[i][j], cnt))) return rc;
            for (int j = 0; j < ((synthOn && outR) ? 2 : 1); ++j) if (!e->pOut[i][j] && (rc = wsalloc(e, &e->pOut[i][j], cnt))) return rc;
        }
    }
    if ((rc = upload_stream_params(e))) return rc;
    if ((rc = issue_schedule(e, nBlocks))) return rc;
    if ((rc = apply_stream_resets(e))) return rc;
    begin_call(e);
    e->sidePending = e->mixPending = false;
    VPGeom g;
    make_geom(e, nBlocks, (size_t)n, &g);  // staged rows are dense
    e->lastBlocks = nBlocks;
    e->lastG = g;
    e->passCount = 0;
    const size_t rowB = (size_t)n * esz;
    int slice = 0;
    if (!e->timingOpen) { e->evUsed = 0; e->evSideUsed = 0; VP_CUDA_OK(cudaEventRecord(e->evT0, e->st)); e->timingOpen = e->timingAccumulate; }
    // Slice schedule: full slices of Sh streams, tapered at both ends (Sh/4, Sh/2, Sh ... Sh, Sh/2, Sh/4) -- the pipeline
    // (H2D of slice i+1 | kernels of slice i | D2H of slice i-1) is bound by the host link, so what is not overlapped is the
    // first upload and the last compute + download, and both shrink with the slice they belong to.
    std::vector<int> sizes;
    {
        const int Sh = e->Sh, q = std::max(1, Sh / 4), h = std::max(1, Sh / 2);
        int rem = e->S;
        const bool taper = e->S >= 3 * Sh && Sh >= 8;
        if (taper) { sizes.push_back(q); sizes.push_back(h); rem -= 2 * (q + h); }
        while (rem > 0) { const int k = std::min(Sh, rem); sizes.push_back(k); rem -= k; }
        if (taper) { sizes.push_back(h); sizes.push_back(q); }
    }
    // dense host rows (stride == n) go as ONE 1-D copy per array and slice: the strided 2-D form is slower on the upload
    // (39.7 vs 48.6 GB/s with the download running, profiles/link_probe_1gpu_r02a.jsonl)
    auto copyIn = [&](void* dst, const char* src, int Sp) -> cudaError_t {
        if (stride == (size_t)n) return cudaMemcpyAsync(dst, src, rowB * (size_t)Sp, cudaMemcpyHostToDevice, e->stIn);
        return cudaMemcpy2DAsync(dst, rowB, src, stride * esz, rowB, Sp, cudaMemcpyHostToDevice, e->stIn);
    };
    auto copyOut = [&](char* dst, const void* src, int Sp) -> cudaError_t {
        if (stride == (size_t)n) return cudaMemcpyAsync(dst, src, rowB * (size_t)Sp, cudaMemcpyDeviceToHost, e->stOut);
        return cudaMemcpy2DAsync(dst, stride * esz, src, rowB, rowB, Sp, cudaMemcpyDeviceToHost, e->stOut);
    };
    int s0 = 0;
    for (size_t si = 0; si < sizes.size(); s0 += sizes[si], ++si, ++slice) {
        const int Sp = sizes[si];
        const int bi = slice % 3;
        // the buffers of this rotation slot must have been drained (D2H of slice-3 done)
        if (slice >= 3) VP_CUDA_OK(cudaStreamWaitEvent(e->stIn, e->evOut[bi], 0));
        const size_t hoff = (size_t)s0 * stride * esz;
        const long long cntS = (long long)Sp * n;
        const char* srcs[3] = {voice, synthL, haveR ? synthR : nullptr};
        for (int j = 0; j < 3; ++j) {
            if (!srcs[j]) continue;
            if (pcm16) {
                VP_CUDA_OK(copyIn(e->pIn[bi][j], srcs[j] + hoff, Sp));
                vp_launch_pcm16_to_float(e->stIn, e->hIn[bi][j], e->pIn[bi][j], cntS);
                e->launches++;
            } else {
                VP_CUDA_OK(copyIn(e->hIn[bi][j], srcs[j] + hoff, Sp));
            }
        }
        VP_CUDA_OK(cudaEventRecord(e->evIn[bi], e->stIn));
        VP_CUDA_OK(cudaStreamWaitEvent(e->st, e->evIn[bi], 0));
        const bool wantR = synthOn && outR;
        rc = run_pass(e, g, Sp, s0, e->hIn[bi][0], e->hIn[bi][1], haveR ? e->hIn[bi][2] : nullptr, e->hOut[bi][0], wantR ? e->hOut[bi][1] : nullptr);
        if (rc) { e->failed = true; return rc; }
        if (pcm16) {
            vp_launch_float_to_pcm16(e->st, e->pOut[bi][0], e->hOut[bi][0], cntS);
            if (wantR) vp_launch_float_to_pcm16(e->st, e->pOut[bi][1], e->hOut[bi][1], cntS);
            e->launches += wantR ? 2 : 1;
        }
        VP_CUDA_OK(cudaEventRecord(e->evComp[bi], e->st));
        VP_CUDA_OK(cudaStreamWaitEvent(e->stOut, e->evComp[bi], 0));
        const void* oL = pcm16 ? (const void*)e->pOut[bi][0] : (const void*)e->hOut[bi][0];
        const void* oR = wantR ? (pcm16 ? (const void*)e->pOut[bi][1] : (const void*)e->hOut[bi][1]) : oL;  // L == R unless the dry synth is mixed in (MyBuffer.cpp:380-448)
        VP_CUDA_OK(copyOut(outL + hoff, oL, Sp));
        if (outR) VP_CUDA_OK(copyOut(outR + hoff, oR, Sp));
        VP_CUDA_OK(cudaEventRecord(e->evOut[bi], e->stOut));
    }
    finish_call(e, g);
    VP_CUDA_OK(cudaEventRecord(e->evT1, e->st));
    VP_CUDA_OK(vp_take_launch_error());
    return vp_engine_sync(e);
}

extern "C" int vp_engine_process_host(vp_engine* e, int nBlocks, const float* voice, const float* synthL,
                                      const float* synthR, float* outL, float* outR, size_t stride) {
    return process_host_impl(e, nBlocks, voice, synthL, synthR, outL, outR, stride, false);
}

extern "C" int vp_engine_process_host_pcm16(vp_engine* e, int nBlocks, const int16_t* voice, const int16_t* synthL,
                                            const int16_t* synthR, int16_t* outL, int16_t* outR, size_t stride) {
    return process_host_impl(e, nBlocks, voice, synthL, synthR, outL, outR, stride, true);
}

// ---- low-latency streaming --------------------------------------------------------------------------------------
extern "C" int vp_engine_stream_buffers(vp_engine* e, float** voice, float** synthL, float** outL) {
    if (!e) return VP_E_ARG;
    if (!e->prepared) return vp_err(e, VP_E_STATE, "vp_engine_prepare has not been called");
    VP_CUDA_OK(cudaSetDevice(e->device));
    const size_t bytes = (size_t)e->S * e->B * sizeof(float);
    if (!e->sHostV) {
        VP_CUDA_OK(cudaHostAlloc((void**)&e->sHostV, bytes, cudaHostAllocDefault));
        VP_CUDA_OK(cudaHostAlloc((void**)&e->sHostS, bytes, cudaHostAllocDefault));
        VP_CUDA_OK(cudaHostAlloc((void**)&e->sHostO, bytes, cudaHostAllocDefault));
        VP_CUDA_OK(cudaMalloc((void**)&e->sDevV, bytes));
        VP_CUDA_OK(cudaMalloc((void**)&e->sDevS, bytes));
        VP_CUDA_OK(cudaMalloc((void**)&e->sDevO, bytes));
        memset(e->sHostV, 0, bytes); memset(e->sHostS, 0, bytes); memset(e->sHostO, 0, bytes);
    }
    if (voice) *voice = e->sHostV;
    if (synthL) *synthL = e->sHostS;
    if (outL) *outL = e->sHostO;
    return VP_OK;
}

extern "C" int vp_engine_stream_block(vp_engine* e) {
    if (!e) return VP_E_ARG;
    if (!e->prepared || !e->sHostV) return vp_err(e, VP_E_STATE, "call vp_engine_prepare and vp_engine_stream_buffers first");
    VP_CUDA_OK(cudaSetDevice(e->device));
    // the block's scheduled changes go into the [S] table here (a one-block call has no event after its first block)
    { int rc = plan_schedule(e, 1); if (rc) return rc; }
    if (e->anySynth) return vp_err(e, VP_E_ARG, "streaming mode carries side-chain channel 0 only: gainSynth must be off on every stream");
    // per-stream key and gains are table data: a change is uploaded here, outside the graph, and needs no new capture
    // so are per-stream resets: one kernel before the graph, the block phase (the graph's key) does not change
    { int rc = upload_stream_params(e); if (!rc) rc = apply_stream_resets(e); if (rc) return rc; }
    begin_call(e);
    e->sidePending = e->mixPending = false;
    VPGeom g;
    make_geom(e, 1, (size_t)e->B, &g);
    e->lastBlocks = 1;
    e->lastG = g;
    // everything that shapes the launch sequence or is baked into kernel arguments
    // (per-stream orders are table data; whether they differ, and the row orders, select the kernels -- the pitch orders as
    // well: a reset that gives a stream a new lpcPitch changes at most that signature)
    std::vector<long long> key = {e->gs.blocksDone > 0 ? 1 : 0, e->histCur, g.offV, g.offP, g.nFramesV, g.nFramesP, g.kV0, g.synV, g.synS,
                                  g.vocOn, g.pitchOn, g.vocMix, g.pitchMix, e->callAnyDry, g.ordV, g.ordS, g.ordTab, g.ordP, g.ordTabP};
    for (int j = 0; j < VP_ORPH; ++j) { key.push_back(g.orphPos[j]); key.push_back(g.orphOrdV[j]); key.push_back(g.orphOrdS[j]); }
    for (int j = 0; j < VP_PC; ++j) { key.push_back(g.carryPosP[j]); key.push_back(g.carryLimP[j]); }
    auto it = e->graphs.find(key);
    if (it == e->graphs.end()) {
        const bool st = e->stageTiming;
        e->stageTiming = false;  // event queries make no sense inside a graph
        e->capturing = true;
        const size_t bytes = (size_t)e->S * e->B * sizeof(float);
        cudaGraph_t graph = nullptr;
        VP_CUDA_OK(cudaStreamBeginCapture(e->st, cudaStreamCaptureModeGlobal));
        int rc = VP_OK;
        cudaError_t ce = cudaMemcpyAsync(e->sDevV, e->sHostV, bytes, cudaMemcpyHostToDevice, e->st);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(e->sDevS, e->sHostS, bytes, cudaMemcpyHostToDevice, e->st);
        if (ce == cudaSuccess) {
            for (int s0 = 0; s0 < e->S && rc == VP_OK; s0 += e->Sc) {
                const int Sp = std::min(e->Sc, e->S - s0);
                const size_t off = (size_t)s0 * e->B;
                e->passCount = 0;
                rc = run_pass(e, g, Sp, s0, e->sDevV + off, e->sDevS + off, nullptr, e->sDevO + off, nullptr);
            }
            if (rc == VP_OK) ce = cudaMemcpyAsync(e->sHostO, e->sDevO, bytes, cudaMemcpyDeviceToHost, e->st);
        }
        cudaError_t ce2 = cudaStreamEndCapture(e->st, &graph);
        e->stageTiming = st;
        e->capturing = false;
        if (rc != VP_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (ce != cudaSuccess) { if (graph) cudaGraphDestroy(graph); return vp_fail(e, ce, "stream capture", __FILE__, __LINE__); }
        if (ce2 != cudaSuccess) return vp_fail(e, ce2, "cudaStreamEndCapture", __FILE__, __LINE__);
        cudaGraphExec_t exec = nullptr;
        ce = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) return vp_fail(e, ce, "cudaGraphInstantiate", __FILE__, __LINE__);
        it = e->graphs.emplace(key, exec).first;
        e->graphCaptures++;
    }
    VP_CUDA_OK(cudaGraphLaunch(it->second, e->st));
    e->graphLaunches++;
    finish_call(e, g);
    VP_CUDA_OK(cudaStreamSynchronize(e->st));
    return VP_OK;
}

extern "C" int vp_engine_stream_stats(const vp_engine* e, uint64_t* graphLaunches, uint64_t* graphCaptures) {
    if (!e) return VP_E_ARG;
    if (graphLaunches) *graphLaunches = e->graphLaunches;
    if (graphCaptures) *graphCaptures = e->graphCaptures;
    return VP_OK;
}

extern "C" int vp_engine_get_pitch_frames(vp_engine* e, int stream, vp_pitch_frame* out, int cap, int* nFrames) {
    if (!e || stream < 0) return VP_E_ARG;
    if (!e->prepared || e->lastBlocks == 0 || !e->keepDecisions) return VP_E_STATE;
    if (stream >= e->S) return VP_E_ARG;
    VP_CUDA_OK(cudaSetDevice(e->device));
    const VPGeom& g = e->lastG;
    const int nP = g.pitchOn ? g.nFramesP : 0;
    if (nFrames) *nFrames = nP;
    if (out && cap > 0 && nP > 0) {
        VP_CUDA_OK(cudaStreamSynchronize(e->st));
        VP_CUDA_OK(cudaMemcpy(out, e->dFramesAll + (size_t)stream * g.nFramesP, (size_t)std::min(cap, nP) * sizeof(vp_pitch_frame),
                              cudaMemcpyDeviceToHost));
    }
    return VP_OK;
}

extern "C" int vp_engine_get_voc_frames(vp_engine* e, int stream, int cap, int* nFrames, uint8_t* gated, double* EeVoice,
                                        double* EeSynth, double* gOut) {
    if (!e || stream < 0) return VP_E_ARG;
    if (!e->prepared || e->lastBlocks == 0 || !e->keepDecisions) return VP_E_STATE;
    if (stream >= e->S) return VP_E_ARG;
    VP_CUDA_OK(cudaSetDevice(e->device));
    const VPGeom& g = e->lastG;
    const int nV = g.vocOn ? g.nFramesV : 0;
    if (nFrames) *nFrames = nV;
    const int m = std::min(cap, nV);
    if (m <= 0) return VP_OK;
    VP_CUDA_OK(cudaStreamSynchronize(e->st));
    const size_t off = (size_t)stream * g.nFramesV;
    if (EeVoice) VP_CUDA_OK(cudaMemcpy(EeVoice, e->dEeVAll + off, (size_t)m * 8, cudaMemcpyDeviceToHost));
    if (EeSynth) VP_CUDA_OK(cudaMemcpy(EeSynth, e->dEeSAll + off, (size_t)m * 8, cudaMemcpyDeviceToHost));
    if (gOut) VP_CUDA_OK(cudaMemcpy(gOut, e->dGAll + off, (size_t)m * 8, cudaMemcpyDeviceToHost));
    if (gated) {
        std::vector<uint8_t> gb(g.nBlocks);
        VP_CUDA_OK(cudaMemcpy(gb.data(), e->dGateAll + (size_t)stream * g.nBlocks, (size_t)g.nBlocks, cudaMemcpyDeviceToHost));
        for (int k = 0; k < m; ++k) {
            const int b = (int)(((long long)k * g.hopV + g.offV) / g.B);
            gated[k] = (gb[b] & (VP_GATE_VOICE | VP_GATE_SYNTH)) ? 1 : 0;
        }
    }
    return VP_OK;
}

extern "C" int vp_engine_get_stats(const vp_engine* e, uint64_t* launches, uint64_t* yinRechecked, uint64_t* yinFrames) {
    if (!e) return VP_E_ARG;
    if (launches) *launches = e->launches;
    if (yinFrames) *yinFrames = e->yinFrames;
    if (yinRechecked) {
        // re-check list counters of the passes of the most recent call
        uint64_t cnt = 0;
        if (e->dListCount && e->prepared && e->passCount > 0) {
            int h[1024];
            cudaSetDevice(e->device);
            cudaStreamSynchronize(e->st);
            const int np = e->passCount < 1024 ? e->passCount : 1024;
            cudaMemcpy(h, e->dListCount, sizeof(int) * (size_t)np, cudaMemcpyDeviceToHost);
            for (int i = 0; i < np; ++i) cnt += (uint64_t)h[i];
        }
        *yinRechecked = cnt;
    }
    return VP_OK;
}

extern "C" const char* vp_stage_name(int stage) { return (stage >= 0 && stage < VP_NSTAGES) ? kStageNames[stage] : ""; }

extern "C" int vp_engine_last_timing_counts(vp_engine* e, int* stageCount) {
    if (!e || !stageCount) return VP_E_ARG;
    for (int i = 0; i < VP_NSTAGES; ++i) stageCount[i] = 0;
    for (size_t i = 1; i < e->evUsed; ++i) stageCount[e->evStage[i]]++;
    for (size_t i = 1; i < e->evSideUsed; i += 2) stageCount[e->evSideStage[i]]++;
    return VP_OK;
}

extern "C" int vp_engine_timing_reset(vp_engine* e, int accumulate) {
    if (!e) return VP_E_ARG;
    e->timingOpen = false;
    e->timingAccumulate = accumulate != 0;
    e->evUsed = 0;
    e->evSideUsed = 0;
    return VP_OK;
}

extern "C" int vp_engine_timer_record(vp_engine* e, int slot) {
    if (!e || slot < 0 || slot >= 8) return VP_E_ARG;
    VP_CUDA_OK(cudaSetDevice(e->device));
    VP_CUDA_OK(cudaEventRecord(e->evTimer[slot], e->st));
    return VP_OK;
}

extern "C" int vp_engine_timer_elapsed_ms(vp_engine* e, int slotA, int slotB, float* ms) {
    if (!e || !ms || slotA < 0 || slotA >= 8 || slotB < 0 || slotB >= 8) return VP_E_ARG;
    VP_CUDA_OK(cudaSetDevice(e->device));
    VP_CUDA_OK(cudaEventSynchronize(e->evTimer[slotB]));
    VP_CUDA_OK(cudaEventElapsedTime(ms, e->evTimer[slotA], e->evTimer[slotB]));
    return VP_OK;
}

extern "C" int vp_engine_last_timing(vp_engine* e, float* totalMs, float* stageMs) {
    if (!e) return VP_E_ARG;
    if (!e->prepared || e->lastBlocks == 0) return VP_E_STATE;
    VP_CUDA_OK(cudaSetDevice(e->device));
    VP_CUDA_OK(cudaEventSynchronize(e->evT1));
    if (totalMs) VP_CUDA_OK(cudaEventElapsedTime(totalMs, e->evT0, e->evT1));
    if (stageMs) {
        for (int i = 0; i < VP_NSTAGES; ++i) stageMs[i] = 0.f;
        for (size_t i = 1; i < e->evUsed; ++i) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, e->ev[i - 1], e->ev[i]) == cudaSuccess) stageMs[e->evStage[i]] += ms;
        }
        // the pitch-mark chain on the side stream: its own (start, end) pairs; it overlaps the vocoder stages
        for (size_t i = 1; i < e->evSideUsed; i += 2) {
            float ms = 0.f;
            cudaEventSynchronize(e->evSide[i]);
            if (cudaEventElapsedTime(&ms, e->evSide[i - 1], e->evSide[i]) == cudaSuccess) stageMs[e->evSideStage[i]] += ms;
        }
    }
    return VP_OK;
}

// ---- memory helpers ------------------------------------------------------------
extern "C" int vp_host_alloc(void** p, size_t bytes) {
    if (!p) return VP_E_ARG;
    if (cudaHostAlloc(p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); *p = nullptr; return VP_E_NOMEM; }
    return VP_OK;
}
extern "C" void vp_host_free(void* p) { if (p) cudaFreeHost(p); }
extern "C" int vp_device_alloc(vp_engine* e, void** p, size_t bytes) {
    if (!e || !p) return VP_E_ARG;
    VP_CUDA_OK(cudaSetDevice(e->device));
    VP_CUDA_OK(cudaMalloc(p, bytes));
    return VP_OK;
}
extern "C" void vp_device_free(vp_engine* e, void* p) { if (e && p) { cudaSetDevice(e->device); cudaFree(p); } }
extern "C" int vp_memcpy_h2d(vp_engine* e, void* dst, const void* src, size_t bytes) {
    if (!e) return VP_E_ARG;
    VP_CUDA_OK(cudaSetDevice(e->device));
    VP_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, e->st));
    VP_CUDA_OK(cudaStreamSynchronize(e->st));
    return VP_OK;
}
extern "C" int vp_memcpy_d2h(vp_engine* e, void* dst, const void* src, size_t bytes) {
    if (!e) return VP_E_ARG;
    VP_CUDA_OK(cudaSetDevice(e->device));
    VP_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, e->st));
    VP_CUDA_OK(cudaStreamSynchronize(e->st));
    return VP_OK;
}

// ---- synthetic inputs (definitions: vp_synth.h, vp_synth_host.hpp) -----------------
extern "C" int vp_synth_host(double fs, int flavour, int first, int S, size_t nSamples, size_t stride, float* voice,
                             float* synthL, float* synthR) {
    return vps_fill_host(fs, flavour, first, S, nSamples, stride, voice, synthL, synthR) ? VP_OK : VP_E_ARG;
}

extern "C" int vp_synth_device(vp_engine* e, double fs, int flavour, int first, int S, size_t nSamples, size_t stride,
                               float* voice, float* synthL, float* synthR) {
    if (!e || !voice || S <= 0 || stride < nSamples || !(fs > 0)) return VP_E_ARG;
    VP_CUDA_OK(cudaSetDevice(e->device));
    std::vector<vp_synth_stream> ps;
    vps_make_streams(fs, flavour, first, S, nSamples, ps);
    vp_synth_stream* d = nullptr;
    VP_CUDA_OK(cudaMalloc((void**)&d, ps.size() * sizeof(vp_synth_stream)));
    VP_CUDA_OK(cudaMemcpy(d, ps.data(), ps.size() * sizeof(vp_synth_stream), cudaMemcpyHostToDevice));
    vp_launch_synth(e->st, d, S, (long long)nSamples, (long long)stride, voice, synthL, synthR);
    cudaError_t ce = cudaStreamSynchronize(e->st);
    cudaFree(d);
    if (ce != cudaSuccess) return vp_fail(e, ce, "k_synth", __FILE__, __LINE__);
    return VP_OK;
}

// ---- measurement -------------------------------------------------------------------
static int measure_peaks_impl(vp_engine* e, double* out4) {
    VP_CUDA_OK(cudaSetDevice(e->device));
    cudaDeviceProp prop;
    VP_CUDA_OK(cudaGetDeviceProperties(&prop, e->device));
    void* sink = nullptr;
    VP_CUDA_OK(cudaMalloc(&sink, 64));
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    for (int pass = 0; pass < 4; ++pass) {
        const int iters = (pass & 1) == 0 ? 4096 : 1024;
        double best = 0;
        for (int rep = 0; rep < 4; ++rep) {
            cudaEventRecord(a, e->st);
            if (pass == 0) vp_launch_peak_fp32(e->st, (float*)sink, iters, blocks, threads);
            else if (pass == 1) vp_launch_peak_fp64(e->st, (double*)sink, iters, blocks, threads);
            else if (pass == 2) vp_launch_peak2_fp32(e->st, (float*)sink, iters, blocks, threads);
            else vp_launch_peak2_fp64(e->st, (double*)sink, iters, blocks, threads);
            cudaEventRecord(b, e->st);
            cudaEventSynchronize(b);
            float ms = 0;
            cudaEventElapsedTime(&ms, a, b);
            const double ops = (double)blocks * threads * (double)iters * 16.0 * 8.0;
            if (rep > 0 && ms > 0) best = std::max(best, ops / (ms * 1e-3));
        }
        out4[pass] = best;
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaFree(sink);
    VP_CUDA_OK(cudaGetLastError());
    return VP_OK;
}

extern "C" int vp_measure_peaks(vp_engine* e, double* fp32, double* fp64) {
    if (!e) return VP_E_ARG;
    double v[4];
    int rc = measure_peaks_impl(e, v);
    if (rc) return rc;
    if (fp32) *fp32 = v[0];
    if (fp64) *fp64 = v[1];
    return VP_OK;
}

extern "C" int vp_measure_peaks2(vp_engine* e, double* fp32TwoOperand, double* fp64TwoOperand) {
    if (!e) return VP_E_ARG;
    double v[4];
    int rc = measure_peaks_impl(e, v);
    if (rc) return rc;
    if (fp32TwoOperand) *fp32TwoOperand = v[2];
    if (fp64TwoOperand) *fp64TwoOperand = v[3];
    return VP_OK;
}
