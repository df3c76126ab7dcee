// vp_facade.hpp -- header-only C++ facade over the C ABI (include/vp_engine.h) that keeps the reference's class and
// method names for the path VocoderAudioProcessor::processBlock drives, extended with a stream count:
//
//   reference (one plug-in instance)                      this facade (nStreams instances on one GPU)
//   ------------------------------------------------------------------------------------------------------------
//   MyBuffer        Source/MyBuffer.h:25-55               vpb200::MyBuffer
//   VocoderProcess  Source/VocoderProcess.h:29-34         vpb200::VocoderProcess
//   PitchProcess    Source/PitchProcess.h:40-48           vpb200::PitchProcess
//   Notes           Source/Notes.h:27-28                  vpb200::Notes
//   VocoderAudioProcessor::prepareToPlay / processBlock   vpb200::VocoderBatchProcessor::prepareToPlay / processBlock
//                   Source/PluginProcessor.cpp:144-184, :203-234
//
// The DSP classes do not compute on the host. The call sequence of processBlock -- fillInputBuffers, VocoderProcess::
// process, PitchProcess::process (or silence), addDryVoice, addSynth, fillOutputBuffer -- is recorded on the MyBuffer
// and executed as ONE engine call (all CUDA kernels of the block for all streams) when fillOutputBuffer asks for the
// block's output; the result is what the reference's sequence produces. Parameters are pushed (vp_params, and per stream
// the key and gains of each instance's parameter tree, vp_stream_params) instead of pulled through audioProcPtr->treeState. Errors are exceptions (vpb200::Error) carrying the ABI's status code; there
// is no CPU fallback.
#pragma once
#include <cmath>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/vp_engine.h"

namespace vpb200 {

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error("vp_engine error " + std::to_string(c) + ": " + m), code(c) {}
};

// Notes::key (Source/Notes.h:26)
enum key { A = 0, Bb, B, C, Db, D, Eb, E, F, Gb, G, Ab, Chrom };

// Host-side equal-tempered note table with the reference's arithmetic (Source/Notes.cpp:25-110). The engine builds
// the same table internally for its period -> (closestFreq, beta, periodNew) look-up.
class Notes {
public:
    void prepare(key k, double fMinIn, double fMaxIn) {
        currentKey = k; fMin = fMinIn; fMax = fMaxIn;
        buildFreqVect(k);
    }
    double getClosestFreq(const double& pitch, key k) {
        if (k != currentKey) { currentKey = k; buildFreqVect(k); }
        size_t idx = 0;
        while (idx < n && freq[idx] < pitch) ++idx;  // std::lower_bound (Notes.cpp:92)
        if (idx > 0) return (std::fabs(freq[idx] - pitch) <= std::fabs(freq[idx - 1] - pitch)) ? freq[idx] : freq[idx - 1];
        return freq[0];  // idx == n reads the popped slot freq[n], exactly like the reference (SURVEY App. B U6)
    }
    size_t size() const { return n; }
    const double* data() const { return freq; }

private:
    void buildFreqVect(key k) {
        static const int intervals[7] = {2, 2, 1, 2, 2, 2, 1};
        n = 0;
        int i = 0;
        double f = 27.5 * std::pow(2, (double)k / 12.0);
        const double semi = std::pow(2, 1.0 / 12);
        while (n == 0 || freq[n - 1] < fMax) {
            f = (k != Chrom) ? f * std::pow(semi, intervals[i % 7]) : f * semi;
            if (f > fMin && n < 127) freq[n++] = f;
            ++i;
        }
        --n;  // pop_back(); freq[n] keeps the popped value
    }
    key currentKey = Chrom;
    double fMin = 100, fMax = 800;
    double freq[128] = {0};
    size_t n = 0;
};

// RAII handle of one engine (one GPU).
class Engine {
public:
    explicit Engine(int device = 0) {
        const int rc = vp_engine_create(&h, device);
        if (rc != VP_OK) throw Error(rc, "vp_engine_create failed: no usable CUDA device (there is no CPU fallback)");
    }
    ~Engine() { if (h) vp_engine_destroy(h); }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;
    void check(int rc) const { if (rc != VP_OK) throw Error(rc, vp_last_error(h)); }
    vp_engine* h = nullptr;
};

class VocoderProcess;
class PitchProcess;

// Ring buffers / block adapter (Source/MyBuffer.h:25-55). Holds the engine of the batch and the recorded requests of
// the current block.
class MyBuffer {
public:
    explicit MyBuffer(int device = 0) : engine(device) { vp_default_params(&params); }

    // MyBuffer::prepare(samplesPerBlock, samplesToKeep, latency, sampleRate, nVoice, nSynth, nOut) + the stream count.
    // samplesToKeep / latency must be the values prepareToPlay derives (PluginProcessor.cpp:160-176).
    void prepare(int samplesPerBlockIn, int samplesToKeepIn, int latencyIn, double sampleRateIn, int numChannelsVoice,
                 int numChannelsSynth, int numChannelsOut, int nStreamsIn, int maxBlocksPerCall = 1) {
        if (numChannelsVoice != 1 || numChannelsSynth != 2 || numChannelsOut != 2)
            throw Error(VP_E_ARG, "the path is 1 voice + 2 side-chain channels in, 2 out (PluginProcessor.cpp:153-157)");
        vp_sizes z;
        if (vp_sizes_for(sampleRateIn, samplesPerBlockIn, params.keyPitch, &z) != VP_OK) throw Error(VP_E_ARG, "unsupported sample rate / block size");
        if (samplesToKeepIn != z.keep || latencyIn != z.latency)
            throw Error(VP_E_ARG, "samplesToKeep / latency differ from what prepareToPlay derives for this sample rate");
        B = samplesPerBlockIn; S = nStreamsIn; maxBlocks = maxBlocksPerCall; sampleRate = sampleRateIn; sizes = z;
        engine.check(vp_engine_set_params(engine.h, &params));
        engine.check(vp_engine_prepare(engine.h, sampleRate, B, S, maxBlocks, 0));
        beginBlock();
    }
    // the engine-wide parameters; the key, the gains and the vocoder orders go to every stream (and replace what
    // setStreamParams / setStreamOrders set)
    void setParams(const vp_params& p) {
        params = p;
        streamParams.clear();
        streamOrders.clear();
        engine.check(vp_engine_set_params(engine.h, &params));
    }
    // key and gains of streams first .. first + count - 1 (after prepare); kept until the next setParams
    void setStreamParams(int first, int count, const vp_stream_params* p) {
        engine.check(vp_engine_set_stream_params(engine.h, first, count, p));
        if (streamParams.empty()) {
            streamParams.resize((size_t)S);
            engine.check(vp_engine_get_stream_params(engine.h, 0, S, streamParams.data()));
        } else {
            for (int i = 0; i < count; ++i) streamParams[(size_t)(first + i)] = p[i];
        }
    }
    // vocoder orders (lpcVoice, lpcSynth) of streams first .. first + count - 1 (after prepare); kept until the next setParams
    void setStreamOrders(int first, int count, const vp_stream_orders* o) {
        engine.check(vp_engine_set_stream_orders(engine.h, first, count, o));
        if (streamOrders.empty()) {
            streamOrders.resize((size_t)S);
            engine.check(vp_engine_get_stream_orders(engine.h, 0, S, streamOrders.data()));
        } else {
            for (int i = 0; i < count; ++i) streamOrders[(size_t)(first + i)] = o[i];
        }
    }
    // largest lpcVoice / lpcSynth that may be set while the streams run (before prepare; VocoderProcess.cpp:50-57 sizes its
    // vectors for the ends of the parameter ranges: 100 / 30)
    void setWindow(bool hann) { engine.check(vp_engine_set_window(engine.h, hann ? VP_WINDOW_HANN : VP_WINDOW_SINE)); }
    void reserveOrders(int maxLpcVoice, int maxLpcSynth) { engine.check(vp_engine_reserve_orders(engine.h, maxLpcVoice, maxLpcSynth)); }
    // largest per-stream lpcPitch (before prepare; 0 = params.lpcPitch)
    void reservePitchOrder(int maxLpcPitch) { engine.check(vp_engine_reserve_pitch_order(engine.h, maxLpcPitch)); }
    // lpcPitch of streams first .. first + count - 1 (after prepare): read when a stream starts (PitchProcess.cpp:70) -- at
    // once for a stream that has processed nothing since prepare / restart / its restartStreams, else at its next start.
    // setParams does not touch it (nothing to push again per block)
    void setStreamPitchOrders(int first, int count, const int* lpcPitch) {
        engine.check(vp_engine_set_stream_pitch_orders(engine.h, first, count, lpcPitch));
    }
    // the order each stream runs its next block at / takes at its next start (either pointer may be null)
    void getStreamPitchOrders(int first, int count, int* inForce, int* next) const {
        engine.check(vp_engine_get_stream_pitch_orders(engine.h, first, count, inForce, next));
    }
    // prepareToPlay on a running instance: back to the freshly prepared state first
    void restart() { if (B > 0) engine.check(vp_engine_reset(engine.h)); }
    // prepareToPlay for some instances of the running batch (a slot handed to a new user): from the next block on, each
    // listed stream continues as one that has heard only silence since prepare; the others are not touched
    void restartStreams(const int* streams, int count) { engine.check(vp_engine_reset_streams(engine.h, streams, count)); }
    // per-stream state snapshots: the state streams[0 .. count) start their next block with, as an opaque self-checking blob
    // (waits for the GPU; changes nothing), and back into slots of this or a compatible instance set (same sample rate, block
    // size, reservations and window; same grid phase, or nothing processed since prepare / restart)
    std::vector<uint8_t> saveStreams(const int* streams, int count) {
        size_t bytes = 0;
        engine.check(vp_engine_snapshot_size(engine.h, count, &bytes));
        std::vector<uint8_t> blob(bytes);
        engine.check(vp_engine_save_streams(engine.h, streams, count, blob.data(), blob.size()));
        return blob;
    }
    // each loaded slot takes the saved key, gains and orders: the per-stream values pushed with every block are refreshed
    void loadStreams(const int* streams, int count, const std::vector<uint8_t>& blob) {
        engine.check(vp_engine_load_streams(engine.h, streams, count, blob.data(), blob.size()));
        streamParams.resize((size_t)S);
        engine.check(vp_engine_get_stream_params(engine.h, 0, S, streamParams.data()));
        streamOrders.resize((size_t)S);
        engine.check(vp_engine_get_stream_orders(engine.h, 0, S, streamOrders.data()));
    }
    // automation at block accuracy: each event gives one stream its key and gains from an absolute block on (blocks counted
    // since prepare / restart); the engine applies them where the reference reads each value, also inside one multi-block call.
    // Pending events survive setParams / setStreamParams (which change the value from the next block on); restart drops them,
    // restartStreams those of the listed streams
    void scheduleStreamParams(const vp_stream_event* events, int count) {
        engine.check(vp_engine_schedule_stream_params(engine.h, events, count));
    }
    // the same for the vocoder orders: each event gives one stream its lpcVoice / lpcSynth from an absolute block on
    void scheduleStreamOrders(const vp_stream_order_event* events, int count) {
        engine.check(vp_engine_schedule_stream_orders(engine.h, events, count));
    }
    const vp_params& getParams() const { return params; }

    // fillInputBuffers(voiceBuffer, synthBuffer): host rows [S][stride]; synth channel 1 may be null when gainSynth is off
    void fillInputBuffers(const float* voice, const float* synthL, const float* synthR, size_t strideSamples, int nBlocks = 1) {
        inVoice = voice; inSynthL = synthL; inSynthR = synthR; stride = strideSamples; blocks = nBlocks;
    }
    void addDryVoice(double gainDb) { dryVoiceDb = (float)gainDb; }   // PluginProcessor.cpp:226-227 (called when > -59 dB)
    void addSynth(double gainDb) { drySynthDb = (float)gainDb; }      // PluginProcessor.cpp:229-230
    // fillOutputBuffer(buffer, nOutputChannels): runs the recorded block(s) and writes out[S][stride] (R may be null)
    void fillOutputBuffer(float* outL, float* outR) {
        vp_params p = params;
        p.vocBool = vocRequested ? 1 : 0;
        p.pitchBool = pitchRequested ? 1 : 0;
        p.gainVoice = dryVoiceDb;
        p.gainSynth = drySynthDb;
        engine.check(vp_engine_set_params(engine.h, &p));
        // per-stream values set since the last setParams: pushed again after the broadcast above (unchanged values cost nothing)
        if (!streamParams.empty()) engine.check(vp_engine_set_stream_params(engine.h, 0, S, streamParams.data()));
        if (!streamOrders.empty()) engine.check(vp_engine_set_stream_orders(engine.h, 0, S, streamOrders.data()));
        engine.check(vp_engine_process_host(engine.h, blocks, inVoice, inSynthL, inSynthR, outL, outR, stride));
        beginBlock();
    }
    int getSamplesPerBlock() const { return B; }
    int getNumStreams() const { return S; }
    const vp_sizes& getSizes() const { return sizes; }
    Engine engine;

private:
    friend class VocoderProcess;
    friend class PitchProcess;
    void beginBlock() { vocRequested = pitchRequested = false; dryVoiceDb = drySynthDb = -60.0f; }
    vp_params params;
    std::vector<vp_stream_params> streamParams;  // [S] once setStreamParams was called, else empty
    std::vector<vp_stream_orders> streamOrders;  // [S] once setStreamOrders was called, else empty
    vp_sizes sizes{};
    int B = 0, S = 0, maxBlocks = 1, blocks = 1;
    double sampleRate = 0;
    const float *inVoice = nullptr, *inSynthL = nullptr, *inSynthR = nullptr;
    size_t stride = 0;
    bool vocRequested = false, pitchRequested = false;
    float dryVoiceDb = -60.0f, drySynthDb = -60.0f;
};

// Source/VocoderProcess.h:29-34
class VocoderProcess {
public:
    void prepare(int wlenIn, int hopIn, std::string windowType, double silenceThresholdDbIn) {
        if (windowType != "sine" && windowType != "hann") throw Error(VP_E_ARG, "unknown window type (VocoderProcess.cpp:131-134)");
        hann = windowType == "hann";
        if (wlenIn != 4 * hopIn) throw Error(VP_E_ARG, "overlap must be 0.75 (VocoderProcess.cpp:110-114)");
        if (silenceThresholdDbIn != -60.0) throw Error(VP_E_ARG, "the gate threshold is the plug-in's -60 dB (PluginProcessor.cpp:148)");
        wlen = wlenIn; hop = hopIn;
    }
    int getLatency(int /*samplesPerBlock*/) const { return wlen; }  // VocoderProcess.cpp:86
    bool isHann() const { return hann; }
    void process(MyBuffer& myBuffer) {
        if (myBuffer.sizes.wlenV != wlen || myBuffer.sizes.hopV != hop) throw Error(VP_E_ARG, "wlen / hop differ from prepareToPlay's derivation");
        myBuffer.vocRequested = true;
    }

private:
    int wlen = 0, hop = 0;
    bool hann = false;
};

// Source/PitchProcess.h:40-48
class PitchProcess {
public:
    void prepare(double fSIn, double fMinIn, double fMaxIn, int frameLenIn, int hopIn, int samplesPerBlockIn, double silenceThresholdDbIn) {
        if (fMinIn != 100.0 || fMaxIn != 800.0 || silenceThresholdDbIn != -60.0)
            throw Error(VP_E_ARG, "fMin / fMax / gate threshold are the plug-in's constants (PluginProcessor.cpp:148,172)");
        fS = fSIn; frameLen = frameLenIn; hop = hopIn; B = samplesPerBlockIn;
    }
    void prepare2(MyBuffer& myBuffer) {  // PitchProcess.cpp:134-141
        if (myBuffer.sizes.frameLenP != frameLen || myBuffer.sizes.hopP != hop || myBuffer.B != B)
            throw Error(VP_E_ARG, "frameLen / hop / block differ from prepareToPlay's derivation");
    }
    int getLatency(int /*samplesPerBlock*/) const { return frameLen; }  // PitchProcess.cpp:37
    void process(MyBuffer& myBuffer) { myBuffer.pitchRequested = true; }
    // silence(): pitchBool off for this block (PitchProcess.cpp:146-158). Nothing to record: a block whose
    // PitchProcess::process was not requested reaches the engine with pitchBool = 0, and the engine then does what silence()
    // does -- both mark vectors cleared, pitch / period zeroed, the frame in flight cut -- for every stream.
    void silence() {}

private:
    double fS = 0;
    int frameLen = 0, hop = 0, B = 0;
};

// The two driver functions of VocoderAudioProcessor (Source/PluginProcessor.cpp:144-184 and :203-234), for nStreams
// plug-in instances at once. `params` plays the role of the AudioProcessorValueTreeState.
class VocoderBatchProcessor {
public:
    explicit VocoderBatchProcessor(int device = 0) : myBuffer(device) { vp_default_params(&params); }

    // maxLpcVoice / maxLpcSynth: the largest orders the parameters may take while the streams run (0 = the current ones);
    // maxLpcPitch: the largest per-stream lpcPitch (myBuffer.setStreamPitchOrders; 0 = params.lpcPitch)
    void prepareToPlay(double sampleRate, int samplesPerBlock, int nStreams, int maxBlocksPerCall = 1, int maxLpcVoice = 0,
                       int maxLpcSynth = 0, int maxLpcPitch = 0) {
        const double ratioSR = sampleRate / 44100.0;                       // :160
        const int hopVoc = (int)std::floor(128.0 * ratioSR);               // :163
        const int wlenVoc = 4 * hopVoc;                                    // :164
        const int c256 = (int)std::floor(256.0 * ratioSR);                 // :168
        const int hopPitch = 3 * c256, frameLenPitch = 4 * c256;           // :169-170
        const double silenceDb = -60.0;                                    // :148
        myBuffer.restart();
        myBuffer.reserveOrders(maxLpcVoice, maxLpcSynth);
        myBuffer.reservePitchOrder(maxLpcPitch);
        myBuffer.setParams(params);
        pitchProcess.prepare(sampleRate, 100.0, 800.0, frameLenPitch, hopPitch, samplesPerBlock, silenceDb);   // :172
        vocoderProcess.prepare(wlenVoc, hopVoc, windowType, silenceDb);                                         // :173
        myBuffer.setWindow(vocoderProcess.isHann());
        latency = std::max(pitchProcess.getLatency(samplesPerBlock), vocoderProcess.getLatency(samplesPerBlock));  // :175
        myBuffer.prepare(samplesPerBlock, frameLenPitch, latency, sampleRate, 1, 2, 2, nStreams, maxBlocksPerCall);  // :176-179
        pitchProcess.prepare2(myBuffer);                                   // :181
    }
    int getLatencySamples() const { return latency; }                     // setLatencySamples(latency), :183

    // processBlock for all streams: voice [S][stride], side-chain L/R [S][stride] in, out L/R [S][stride].
    // nBlocks > 1 processes that many consecutive host blocks in one call (same result as nBlocks calls).
    void processBlock(const float* voice, const float* synthL, const float* synthR, float* outL, float* outR, size_t stride,
                      int nBlocks = 1) {
        myBuffer.setParams(params);
        // one parameter tree per instance: pushed after setParams, which broadcasts; each stream then has its own dry mix
        if (!streamParams.empty()) {
            if (streamParams.size() != (size_t)myBuffer.getNumStreams()) throw Error(VP_E_ARG, "streamParams must hold one entry per stream");
            myBuffer.setStreamParams(0, (int)streamParams.size(), streamParams.data());
        }
        if (!streamOrders.empty()) {
            if (streamOrders.size() != (size_t)myBuffer.getNumStreams()) throw Error(VP_E_ARG, "streamOrders must hold one entry per stream");
            myBuffer.setStreamOrders(0, (int)streamOrders.size(), streamOrders.data());
        }
        myBuffer.fillInputBuffers(voice, synthL, synthR, stride, nBlocks);   // :212
        if (params.vocBool) vocoderProcess.process(myBuffer);                // :214-215
        if (params.pitchBool) pitchProcess.process(myBuffer);                // :218-221
        else pitchProcess.silence();
        if (params.gainVoice > -59.0f) myBuffer.addDryVoice(params.gainVoice);  // :226-227
        if (params.gainSynth > -59.0f) myBuffer.addSynth(params.gainSynth);     // :229-230
        myBuffer.fillOutputBuffer(outL, outR);                               // :232
    }

    vp_params params;   // the ten plug-in parameters (PluginProcessor.cpp:37-73)
    // optional, one entry per stream: that instance's key and gains (its value tree); empty = params' values for every stream
    std::vector<vp_stream_params> streamParams;
    // optional, one entry per stream: that instance's lpcVoice / lpcSynth; empty = params' orders for every stream (orders
    // above params' need maxLpcVoice / maxLpcSynth at prepareToPlay)
    std::vector<vp_stream_orders> streamOrders;
    std::string windowType = "sine";  // the literal prepareToPlay passes to VocoderProcess::prepare (:173); "hann" = the class's other branch
    MyBuffer myBuffer;
    VocoderProcess vocoderProcess;
    PitchProcess pitchProcess;

private:
    int latency = 0;
};

}  // namespace vpb200
