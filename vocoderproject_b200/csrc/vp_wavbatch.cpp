// vp_wavbatch -- WAV front-end of the batch engine (SURVEY.md 8(f)#3): every line of a manifest is one plug-in
// instance = one stream,
//
//     voice.wav  sidechain.wav  out.wav  [key=N] [gainVoc=dB] [gainPitch=dB] [gainVoice=dB] [gainSynth=dB]
//                                        [lpcVoice=N] [lpcSynth=N] [lpcPitch=N]
//
// (voice: channel 0 is used, PluginProcessor.cpp:153-157 mono main bus; side-chain: stereo, a mono file feeds both
// channels). The optional tokens are that instance's own key, gains, vocoder orders and pitch-corrector order: they
// override the command-line values for the job, so files in different keys, with different mixes or timbres still run as
// one batch. All jobs run as ONE batch on the GPU through the facade's prepareToPlay / processBlock (vp_facade.hpp):
// same sample rate for all files, shorter jobs are zero-padded to the longest and trimmed again on output.
//
//   vp_wavbatch manifest.txt [--block 1024] [--blocks-per-call 64] [--key 12] [--voc 0|1] [--pitch 0|1]
//               [--gain-voice dB] [--gain-synth dB] [--gain-voc dB] [--gain-pitch dB] [--pcm16] [--keep-latency] [--device d]
//
// Output: stereo WAV (float32, or PCM16 with --pcm16), as long as the voice file. The plug-in delays its output by
// getLatencySamples() (1024 @ 44.1 kHz); like a latency-compensating host the tool drops that delay (it feeds `latency`
// extra zero samples at the end) unless --keep-latency asks for the raw processBlock output.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "vp_facade.hpp"
#include "vp_wav.hpp"

struct Job { std::string voice, synth, out; vpb200::WavData v, s; vp_stream_params sp; vp_stream_orders so; int lpcPitch; };

// "name=value" tokens of a manifest line -> the job's per-instance parameters; false when any token is not one of them.
// any / anyOrd / anyPitch: some token set a key or gain / a vocoder order / lpcPitch
static bool parse_stream_tokens(std::istringstream& ls, vp_stream_params& sp, vp_stream_orders& so, int& lpcPitch, bool& any,
                                bool& anyOrd, bool& anyPitch) {
    std::string tok;
    while (ls >> tok) {
        const size_t eq = tok.find('=');
        if (eq == std::string::npos || eq + 1 == tok.size()) return false;
        const std::string name = tok.substr(0, eq), val = tok.substr(eq + 1);
        char* end = nullptr;
        const double x = strtod(val.c_str(), &end);
        if (*end != '\0') return false;
        if (name == "key") {
            if (x != (double)(int)x) return false;
            sp.keyPitch = (int)x;
        } else if (name == "lpcVoice" || name == "lpcSynth") {
            if (x != (double)(int)x) return false;
            (name == "lpcVoice" ? so.lpcVoice : so.lpcSynth) = (int)x;
            anyOrd = true;
            continue;
        } else if (name == "lpcPitch") {
            if (x != (double)(int)x) return false;
            lpcPitch = (int)x;
            anyPitch = true;
            continue;
        } else if (name == "gainVoc") sp.gainVoc = (float)x;
        else if (name == "gainPitch") sp.gainPitch = (float)x;
        else if (name == "gainVoice") sp.gainVoice = (float)x;
        else if (name == "gainSynth") sp.gainSynth = (float)x;
        else return false;
        any = true;
    }
    return true;
}

int main(int argc, char** argv) {
    int B = 1024, K = 64, device = 0;
    bool pcm16 = false, keepLatency = false;
    vp_params prm;
    vp_default_params(&prm);
    std::string manifest;
    for (int i = 1; i < argc; ++i) {
        auto arg = [&](const char* name) { return !strcmp(argv[i], name) && i + 1 < argc; };
        if (arg("--block")) B = atoi(argv[++i]);
        else if (arg("--blocks-per-call")) K = atoi(argv[++i]);
        else if (arg("--key")) prm.keyPitch = atoi(argv[++i]);
        else if (arg("--voc")) prm.vocBool = atoi(argv[++i]);
        else if (arg("--pitch")) prm.pitchBool = atoi(argv[++i]);
        else if (arg("--gain-voice")) prm.gainVoice = (float)atof(argv[++i]);
        else if (arg("--gain-synth")) prm.gainSynth = (float)atof(argv[++i]);
        else if (arg("--gain-voc")) prm.gainVoc = (float)atof(argv[++i]);
        else if (arg("--gain-pitch")) prm.gainPitch = (float)atof(argv[++i]);
        else if (arg("--device")) device = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--pcm16")) pcm16 = true;
        else if (!strcmp(argv[i], "--keep-latency")) keepLatency = true;
        else if (!strcmp(argv[i], "--help")) {
            printf("usage: vp_wavbatch manifest.txt [--block B] [--blocks-per-call K] [--key 0..12] [--voc 0|1] [--pitch 0|1] "
                   "[--gain-voice dB] [--gain-synth dB] [--gain-voc dB] [--gain-pitch dB] [--pcm16] [--keep-latency] [--device d]\n"
                   "manifest lines: voice.wav sidechain.wav out.wav [key=N] [gainVoc=dB] [gainPitch=dB] [gainVoice=dB] [gainSynth=dB] "
                   "[lpcVoice=N] [lpcSynth=N] [lpcPitch=N]\n"
                   "  (the tokens set that job's key, gains, vocoder orders and pitch-corrector order; they override --key / --gain-* "
                   "for the job)\n");
            return 0;
        } else if (argv[i][0] != '-' && manifest.empty()) manifest = argv[i];
        else { fprintf(stderr, "unknown argument %s\n", argv[i]); return 2; }
    }
    if (manifest.empty() || B <= 0 || K <= 0) { fprintf(stderr, "vp_wavbatch: no manifest (see --help)\n"); return 2; }
    try {
        std::vector<Job> jobs;
        bool perJob = false, perJobOrd = false, perJobPitch = false;  // some line sets its own key or gains / orders / lpcPitch
        {
            std::ifstream mf(manifest);
            if (!mf) throw std::runtime_error("cannot open " + manifest);
            std::string line;
            while (std::getline(mf, line)) {
                std::istringstream ls(line);
                Job j;
                if (!(ls >> j.voice)) continue;
                if (j.voice[0] == '#') continue;
                if (!(ls >> j.synth >> j.out)) throw std::runtime_error("manifest line needs three paths: " + line);
                j.sp.gainPitch = prm.gainPitch; j.sp.gainVoice = prm.gainVoice; j.sp.gainSynth = prm.gainSynth;
                j.sp.gainVoc = prm.gainVoc; j.sp.keyPitch = prm.keyPitch;
                j.so.lpcVoice = prm.lpcVoice; j.so.lpcSynth = prm.lpcSynth; j.lpcPitch = prm.lpcPitch;
                if (!parse_stream_tokens(ls, j.sp, j.so, j.lpcPitch, perJob, perJobOrd, perJobPitch))
                    throw std::runtime_error("manifest tokens after the paths are key=N gainVoc= gainPitch= gainVoice= gainSynth= "
                                             "lpcVoice=N lpcSynth=N lpcPitch=N: " + line);
                jobs.push_back(std::move(j));
            }
        }
        if (jobs.empty()) throw std::runtime_error("empty manifest");
        int fs = 0;
        size_t longest = 0;
        for (Job& j : jobs) {
            j.v = vpb200::wav_read(j.voice);
            j.s = vpb200::wav_read(j.synth);
            if (fs == 0) fs = j.v.sampleRate;
            if (j.v.sampleRate != fs || j.s.sampleRate != fs)
                throw std::runtime_error("all files of a batch must share one sample rate (" + j.voice + " / " + j.synth + ")");
            longest = std::max(longest, j.v.frames);
        }
        const int S = (int)jobs.size();
        vpb200::VocoderBatchProcessor proc(device);
        proc.params = prm;
        int maxV = 0, maxS = 0, maxP = 0;  // the workspace rows are sized for the largest orders of the manifest
        for (const Job& j : jobs) {
            maxV = std::max(maxV, j.so.lpcVoice); maxS = std::max(maxS, j.so.lpcSynth); maxP = std::max(maxP, j.lpcPitch);
        }
        proc.prepareToPlay((double)fs, B, S, K, maxV, maxS, maxP);
        if (perJobPitch) {  // read when a stream starts: set before the first block, each job starts with its own
            std::vector<int> lp;
            for (const Job& j : jobs) lp.push_back(j.lpcPitch);
            proc.myBuffer.setStreamPitchOrders(0, S, lp.data());
        }
        if (perJob)
            for (const Job& j : jobs) proc.streamParams.push_back(j.sp);
        if (perJobOrd)
            for (const Job& j : jobs) proc.streamOrders.push_back(j.so);
        const size_t lat = keepLatency ? 0 : (size_t)proc.getLatencySamples();
        const size_t m = (size_t)K * B;
        const size_t nCalls = (longest + lat + m - 1) / m;
        const size_t n = nCalls * m;
        std::vector<std::vector<float>> outL((size_t)S, std::vector<float>(n)), outR((size_t)S, std::vector<float>(n));
        std::vector<float> bv(S * m), bl(S * m), br(S * m), ol(S * m), orr(S * m);
        const auto t0 = std::chrono::steady_clock::now();
        for (size_t c = 0; c < nCalls; ++c) {
            const size_t t = c * m;
            for (int s = 0; s < S; ++s) {
                const Job& j = jobs[(size_t)s];
                const std::vector<float>& v = j.v.ch[0];
                const std::vector<float>& l = j.s.ch[0];
                const std::vector<float>& r = j.s.ch[j.s.channels > 1 ? 1 : 0];
                for (size_t i = 0; i < m; ++i) {
                    const size_t u = t + i;
                    bv[s * m + i] = u < v.size() ? v[u] : 0.0f;
                    bl[s * m + i] = u < l.size() ? l[u] : 0.0f;
                    br[s * m + i] = u < r.size() ? r[u] : 0.0f;
                }
            }
            proc.processBlock(bv.data(), bl.data(), br.data(), ol.data(), orr.data(), m, K);
            for (int s = 0; s < S; ++s) {
                memcpy(&outL[(size_t)s][t], &ol[s * m], m * sizeof(float));
                memcpy(&outR[(size_t)s][t], &orr[s * m], m * sizeof(float));
            }
        }
        const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        double audio = 0;
        for (int s = 0; s < S; ++s) {
            const Job& j = jobs[(size_t)s];
            vpb200::wav_write(j.out, fs, {outL[(size_t)s].data() + lat, outR[(size_t)s].data() + lat}, j.v.frames, pcm16);
            audio += (double)j.v.frames / fs;
        }
        printf("{\"host\": \"vp_wavbatch\", \"streams\": %d, \"sample_rate\": %d, \"block\": %d, \"blocks_per_call\": %d, \"calls\": %zu, "
               "\"latency_samples\": %d, \"latency_compensated\": %s, \"audio_s\": %.3f, \"wall_s\": %.4f}\n",
               S, fs, B, K, nCalls, proc.getLatencySamples(), keepLatency ? "false" : "true", audio, wall);
    } catch (const vpb200::Error& e) {
        fprintf(stderr, "vp_wavbatch: %s (there is no CPU fallback)\n", e.what());
        return 1;
    } catch (const std::exception& e) {
        fprintf(stderr, "vp_wavbatch: %s\n", e.what());
        return 2;
    }
    return 0;
}
