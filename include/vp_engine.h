/* vp_engine.h -- C ABI of the B200 batch engine for VocoderProject's DSP core.
 *
 * Drop-in boundary for the path VocoderAudioProcessor::processBlock drives
 * (reference: Source/PluginProcessor.cpp:203-234) -- MyBuffer ring buffering,
 * LPC, VocoderProcess, PitchProcess, Notes -- batched over independent
 * streams. Plain pointers and sizes only; no C++/CUDA/torch types. The C++
 * facade with the reference's class names lives in
 * vocoderproject_b200/csrc/vp_facade.hpp and is implemented on top of this
 * ABI; INTEGRATION.md shows the PluginProcessor-side binding.
 *
 * Semantics. One "stream" is one plug-in instance (1 mono voice + stereo
 * side-chain in, stereo out). Each stream has its own key and gains
 * (vp_stream_params, vp_engine_set_stream_params), its own vocoder LPC
 * orders (vp_stream_orders, vp_engine_set_stream_orders) and its own
 * pitch-corrector LPC order (vp_engine_set_stream_pitch_orders); the remaining
 * parameters (vocBool / pitchBool, window, mode) are one set per engine.
 * vp_engine_prepare is prepareToPlay(sampleRate,
 * samplesPerBlock) for every stream; each vp_engine_process* call is, per
 * stream, nBlocks further consecutive processBlock calls. Results do
 * depend (sparsely) on samplesPerBlock exactly as in the reference (whole-ring
 * RMS gate, MyBuffer.cpp:258-261; PSOLA look-ahead test, PitchProcess.cpp:
 * 799-803), hence the "virtual block size" argument of vp_engine_prepare.
 *
 * All functions return VP_OK (0) or a negative VP_E_* code; none throws, none
 * aborts. There is no CPU fallback: without a usable CUDA device every
 * compute entry point returns VP_E_CUDA.
 */
#ifndef VP_ENGINE_H
#define VP_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VP_OK 0
#define VP_E_ARG (-1)     /* bad argument */
#define VP_E_STATE (-2)   /* call order (e.g. process before prepare) */
#define VP_E_CUDA (-3)    /* CUDA runtime error / no device; see vp_last_error */
#define VP_E_NOMEM (-4)   /* device or host allocation failed */
#define VP_E_RANGE (-5)   /* parameter outside the plug-in's range */

/* The ten plug-in parameters (Source/PluginProcessor.cpp:37-73), pushed by
 * the caller instead of pulled through audioProcPtr->treeState. Gains in dB
 * as float, exactly what the plug-in's std::atomic<float> holds. */
typedef struct vp_params {
    float gainPitch; /* [-60, 6]  default 0    PitchProcess.cpp:336 */
    float gainVoice; /* [-60, 6]  default -60  PluginProcessor.cpp:226 (dry voice, off <= -59) */
    float gainSynth; /* [-60, 6]  default -60  PluginProcessor.cpp:229 (dry synth, off <= -59) */
    float gainVoc;   /* [-60, 6]  default 0    VocoderProcess.cpp:291 */
    int lpcVoice;    /* [2, 100]  default 40   VocoderProcess.cpp:139 */
    int lpcPitch;    /* [2, 100]  default 15   PitchProcess.cpp:70 (read in prepare only) */
    int lpcSynth;    /* [2, 30]   default 5    VocoderProcess.cpp:155 */
    int keyPitch;    /* Notes::key 0..12 (A..G#, 12 = chromatic), default 12; Notes.h:26 */
    int pitchBool;   /* default 1 */
    int vocBool;     /* default 1 */
} vp_params;

/* The per-instance part of vp_params: what one stream's plug-in instance holds in its parameter tree and the engine reads
 * per stream. These five, the two vocoder orders (vp_stream_orders) and lpcPitch (vp_engine_set_stream_pitch_orders, taken
 * when a stream starts) are per stream. The others stay per engine: vocBool and pitchBool move the frame grids, which are
 * host state every stream shares (a bypassed block freezes them); the window and the mode are prepare-time choices. 20 bytes. */
typedef struct vp_stream_params {
    float gainPitch, gainVoice, gainSynth, gainVoc; /* dB, [-60, 6]; the dry paths are on above -59 dB */
    int keyPitch;                                   /* 0..12 */
} vp_stream_params;

/* The vocoder's two LPC orders of one stream (VocoderProcess.cpp:193-194, read at every vocoder frame start): they set the
 * stream's timbre and move no frame grid. 8 bytes. */
typedef struct vp_stream_orders {
    int lpcVoice;  /* [2, 100] */
    int lpcSynth;  /* [2, 30] */
} vp_stream_orders;

/* Sizes prepareToPlay derives from the sample rate
 * (PluginProcessor.cpp:160-176, PitchProcess.cpp:100-107, MyBuffer.cpp:46-48). */
typedef struct vp_sizes {
    int hopV, wlenV;           /* vocoder hop / frame length */
    int hopP, frameLenP, chunk;/* pitch hop / frame length / chunk */
    int tauMin, tauMax;        /* YIN lag search range [tauMin, tauMax) */
    int latency, keep;         /* plug-in latency, samplesToKeep */
    int inSize, outSize;       /* MyBuffer ring lengths for this block size */
    int anCap;                 /* capacity of the pitch-mark vectors */
    int nFreq;                 /* entries in the note table for the engine's keyPitch (vp_params) */
} vp_sizes;

/* Per pitch frame decisions (one record per processChunkStart call,
 * PitchProcess.cpp:203-247). */
#define VP_MAX_MARKS 24
#define VP_NO_MARK (-2147483647 - 1)
#define VP_PF_GATED 1u       /* silence gate fired (PitchProcess.cpp:208-214) */
#define VP_PF_VOICED 2u      /* pitch > 1 */
#define VP_PF_HAS_MARKS 4u   /* anMarks non-empty -> frame is synthesised */
#define VP_PF_NEAR_GATE 16u      /* gate level within eps of -60 dB */
#define VP_PF_NEAR_YIN 32u       /* a deciding YIN comparison within eps (after the FP64 re-check) */
#define VP_PF_UB 64u             /* the reference has undefined behaviour here (SURVEY App. B U2-U5) */
#define VP_PF_YIN_RECHECKED 128u /* FP32 YIN was inconclusive; decided by the FP64 pass */
typedef struct vp_pitch_frame {
    uint32_t flags;
    int32_t period;           /* detected period in samples (0 = unvoiced) */
    int32_t periodPsola;      /* period else prevVoicedPeriod (PitchProcess.cpp:669-672) */
    int32_t periodNew;        /* synthesis mark spacing */
    int32_t note;             /* snapped note index in the table of the stream's key, -1 if none */
    int32_t nAn, nSt;
    int32_t anStale;          /* storage slot anMarks[nAn] (PitchProcess.cpp:818) */
    int32_t nAnOv;
    int32_t prevAnLast;       /* last mark of the previous frame that does not overlap this one, in this frame's
                                 coordinates (what PitchProcess.cpp:812 means to fall back to); VP_NO_MARK if none */
    int32_t anMarks[VP_MAX_MARKS];
    int32_t stMarks[VP_MAX_MARKS];
    double beta;              /* closestFreq / pitch, carried over unvoiced frames */
} vp_pitch_frame;

typedef struct vp_engine vp_engine;

/* ---- lifecycle ----------------------------------------------------------- */
void vp_default_params(vp_params* p);
/* Host-only helper: the sizes prepareToPlay would derive. */
int vp_sizes_for(double sampleRate, int samplesPerBlock, int keyPitch, vp_sizes* out);
/* Number of visible CUDA devices (0 when there is none). */
int vp_device_count(void);

int vp_engine_create(vp_engine** e, int device);
void vp_engine_destroy(vp_engine* e);
const char* vp_last_error(const vp_engine* e);

/* Largest lpcVoice / lpcSynth that vp_engine_set_params may be given on a RUNNING stream (the reference re-reads both orders
 * at every vocoder frame, VocoderProcess.cpp:193-194, and sizes its vectors for the ends of the parameter ranges, :50-57).
 * Call before vp_engine_prepare: the coefficient rows of the workspace are sized for it. Without it the maximum is what the
 * parameters say at vp_engine_prepare. 0 = no reservation. */
int vp_engine_reserve_orders(vp_engine* e, int maxLpcVoice, int maxLpcSynth);

/* prepareToPlay(sampleRate, samplesPerBlock) for nStreams independent
 * plug-in instances. maxBlocks bounds nBlocks of later process calls.
 * workspaceBytes: device memory the engine may use for intermediates
 * (0 = default); it decides how many streams are in flight per pass. */
int vp_engine_prepare(vp_engine* e, double sampleRate, int samplesPerBlock, int nStreams, int maxBlocks,
                      size_t workspaceBytes);
/* Replaces the reference's parameter pulls (treeState.getRawParameterValue(id)->load(); VocoderProcess.cpp:193-194,291,
 * PitchProcess.cpp:70,206,336, PluginProcessor.cpp:212-230). Before prepare: anything in the plug-in's ranges. Between
 * process calls of a running stream (automation) every parameter takes effect where the reference reads it: gainVoc per
 * vocoder frame, gainPitch per emitted chunk, gainVoice / gainSynth per block, keyPitch per pitch frame, lpcVoice / lpcSynth
 * per vocoder frame (frames in flight keep the order they started with; VP_E_STATE beyond vp_engine_reserve_orders / the
 * orders at prepare), vocBool / pitchBool per block: a block with vocBool off skips VocoderProcess::process (its frame grid
 * freezes relative to the block, frames in flight still come out), a block with pitchBool off is PitchProcess::silence()
 * (PluginProcessor.cpp:214-221, PitchProcess.cpp:146-158). lpcPitch is read in PitchProcess::prepare only (:70): it is the
 * value every stream starts with at vp_engine_prepare, a change on a running stream is ignored until the next
 * vp_engine_prepare, as in the reference, and it never overwrites the per-stream values of
 * vp_engine_set_stream_pitch_orders.
 * The five per-instance fields (gainPitch, gainVoice, gainSynth, gainVoc, keyPitch) and the orders lpcVoice / lpcSynth are
 * written to EVERY stream, replacing what vp_engine_set_stream_params / vp_engine_set_stream_orders set: a caller that never
 * sets streams one by one has one parameter set for the batch. */
int vp_engine_set_params(vp_engine* e, const vp_params* p);
/* Per-stream key and gains: streams firstStream .. firstStream + count - 1 take p[0 .. count). Valid after vp_engine_prepare,
 * which sets every stream from the engine's vp_params (VP_E_STATE before). A range outside [0, nStreams) is VP_E_ARG; a
 * value outside the plug-in's range is VP_E_RANGE, and then no stream changes. A new value takes effect at the next process
 * call of those streams, where the reference reads it (vp_engine_set_params): gainVoc per vocoder frame, gainPitch per
 * emitted chunk, gainVoice / gainSynth per block, keyPitch per pitch frame. vp_engine_reset keeps the values (a plug-in's
 * parameter tree survives prepareToPlay). Setting the values a stream already has costs nothing. The table goes to the
 * device with the next process call: a call already issued (vp_engine_process_device is asynchronous) keeps the values it
 * was issued with. For changes at arbitrary blocks inside one call see vp_engine_schedule_stream_params. */
int vp_engine_set_stream_params(vp_engine* e, int firstStream, int count, const vp_stream_params* p);
/* The values in force at the last block issued (after a call with scheduled changes: at its last block). */
int vp_engine_get_stream_params(const vp_engine* e, int firstStream, int count, vp_stream_params* out);

/* Block-accurate per-stream automation: stream `stream` takes p from absolute block `block` on (blocks counted since
 * vp_engine_prepare / vp_engine_reset, the count of vp_call_plan.firstBlock), until its next change. 40 bytes. */
typedef struct vp_stream_event {
    int stream;
    int reserved;     /* 0 */
    long long block;
    vp_stream_params p;
    int pad;          /* 0 */
} vp_stream_event;
/* Queues changes for any block not yet issued; a process call of any kind (including vp_engine_stream_block) applies them
 * at their blocks, where the reference reads each value: a value scheduled for block b applies to every read site whose
 * delayed-timeline position lies in block b or later -- the start of a vocoder frame (gainVoc), the start of a pitch frame
 * (keyPitch), the start of a pitch chunk (gainPitch: the whole chunk, also the part past the block's end), the output
 * sample (gainVoice, gainSynth). The output does not depend on how the blocks are cut into calls: one call, any cut into
 * several calls, or vp_engine_stream_block block by block give bit-identical output and frame records.
 * Valid after vp_engine_prepare (VP_E_STATE before). count < 0, events == NULL with count > 0, a stream outside
 * [0, nStreams) or a block already issued is VP_E_ARG; a value outside the plug-in's range is VP_E_RANGE; on any error
 * nothing is queued. The same (stream, block) twice: the later one (list order, then call order) wins. An event at the next
 * block to be issued is exactly vp_engine_set_stream_params before that call. Does not wait for the GPU; a call already
 * issued keeps its values. vp_engine_set_stream_params / vp_engine_set_params change the value from the next block on and
 * leave pending events in place (they apply at their blocks); vp_engine_reset and vp_engine_prepare drop every pending
 * event, vp_engine_reset_streams those of the listed streams. A call with no event inside its blocks costs nothing extra; a
 * call with events after its first block builds a per-block parameter table (one kernel launch; 32 bytes x nStreams x
 * nBlocks of device memory, allocated at the first such call outside the workspace budget: VP_E_NOMEM before anything is
 * issued when it cannot be had). */
int vp_engine_schedule_stream_params(vp_engine* e, const vp_stream_event* events, int count);

/* Per-stream vocoder orders: streams firstStream .. firstStream + count - 1 take o[0 .. count). Valid after vp_engine_prepare,
 * which sets every stream from the engine's vp_params (VP_E_STATE before). A range outside [0, nStreams) or o == NULL is
 * VP_E_ARG; an order outside the plug-in's ranges ([2, 100] / [2, 30]) is VP_E_RANGE; an order above what the workspace was
 * sized for (the orders at vp_engine_prepare or vp_engine_reserve_orders, at least 40 / 5) is VP_E_STATE. On any error no
 * stream changes. A new value takes effect from the next block on, at the start of each vocoder frame (VocoderProcess.cpp:
 * 193-194): frames in flight keep the order they started with. Setting the values a stream already has costs nothing;
 * vp_engine_reset and vp_engine_reset_streams keep them. A call in which every stream has the same orders in every block runs
 * exactly the kernels an engine with those orders in its vp_params runs; otherwise the Levinson kernels solve each frame at
 * its own orders, and every stream's coefficient rows are as wide as the widest (zero padded: a call whose orders are all
 * <= 40 / <= 5 keeps the tuned autocorrelation and synthesis kernels). */
int vp_engine_set_stream_orders(vp_engine* e, int firstStream, int count, const vp_stream_orders* o);
/* The values in force at the last block issued (after a call with scheduled changes: at its last block). */
int vp_engine_get_stream_orders(const vp_engine* e, int firstStream, int count, vp_stream_orders* out);

/* Block-accurate order automation: stream `stream` takes o from absolute block `block` on. 24 bytes. */
typedef struct vp_stream_order_event {
    int stream;
    int reserved;     /* 0 */
    long long block;
    vp_stream_orders o;
} vp_stream_order_event;
/* The rules of vp_engine_schedule_stream_params, for the orders: a value scheduled at block b applies to every vocoder frame
 * whose delayed-timeline start lies in block b or later; one call, any cut into calls, and vp_engine_stream_block give
 * bit-identical output and frame records. VP_E_STATE before vp_engine_prepare; VP_E_ARG for count < 0, a NULL list, a stream
 * outside [0, nStreams) or a block already issued; VP_E_RANGE / VP_E_STATE for values as vp_engine_set_stream_orders; on any
 * error nothing is queued. The same (stream, block) twice: the later one wins. vp_engine_set_stream_orders /
 * vp_engine_set_params change the value from the next block on and leave pending events in place; vp_engine_reset and
 * vp_engine_prepare drop every pending event, vp_engine_reset_streams those of the listed streams. Order and parameter events
 * share the per-block table of a call (see vp_engine_schedule_stream_params for its cost). */
int vp_engine_schedule_stream_orders(vp_engine* e, const vp_stream_order_event* events, int count);

/* Largest per-stream lpcPitch (vp_engine_set_stream_pitch_orders). Call before vp_engine_prepare: the pitch coefficient rows
 * of the workspace are sized for max(vp_params.lpcPitch, maxLpcPitch). Without it the widest allowed order is
 * vp_params.lpcPitch at vp_engine_prepare. 0 = no reservation; outside [0, 100] is VP_E_RANGE; a reservation above the
 * prepared size on a running engine is VP_E_STATE. */
int vp_engine_reserve_pitch_order(vp_engine* e, int maxLpcPitch);
/* Per-stream pitch-corrector LPC order. The reference reads lpcPitch in PitchProcess::prepare only (PitchProcess.cpp:70), so
 * a stream's order is fixed between two starts of that stream. A stream starts
 *   - at vp_engine_prepare, with vp_params.lpcPitch (values set earlier are dropped);
 *   - at vp_engine_reset, with its own set value (set values survive a reset, as the key and gains do);
 *   - at the process call where its vp_engine_reset_streams takes effect, with its set value.
 * Streams firstStream .. firstStream + count - 1 take lpcPitch[0 .. count) as the value they start with. For a stream that
 * has processed no block since its last start (no block since vp_engine_prepare / vp_engine_reset, or a reset of it
 * pending) the value is in force from the next process call; any other stream keeps its order until its next start.
 * Setting the value a stream already has costs nothing. vp_engine_set_params never changes these values. VP_E_STATE before
 * vp_engine_prepare; VP_E_ARG for a range outside [0, nStreams) or lpcPitch == NULL with count > 0; VP_E_RANGE outside
 * [2, 100]; VP_E_STATE above the reservation (vp_engine_reserve_pitch_order); on any error no stream changes.
 * A call in which every stream has the same order runs exactly the kernels an engine with that order in its vp_params runs;
 * otherwise the pitch rows are as wide as the widest order (zero padded, at least 15 when the rows hold 15) and the
 * Levinson and all-pole kernels take each frame's own order -- bit-identical, stream by stream, to an engine whose
 * vp_params.lpcPitch is that stream's. */
int vp_engine_set_stream_pitch_orders(vp_engine* e, int firstStream, int count, const int* lpcPitch);
/* inForce[i]: the order stream firstStream + i runs its next block at; next[i]: the order it takes at its next start. Either
 * pointer may be NULL. VP_E_STATE before vp_engine_prepare, VP_E_ARG for a range outside [0, nStreams). */
int vp_engine_get_stream_pitch_orders(const vp_engine* e, int firstStream, int count, int* inForce, int* next);

/* Behaviour at the places where the reference's C++ has undefined behaviour (SURVEY.md App. B U1-U6):
 *   VP_MODE_PARITY  (default) what the reference build actually does: the stale vector slot of PitchProcess.cpp:818 and the
 *                   popped table slot of Notes.cpp:99 are modelled, the other sites keep going and the frame is flagged VP_PF_UB;
 *   VP_MODE_DEFINED every such site takes the bounds-correct reading of what the code says it wants:
 *                   :818  the completeness test looks at the mark it is about to return (the last one), not one past the end;
 *                   :812  "last non-overlapping mark of the previous frame" = prevAnMarks[size - nOv - 1] (vp_pitch_frame.prevAnLast),
 *                         the frame's first mark when there is none;
 *                   :435  the descent ends at the last lag;   :487  "previous frame voiced" without previous marks searches the
 *                         frame like a first voiced frame;    :856  the interval search restarts at begin();
 *                   Notes.cpp:99  above the note table the closest note is the last one.
 *                   No frame is flagged VP_PF_UB for these sites. Identical to VP_MODE_PARITY wherever none of them is reached
 *                   with a different outcome. The CPU oracle has the same switch (oracle/vp_oracle.h).
 * May be called between process calls; takes effect with the next call. */
/* Window type of VocoderProcess::prepare (VocoderProcess.cpp:35-71, setWindows :95-135): VP_WINDOW_SINE is what
 * prepareToPlay passes (PluginProcessor.cpp:165); VP_WINDOW_HANN is the class's other branch (:116-124: no analysis window,
 * Hann synthesis window). Before vp_engine_prepare (or after vp_engine_reset, followed by vp_engine_prepare). */
#define VP_WINDOW_SINE 0
#define VP_WINDOW_HANN 1
int vp_engine_set_window(vp_engine* e, int window);

#define VP_MODE_PARITY 0
#define VP_MODE_DEFINED 1
int vp_engine_set_mode(vp_engine* e, int mode);
int vp_engine_get_sizes(const vp_engine* e, vp_sizes* out);
/* Layout the engine chose in vp_engine_prepare: streams processed per pass (nStreams / streamsPerPass passes per call),
 * carried input history per stream (samples) and the device workspace in use. Any pointer may be NULL. */
int vp_engine_get_info(const vp_engine* e, int* streamsPerPass, int* historySamples, size_t* workspaceBytes);

/* Back to the state right after vp_engine_prepare (= prepareToPlay): rings cleared, histories and pitch marks
 * forgotten, block counter 0. Consecutive vp_engine_process_* calls otherwise CONTINUE the streams: calling with
 * nBlocks = a then nBlocks = b gives the output of one call with nBlocks = a + b (the carried per-stream state is what
 * MyBuffer / VocoderProcess / PitchProcess keep between processBlock calls). */
int vp_engine_reset(vp_engine* e);

/* Per-stream counterpart of vp_engine_reset, for a host that hands a slot of a running batch to a new plug-in instance
 * (user, track): streams[0 .. count) continue as streams that have received ZEROS on every input channel since
 * vp_engine_prepare / vp_engine_reset -- their rings, histories, pitch marks and the frames of theirs still in flight are
 * forgotten. The frame grids are shared by all streams (vocBool / pitchBool are per engine), so a reset stream
 * keeps the batch's grid phase: it is exactly a freshly prepared instance only where the grids are in their prepare phase
 * (no vocBool / pitchBool-off block since prepare, and blocksDone * samplesPerBlock a multiple of both frame hops -- every
 * 3rd block at 44.1 kHz / 1024). Elsewhere it is what the reference's processBlock gives for zeros up to that block.
 * Valid after vp_engine_prepare (VP_E_STATE before). count == 0 does nothing; count < 0, streams == NULL with count > 0, or
 * any index outside [0, nStreams) is VP_E_ARG, and then nothing is queued. Duplicates, and repeated requests before one
 * process call, act as one. The reset takes effect at the next process call of any kind (process_device, process_host,
 * process_host_pcm16, stream_block), before its first kernel; a call already issued keeps the state it was issued with.
 * Does not wait for the GPU. Keeps each stream's vp_stream_params (the values in force now) but drops the listed streams'
 * pending vp_engine_schedule_stream_params events: a slot handed to a new user does not inherit the old user's automation
 * (the other streams keep theirs). Keeps the engine-wide parameters, the grids, every other
 * stream (bit for bit) and the records of the most recent call (get_pitch_frames / get_voc_frames); does not clear the
 * failed mark of a half-done call (only vp_engine_reset / vp_engine_prepare do, and both drop pending stream resets). The
 * listed streams keep their vp_stream_orders and drop their pending vp_engine_schedule_stream_orders events as well. They
 * start with the lpcPitch set for them (vp_engine_set_stream_pitch_orders), which is in force from this request on.
 * Streaming needs no new graph capture for it, unless the new lpcPitch changes whether the batch's pitch orders differ or
 * their widest (one capture). Cost: one kernel launch in the next call, none when no reset is pending. */
int vp_engine_reset_streams(vp_engine* e, const int* streams, int count);

/* ---- per-stream state snapshots: move a running stream to another slot or engine, checkpoint a render ----------------
 * A snapshot holds what a stream carries from one process call to the next (input histories, gate sums, carried and
 * orphan vocoder rows, energy histories, the last two pitch records, the mark state, the carried chunk gains), its
 * vp_stream_params and vp_stream_orders in force and its lpcPitch in force and next. Scheduled events are not state and are
 * not saved.
 *
 * Format (opaque to callers, versioned, self-checking): one header of VP_SNAPSHOT_HEADER_BYTES, then `count` records of
 * VP_SNAPSHOT_RECORD_BYTES + 16 x unitsPerStream bytes each. The header holds a magic ("VPSS"), the format version
 * (VP_SNAPSHOT_VERSION), a checksum, the layout key -- sample rate, samplesPerBlock, history length H, gate-carry rows,
 * the reserved row widths (capV / capS / capP), the window and the 16-byte units of each carried segment -- the record
 * count and the source's frame grids. A record is a fixed part (checksum, the stream's params, orders, lpcPitch in force /
 * next, the own order of each carried and orphan vocoder row = its last non-zero coefficient) followed by the raw state.
 * Checksums are FNV-1a 64 over little-endian 64-bit words with the checksum field zero (header: over the header; record:
 * over the fixed part, then the raw state).
 *
 * Compatibility. A record loads only into an engine with the same layout key (VP_E_STATE otherwise) and the same GRID
 * PHASE: the frame grids with every position taken relative to blocksDone x samplesPerBlock (next vocoder frame, live
 * orphan frames, next pitch chunk and its nChunk, carried pitch frames and their processed chunks, carried vocoder
 * frames on the grid). Engines that ran the same block sequence with the same vocBool / pitchBool switches have the same
 * phase -- the shards of one streaming host, also when their blocksDone differ by a whole grid period -- and any move
 * within one engine does. VP_E_STATE on a phase mismatch. Exception: an engine that has processed no block since
 * vp_engine_prepare / vp_engine_reset ADOPTS the snapshot's grids, block count included (checkpoint / resume, and
 * resizing a batch: save the live streams, prepare an engine with another nStreams or workspace, load); its slots that are
 * not loaded then hold the state of silence since prepare (what vp_engine_reset_streams gives). The mode
 * (vp_engine_set_mode) is not part of the key.
 *
 * Cost: one gather / scatter kernel over (listed stream x 16-byte unit) plus the copy over the host link (about 43 KB
 * per stream at 48 kHz); pinned and device staging buffers are allocated at the first save / load that needs them,
 * outside the workspace budget (VP_E_NOMEM before anything is issued when they cannot be had). */
#define VP_SNAPSHOT_VERSION 1
#define VP_SNAPSHOT_HEADER_BYTES 352
#define VP_SNAPSHOT_RECORD_BYTES 144  /* fixed part of a record; the raw state follows */
/* *bytes = the size of a snapshot of `count` streams for the engine as prepared. VP_E_ARG for e or bytes NULL or
 * count < 0, VP_E_STATE before vp_engine_prepare. */
int vp_engine_snapshot_size(const vp_engine* e, int count, size_t* bytes);
/* The state streams[0 .. count) start their next process call with -> buf (any host memory, at least
 * vp_engine_snapshot_size bytes). Waits for every call already issued (the mark chain on the side stream included), then
 * gathers and copies. A stream with a reset pending (vp_engine_reset_streams) is saved as the silent state that reset
 * gives. Changes nothing in the engine. VP_E_STATE before vp_engine_prepare or after a process call that failed half way;
 * VP_E_ARG for count < 0, a NULL list or buffer, an index outside [0, nStreams) or a buffer that is too small. */
int vp_engine_save_streams(vp_engine* e, const int* streams, int count, void* buf, size_t bytes);
/* Record i of buf becomes the state of slot streams[i]; count must be the snapshot's record count. Everything is
 * validated on the host before anything is issued: magic, version and checksums (VP_E_ARG), the layout key and grid phase
 * (VP_E_STATE), the records' params / orders / lpcPitch (VP_E_RANGE outside the plug-in's ranges, VP_E_STATE above the
 * reservation), and every integer of the raw state a kernel uses as a bound or an index -- mark counts, periods
 * (VP_E_RANGE); a buffer shorter than the snapshot, a NULL list, an index outside [0, nStreams) or a slot listed twice is
 * VP_E_ARG. On any error nothing changes. The load is then issued on the engine's stream behind every call already
 * issued (one upload through a pinned staging buffer, one scatter kernel) and returns once buf has been read, without
 * waiting for the GPU otherwise. Each loaded slot takes the record's params, orders and lpcPitch (in force and next: a load
 * is a start of that slot), and drops its pending reset and its pending scheduled events; a reset or an event requested
 * after the load applies on top of it. The engine's row widths grow to cover the loaded rows' own orders, so a stream
 * with low orders keeps a uniform batch on its tuned kernels. Streaming needs no new graph capture for a load unless it
 * changes what selects the captured kernels (whether orders differ and the widest, row widths, some stream's dry path). */
int vp_engine_load_streams(vp_engine* e, const int* streams, int count, const void* buf, size_t bytes);

/* Host-only helper (no CUDA): the frame grids a sequence of process calls produces -- call c processes nBlocks[c] blocks
 * with params[c] in force (only vocBool, pitchBool, lpcVoice, lpcSynth matter). For hosts that want to know how many frame
 * records a call will report, and for the CPU tests of the grid bookkeeping. The orders are the engine-wide ones: the plan
 * describes a batch whose streams all have params[c]'s lpcVoice / lpcSynth (rowOrderV / rowOrderS of a call with per-stream
 * orders are the widest of its streams, at least 40 / 5). */
typedef struct vp_call_plan {
    long long firstBlock;        /* blocks processed before this call */
    int offV, nFramesV;          /* first new vocoder frame (samples after the call's start) and how many start in the call */
    int carriedV;                /* vocoder frames of earlier calls that lie on this call's grid */
    int rowOrderV, rowOrderS;    /* width - 1 of the call's coefficient rows (>= lpcVoice / lpcSynth in force) */
    int offP, nFramesP;          /* same for the pitch frames */
    int vocMix, pitchMix;        /* the call's output contains vocoder / pitch-corrector samples */
    int rowsOrphaned, orphansLive; /* vocoder frames left off the grid by a vocBool-off block: moved at this call / emitting in it */
    int carryPosP[2], carryChunksP[2]; /* carried pitch frames: start relative to the call, chunks of theirs that are ever processed */
} vp_call_plan;
int vp_grid_plan(double sampleRate, int samplesPerBlock, int nCalls, const int* nBlocks, const vp_params* params,
                 vp_call_plan* out);

/* ---- processing ----------------------------------------------------------- */
/* Device-resident batch. Layouts (row stride = strideSamples floats):
 *   voice  [nStreams][stride]   synthL, synthR [nStreams][stride]
 *   outL, outR [nStreams][stride]
 * synthR may be NULL: the right side-chain channel then equals the left one (the
 * vocoder analyses channel 0 only, VocoderProcess.cpp:211,218; channel 1 is only
 * heard through the dry side-chain mix, gainSynth > -59 dB). When it is given its
 * ring is carried on every call whatever gainSynth is, as in the reference
 * (MyBuffer.cpp:69-92), so gainSynth can be automated on mid-stream. outR may be
 * NULL (then only L is written; L == R for every stream whose gainSynth <= -59 dB).
 * The outputs must NOT overlap the inputs (no in-place use: the mix reads the
 * delayed inputs while the outputs are being written) -- VP_E_ARG otherwise.
 * Asynchronous on the engine's stream; vp_engine_sync waits.
 * If a process call fails after its first pass has been issued (VP_E_CUDA /
 * VP_E_NOMEM), part of the streams' carried state has advanced: every later
 * process call returns VP_E_STATE until vp_engine_reset or vp_engine_prepare. */
int vp_engine_process_device(vp_engine* e, int nBlocks, const float* voice, const float* synthL,
                             const float* synthR, float* outL, float* outR, size_t strideSamples);

/* Host buffers (pageable or pinned, see vp_host_alloc), same layouts. Streams
 * are moved in slices with H2D / compute / D2H overlapped on three CUDA
 * streams; returns when the outputs are in host memory. */
int vp_engine_process_host(vp_engine* e, int nBlocks, const float* voice, const float* synthL,
                           const float* synthR, float* outL, float* outR, size_t strideSamples);

/* Same call with 16-bit PCM host arrays (int16 [nStreams][stride]): the samples cross the host link as 2 bytes and are
 * converted on the device exactly as the WAV front-end converts on the host (csrc/vp_wav.hpp: x / 32768 in,
 * clamp(rint(y * 32768)) out), so the result is bit-identical to converting on the host and calling
 * vp_engine_process_host, then quantising its output. For hosts whose audio is PCM anyway (files, capture devices): half
 * the link bytes of the float call, and the link is what bounds the end-to-end rate (DESIGN.md). Not a format of the
 * reference's processBlock (JUCE buffers are float): an extension of the WAV front-end of SURVEY.md 8(f)#3. */
int vp_engine_process_host_pcm16(vp_engine* e, int nBlocks, const int16_t* voice, const int16_t* synthL,
                                 const int16_t* synthR, int16_t* outL, int16_t* outR, size_t strideSamples);

int vp_engine_sync(vp_engine* e);

/* Low-latency streaming, one host block per call (BASELINE config 5). The engine owns pinned host buffers
 * voice / synthL / outL, each float[nStreams][samplesPerBlock]: fill the inputs, call vp_engine_stream_block, read
 * outL when it returns (L == R; gainSynth must be off on every stream, else VP_E_ARG; synthR is not carried). Equivalent to
 * vp_engine_process_host(e, 1, ...). The block's H2D copies, kernels and D2H copy are replayed from a CUDA graph
 * captured the first time each block phase (position of the block on the frame grids) occurs. Per-stream key and gain
 * changes between blocks need no new capture (the table is uploaded before the graph is launched); whether some stream has
 * the dry voice on is part of the graph's identity (it selects the mix kernel). */
int vp_engine_stream_buffers(vp_engine* e, float** voice, float** synthL, float** outL);
int vp_engine_stream_block(vp_engine* e);
int vp_engine_stream_stats(const vp_engine* e, uint64_t* graphLaunches, uint64_t* graphCaptures);

/* Decisions of the most recent process call for one stream: up to cap
 * records, *nFrames = frames available. */
int vp_engine_get_pitch_frames(vp_engine* e, int stream, vp_pitch_frame* out, int cap, int* nFrames);
/* Per vocoder frame of the most recent call: gate flag, excitation energies
 * and gain (VocoderProcess.cpp:199-204, :264-272). Arrays may be NULL. */
int vp_engine_get_voc_frames(vp_engine* e, int stream, int cap, int* nFrames, uint8_t* gated, double* EeVoice,
                             double* EeSynth, double* g);

/* Counters since prepare: kernels launched, frames re-decided in FP64. */
int vp_engine_get_stats(const vp_engine* e, uint64_t* kernelLaunches, uint64_t* yinRechecked,
                        uint64_t* yinFrames);
/* Device time (ms) of the most recent process_device call, measured with
 * CUDA events on the engine's stream; per-stage breakdown optional. */
#define VP_NSTAGES 16
int vp_engine_last_timing(vp_engine* e, float* totalMs, float* stageMs /* [VP_NSTAGES] or NULL */);
/* Number of timed intervals (= kernel launches of that stage) behind each stageMs entry. */
int vp_engine_last_timing_counts(vp_engine* e, int* stageCount /* [VP_NSTAGES] */);
const char* vp_stage_name(int stage);
/* accumulate != 0: vp_engine_last_timing sums over every process call since this reset
 * (total = first call's start .. last call's end); 0 (default): most recent call only. */
int vp_engine_timing_reset(vp_engine* e, int accumulate);
/* Device timers on the engine's stream (CUDA events), slots 0..7: bracket any sequence of
 * asynchronous calls; _elapsed_ms waits for slotB and returns the time since slotA. */
int vp_engine_timer_record(vp_engine* e, int slot);
int vp_engine_timer_elapsed_ms(vp_engine* e, int slotA, int slotB, float* ms);

/* ---- memory helpers -------------------------------------------------------- */
int vp_host_alloc(void** p, size_t bytes);   /* pinned host memory */
void vp_host_free(void* p);
int vp_device_alloc(vp_engine* e, void** p, size_t bytes);
void vp_device_free(vp_engine* e, void* p);
int vp_memcpy_h2d(vp_engine* e, void* dst, const void* src, size_t bytes);
int vp_memcpy_d2h(vp_engine* e, void* dst, const void* src, size_t bytes);

/* ---- synthetic inputs (SURVEY.md 8(d)) -------------------------------------- */
/* flavour: 0 = breathy voice (-40 dBFS aspiration), 1 = clean (-80 dBFS),
 * 2 = breathy with a silent stretch (exercises the gates). Streams are
 * numbered firstStream.. so shards generate disjoint inputs. */
int vp_synth_host(double sampleRate, int flavour, int firstStream, int nStreams, size_t nSamples,
                  size_t strideSamples, float* voice, float* synthL, float* synthR);
int vp_synth_device(vp_engine* e, double sampleRate, int flavour, int firstStream, int nStreams,
                    size_t nSamples, size_t strideSamples, float* voice, float* synthL, float* synthR);

/* ---- measurement helpers ---------------------------------------------------- */
/* Issue-rate microbenchmarks on the engine's device: FP32 FMA and FP64 FMA
 * lane-operations per second (the roofline denominators of DESIGN.md). */
int vp_measure_peaks(vp_engine* e, double* fp32FmaPerSec, double* fp64FmaPerSec);
/* Same, with the operand pattern of the engine's inner loops (acc_i = fma(x, b_i, acc_i): two distinct register
 * operands per FMA instead of one) -- the rate a real multiply-accumulate loop can reach. */
int vp_measure_peaks2(vp_engine* e, double* fp32FmaPerSec, double* fp64FmaPerSec);

#ifdef __cplusplus
}
#endif
#endif /* VP_ENGINE_H */
