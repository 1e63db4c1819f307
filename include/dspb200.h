/*
 * dspb200.h — C ABI of the B200 batch engine for dsp-stuff's effect-node path.
 *
 * This is the drop-in boundary.  Every entry point below names the reference
 * interface it replaces (paths relative to the reference tree, simmsb/dsp-stuff).
 * Plain pointers and sizes only: no C++ types, no torch types, no exceptions
 * cross this boundary.  All functions return DSPB_OK (0) or a negative
 * dspb_status; dspb_last_error() gives the message for the calling thread.
 *
 * Data model
 *   A graph is instantiated once and run over `channels` independent mono
 *   streams.  All audio is f32, laid out channel-major: buffer[c * n + i] is
 *   sample i of channel c ("[C x n] SoA rows").  Filter/delay/FIR state is per
 *   channel.  Parameters are shared by all channels unless a field is given one
 *   value per channel (dspb_node_set_f32_channels) or a FIR node one impulse
 *   response per channel (dspb_node_set_taps_channels); enum fields,
 *   reverb.seconds and the FIR tap count are always shared.
 *
 * Threading: one caller thread per engine handle at a time; setters are legal
 * between dspb_process calls and take effect at the next call (the reference
 * applies slider changes at the next 128-sample block: runtime.rs:264,
 * dsp-stuff-derive/src/lib.rs:487-497).
 */
#ifndef DSPB200_H
#define DSPB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSPB_ABI_VERSION 2

typedef enum dspb_status {
    DSPB_OK = 0,
    DSPB_ERR_INVALID = -1,      /* bad argument (null, range, size not a multiple of ref_block) */
    DSPB_ERR_UNKNOWN_NODE = -2, /* unknown cfg_name / node id (reference: panic, runtime.rs:634-637) */
    DSPB_ERR_UNKNOWN_PORT = -3, /* unknown port / field / enum variant (reference: .unwrap() panic, nodes/gain.rs:30-31) */
    DSPB_ERR_GRAPH = -4,        /* cycle, not compiled, or graph changed without dspb_compile */
    DSPB_ERR_CUDA = -5,         /* CUDA runtime error (message in dspb_last_error) */
    DSPB_ERR_NOMEM = -6,
    DSPB_ERR_PARSE = -7         /* malformed graph JSON (reference: serde unwrap panic, lib.rs:329) */
} dspb_status;

/* Where the audio buffers handed to dspb_process live. */
#define DSPB_MEM_DEVICE 0 /* device pointers, work is enqueued on `stream`, call returns immediately */
#define DSPB_MEM_HOST 1   /* host pointers (pinned for full speed); H2D, kernels and D2H are pipelined
                             inside the call, which returns after the outputs are complete */

#define DSPB_MEM_HOST_ASYNC 2 /* like DSPB_MEM_HOST, but the call returns as soon as the work is enqueued on the engine's
                                own streams: the next call's H2D overlaps this call's D2H.  The caller keeps both host
                                buffers untouched (pinned memory, or the copies degrade to synchronous ones) until
                                dspb_sync returns, and passes DIFFERENT buffers to calls that may be in flight together. */

typedef struct dspb_engine dspb_engine;

/* Engine configuration.  Constants the reference hard-codes are fields here so
 * they are visible: sample_rate 48000 (README.md:48, nodes/reverb.rs:58,
 * nodes/signal_gen.rs:60), ref_block 128 (node.rs:257). */
typedef struct dspb_config {
    int32_t channels;     /* C: number of independent mono streams on this engine/GPU */
    int32_t block;        /* device block B (multiple of ref_block); dspb_process takes k*B samples */
    int32_t sample_rate;  /* 0 -> 48000 */
    int32_t ref_block;    /* 0 -> 128; Distort::Fuzz and SignalGen are evaluated per ref_block */
    int32_t ring_granule; /* 0 -> 1024.  Reverb ring capacity is rounded up to this many samples
                             (rivulet@b2416e5 page-mirrored ring; UNPINNED, see DESIGN.md).  1 = nominal */
    int32_t device;       /* CUDA device ordinal; -1 = planning only (dspb_compile / dspb_describe_plan work
                             without a GPU, dspb_process fails with DSPB_ERR_CUDA) */
    int64_t max_samples;  /* largest n_samples a single dspb_process call will pass; 0 -> 64*block */
    int32_t fir_fft_log2; /* 0 -> engine default (13); FFT size of the overlap-save FIR path */
    int32_t fir_mode;     /* 0 -> overlap-save FFT in f32 (throughput path); 1 -> direct time-domain sum in f64 in
                             the reference's summation order (bit-exact; 8192 f64 flop/sample at 4096 taps);
                             2 -> Toeplitz-tiled tensor-core GEMM (tcgen05, split bf16 operands, f32 accumulate;
                             the comparison path of BASELINE config 4, within the 1e-5 parity bar);
                             3 -> experimental FFT variant carrying two sub-transforms per f32x2 register pair */
    int32_t iir_mode;     /* 0 -> every recurrence (biquad.rs:87, low_pass.rs:36-39, high_pass.rs:36-39) is evaluated strictly
                             sequentially in the reference's operation order: bit-identical, but a launch with few channels
                             is bound by the 12-cycle dependent chain per sample.
                             1 -> opt-in time-parallel evaluation (chunked zero-state responses + a warp-shuffle scan of the
                             2x2 state transition over the block, FMA): NOT bit-exact.  It is enabled PER FILTER only when
                             the error measured at dspb_compile on a probe signal (scan vs exact, on the device) is below
                             5e-6 of the output peak, half of the 1e-5 parity bar (with the carried states computed in f64
                             the scan is closer to exact filtering than the reference's own f32 evaluation, so what the
                             probe measures is essentially the reference's rounding error); a filter that fails the probe
                             (e.g. a 200 Hz high-pass in f32) keeps the exact path.  dspb_describe_plan shows the verdicts. */
} dspb_config;

/* ---- lifetime ----------------------------------------------------------------------------- */

/* Replaces: UiContext::new (runtime.rs:51-88) minus GUI/tokio.  Fails with DSPB_ERR_CUDA when no
 * CUDA device is usable: there is no CPU fallback. */
int dspb_engine_create(const dspb_config* cfg, dspb_engine** out);
void dspb_engine_destroy(dspb_engine* e);
const char* dspb_last_error(void);
int dspb_abi_version(void);

/* ---- graph construction ------------------------------------------------------------------- */

/* Replaces: nodes::RESTORE / nodes::NODES constructor tables (nodes/mod.rs:65-123) and the
 * derive-generated NodeStatic::new (dsp-stuff-derive/src/lib.rs:163-231).  `cfg_name` is the
 * reference typename: gain, distort, overdrive, chebyshev, biquad, low_pass, high_pass, reverb,
 * fir, add, mix, mux, demux, envelope, signal_gen, plus the graph terminals input / output
 * (nodes/input.rs, nodes/output.rs: here they bind to dspb_process buffers, in creation order).
 * Fields start at the reference defaults (#[dsp(default = ...)]). */
int dspb_node_add(dspb_engine* e, const char* cfg_name, int64_t node_id);

/* Replaces: the derive-generated slider store (lib.rs:487-497) + after_settings_change
 * (lib.rs:560-568): BiQuad::regenerate_filter resets that node's state (nodes/biquad.rs:62-76),
 * Reverb::refresh_seconds replaces the ring with a zero-filled one (nodes/reverb.rs:55-71).
 * Values are NOT clamped to the slider range (restore() does not clamp either, lib.rs:295-309). */
int dspb_node_set_f32(dspb_engine* e, int64_t node_id, const char* field, float value);

/* Per-channel slider values: channel c of this engine runs node `node_id` as if dspb_node_set_f32(field, values[c]) had been
 * called on a one-channel engine holding only channel c.  values: host pointer, n_values == channels.
 *   - Side effects are those of dspb_node_set_f32: a biquad regenerates its coefficients (per channel) and resets the state
 *     of every channel; a reverb replaces its ring with a zero-filled one.  Takes effect at the next dspb_process.
 *   - All values bit-identical (NaN payloads and the sign of zero count): exactly dspb_node_set_f32(values[0]), same plan,
 *     same kernels, same outputs.
 *   - A later dspb_node_set_f32 on the same field makes it shared again; other fields are not affected.
 *   - Every f32 field except reverb.seconds may vary per channel.  reverb.seconds fails with DSPB_ERR_INVALID: it sets the
 *     ring length D, and the ring is one [C x D] array with one D for all channels.
 *   - A linked control port (<field>_input, lib.rs:122-161) still overrides the slider: its per-channel values are unused
 *     while the port is linked.
 *   - Errors: DSPB_ERR_UNKNOWN_NODE (node id), DSPB_ERR_UNKNOWN_PORT (no such f32 field), DSPB_ERR_INVALID (null pointer,
 *     n_values != channels, reverb.seconds).
 *   - Planning engines (device -1) accept the call; dspb_describe_plan marks per-channel parameters ("per-channel[...]").
 *   - Not stored in saved-graph JSON (one scalar per field there). */
int dspb_node_set_f32_channels(dspb_engine* e, int64_t node_id, const char* field, const float* values, int64_t n_values);

/* Replaces: the derive-generated select store; `variant` is the Rust enum variant name
 * ("SoftClip", "Balanced", "A", "Sine", ...), the same string serde writes (lib.rs:266-293). */
int dspb_node_set_enum(dspb_engine* e, int64_t node_id, const char* field, const char* variant);

/* Replaces: Fir.taps (nodes/fir.rs:61-62).  `taps` is stored verbatim, i.e. already REVERSED
 * (taps[i] = h[N-1-i], nodes/fir.rs:153-171), f64.  Clears that node's history. */
int dspb_node_set_taps(dspb_engine* e, int64_t node_id, const double* taps, int64_t n);
/* Convenience for callers holding an impulse response h[0..n): reverses like the WAV loader. */
int dspb_node_set_impulse_response(dspb_engine* e, int64_t node_id, const double* h, int64_t n);

/* Per-channel impulse responses.  taps: [n_sets x n_taps] f64, row k stored REVERSED like dspb_node_set_taps;
 * set_index: [n_channels] int32, channel c runs FIR node `node_id` as if dspb_node_set_taps(taps + set_index[c] * n_taps,
 * n_taps) had been called on a one-channel engine holding only channel c.  Host pointers.
 *   - A bank plus an index: 4096 streams sharing 8 impulse responses pass 8 rows.  Bit-identical rows (memcmp over the
 *     8 * n_taps bytes) count as one set; rows no channel uses are dropped.
 *   - Every used row bit-identical: exactly dspb_node_set_taps(row), same plan, kernels and outputs.  This holds in every
 *     fir_mode (the check comes before the fir_mode check below).
 *   - Side effects are those of dspb_node_set_taps: the node's history is cleared for every channel, and the change takes
 *     effect at the next dspb_process.  A later dspb_node_set_taps / dspb_node_set_impulse_response makes the node shared again.
 *   - One tap count for all channels: the Average divisor 1/n_taps and the warm-up length (n_taps - 1 samples) are one value
 *     per node.
 *   - Cost (fir_mode 0): two channels share one complex transform only when they use the same set.  Channels are paired
 *     inside each aligned group of 32 channels; a set with an odd number of channels in a group leaves one channel that runs
 *     alone.  So a bank whose sets hold an even number of channels in every group runs as many transforms as shared taps,
 *     and fully distinct impulse responses run one channel per transform, about twice the FFT work.  Each set keeps its own
 *     320 KiB of spectra on the device.
 *   - Errors: DSPB_ERR_UNKNOWN_NODE (node id); DSPB_ERR_INVALID (not a fir node, null pointer, n_sets < 1, n_taps < 1,
 *     n_channels != channels, a set_index outside [0, n_sets), distinct sets on an engine with fir_mode 2 or 3: per-channel
 *     taps need fir_mode 0 or 1).
 *   - Planning engines (device -1) accept the call; dspb_describe_plan adds ", per-channel taps: K sets, X transforms
 *     (Y single-channel)" to the fir step line (", per-channel taps: K sets" on the direct path).
 *   - Not stored in saved-graph JSON (one taps array per node there).  dspb_node_process carries them over. */
int dspb_node_set_taps_channels(dspb_engine* e, int64_t node_id, const double* taps, int64_t n_sets, int64_t n_taps,
                                const int32_t* set_index, int64_t n_channels);
/* Same with impulse responses h (each row h[0..n_taps) in time order, reversed per row like dspb_node_set_impulse_response). */
int dspb_node_set_impulse_response_channels(dspb_engine* e, int64_t node_id, const double* h, int64_t n_sets, int64_t n_taps,
                                            const int32_t* set_index, int64_t n_channels);

/* Replaces: UiContext::add_link (runtime.rs:125-134): lhs = (producer node, output port),
 * rhs = (consumer node, input port); ports by name (node.rs:87-89).  Several links may leave one
 * output port (fan-out, node.rs:321-325) or enter one input port (fan-in, averaged by
 * collect_and_average, node.rs:162-194).  The engine sums a port's links in link-creation order; the reference
 * iterates a HashSet<LinkId> (runtime.rs:38-39), i.e. in unspecified order, so with three or more links into one
 * port the sum is reproducible against the reference only up to f32 rounding of the addition order (one or two
 * links: order-independent, bit-exact). */
int dspb_link(dspb_engine* e, int64_t src_node, const char* out_port, int64_t dst_node, const char* in_port);

/* Replaces: UiContext::restore_config (runtime.rs:94-123) for the saved-graph JSON
 * DSPConfig{nodes:[{id,typename,position,cfg}],links:[{lhs:[node,port],rhs:[node,port]}]}
 * (runtime.rs:44-48, 560-564, 606-612).  Adds to an empty engine.  `input` / `output` entries keep their
 * cpal fields selected_host / selected_device (nodes/input.rs:33-38, nodes/output.rs:33-38), which are ignored:
 * terminals bind to dspb_process buffers.  GUI-only sinks (wave_view, spectrogram, pitch: nodes/mod.rs:111-122) are
 * dropped together with the links into them.  `muff` (private GPL crate, source unavailable) and any other unknown
 * typename fail with DSPB_ERR_UNKNOWN_NODE, where the reference panics (runtime.rs:634-637). */
int dspb_load_graph_json(dspb_engine* e, const char* json_utf8);

/* Replaces: UiContext::update_all / NodeInstance::start (runtime.rs:136-151, 646-732): builds the
 * topological kernel schedule.  Must be called after the last structural change. */
int dspb_compile(dspb_engine* e);

/* ---- the hot path ------------------------------------------------------------------------- */

/* Replaces: the per-node task loop `loop { instance.perform(..) }` (runtime.rs:718-728) and the
 * blanket `impl<T: SimpleNode> Perform for T` (node.rs:267-352) over the whole graph, for all
 * channels and n_samples consecutive samples per channel (n_samples % ref_block == 0).
 * inputs[i]  : [C x n_samples] f32 for the i-th `input` terminal (raw samples, nodes/input.rs:226)
 * outputs[j] : [C x n_samples] f32 for the j-th `output` terminal (after its own fan-in average,
 *              nodes/output.rs:223)
 * State (IIR, rings, FIR history, clocks) carries over to the next call. */
int dspb_process(dspb_engine* e, const float* const* inputs, float* const* outputs, int64_t n_samples,
                 int mem_kind, void* cuda_stream);

/* Waits for every DSPB_MEM_HOST_ASYNC call issued on this engine (outputs complete, input buffers free again). */
int dspb_sync(dspb_engine* e);

/* Replaces: one call of SimpleNode::process(ProcessInput, ProcessOutput) (node.rs:135-146) on one
 * node, batched over channels: inputs are taken as ALREADY averaged port buffers with their
 * `present` flags (node.rs:217-238); no fan-in division is applied.  ports in index order
 * (lib.rs:214-219).  A null input pointer means an unconnected port (zeros, present=false). */
int dspb_node_process(dspb_engine* e, int64_t node_id, const float* const* port_inputs,
                      const uint8_t* present, float* const* port_outputs, int64_t n_samples,
                      int mem_kind, void* cuda_stream);

/* ---- device-boundary format steps (SURVEY.md §8f N4) ---------------------------------------- */

/* Replaces: the stereo fold of the capture callback, devices.rs:244-262 `do_read_2`: interleaved frames
 * [C x n_frames x 2] -> mono [C x n_frames], out = a + b (f32 add, not an average).  Any n_frames >= 0. */
int dspb_fold_stereo(dspb_engine* e, const float* interleaved, float* mono, int64_t n_frames, int mem_kind, void* cuda_stream);
/* Replaces: the mono -> stereo duplicate of the playback callback, devices.rs:443-500 `do_write_2`
 * (`o.fill(x)`): mono [C x n_frames] -> interleaved [C x n_frames x 2] at the graph's own rate.  With the 48 kHz ->
 * device-rate converter in front of it: dspb_resample_dup_stereo below. */
int dspb_dup_stereo(dspb_engine* e, const float* mono, float* interleaved, int64_t n_frames, int mem_kind, void* cuda_stream);

/* Replaces: the playback callback's sample-rate converter + duplicate, devices.rs:443-500 `do_write_2` with the converter
 * built at devices.rs:550-556: `Converter::from_hz_to_hz(CountingSignal, Sinc::new(Fixed::from([0.0; 16])), 48_000.0, target)`
 * (dasp_signal 0.11.0 / dasp_interpolate 0.11.0, un-vendored: restated from the published crates, parity UNPINNED).
 * mono [C x n_in] at the engine's sample rate -> interleaved stereo [C x n_out x 2] at target_hz, both slots of a frame equal.
 * The converter state (fractional position, the 16-frame sinc ring) carries over to the next call with the same target_hz; a
 * different target_hz or dspb_reset_state starts a fresh converter.  *consumed (may be NULL) = input samples taken, what
 * do_write_2 releases from the link ring; input beyond n_in reads as zeros (CountingSignal::next, devices.rs:380-386). */
int dspb_resample_dup_stereo(dspb_engine* e, const float* mono, float* interleaved, int64_t n_in, int64_t n_out,
                             double target_hz, int mem_kind, void* cuda_stream, int64_t* consumed);

/* Clears all per-channel state (what a fresh NodeStatic::new / restore gives).  Drops any pending dspb_reset_channels request. */
int dspb_reset_state(dspb_engine* e);

/* Per-channel state reset: from the next dspb_process on, every listed channel behaves as if dspb_reset_state had been
 * called on a one-channel engine holding only that channel (same graph, same parameters, same per-channel values and
 * impulse responses).  Unlisted channels are not touched.  channels: host pointer to n_channels indices in [0, channels).
 * This is how a service recycles a stream slot: reset the slot, then set its per-channel values.
 *   - Reset, for each listed channel: the [C x 4] state row of every biquad, low_pass, high_pass, envelope, gate and
 *     signal_gen node, its reverb ring rows, its FIR input history, and its FIR warm-up (the first n_taps - 1 samples after
 *     the reset are summed over the samples seen since, as for a fresh node, fir.rs:192-216), which may span several calls.
 *   - Not reset: parameters, per-channel values and impulse responses, the plan; the dspb_resample_dup_stereo converter,
 *     whose position is shared by all channels; the sub-engines of dspb_node_process (dspb_reset_state leaves those alone too).
 *   - The call only records the request; it neither blocks nor synchronises.  Requests accumulate until the next
 *     dspb_process, which enqueues the clear in front of its first kernel on the stream that orders it (`cuda_stream` for
 *     DSPB_MEM_DEVICE, the engine's compute stream for the host paths), so a reset recorded between two DSPB_MEM_HOST_ASYNC
 *     calls falls exactly between them.  Duplicate indices are allowed; resetting a channel again restarts its warm-up.
 *   - Cost: nothing while no request is pending and no reset channel is in its warm-up.  Otherwise one clear launch for the
 *     call after the reset, and one direct-kernel launch per FIR step (and channel range) while a reset channel is in its
 *     warm-up.  A FIR node on the short-call (UPC) path re-primes its delay line once.
 *   - n_channels == 0 is a no-op (channels may be NULL).  Errors, nothing recorded: DSPB_ERR_INVALID (null engine,
 *     n_channels < 0, channels NULL with n_channels > 0, an index outside [0, channels)).
 *   - Planning engines (device -1) accept the call; dspb_node_get_i64(e, 0, "pending_resets") counts the distinct channels
 *     recorded and not yet consumed. */
int dspb_reset_channels(dspb_engine* e, const int32_t* channels, int64_t n_channels);

/* ---- introspection (index work that must match the reference bit-exactly) ------------------ */

/* keys: "delay_samples" (reverb: ring length D, nodes/reverb.rs:58-68), "n_taps" (fir),
 *       "n_inputs" / "n_outputs" (port counts), "kernel_launches" (engine, node_id ignored:
 *       kernels launched by the last dspb_process), "n_segments" (engine: fused segments),
 *       "pending_resets" (engine: distinct channels recorded by dspb_reset_channels for the next dspb_process). */
int dspb_node_get_i64(dspb_engine* e, int64_t node_id, const char* key, int64_t* out);
/* Port name -> local index, as PortStorage::get_idx on a freshly built node (node.rs:74-89). */
int dspb_node_port_index(dspb_engine* e, int64_t node_id, const char* port, int is_output, int32_t* out);
/* Per-step device timing (CUDA events on the launching stream around every step of the schedule).
 * dspb_profile_enable(e, 1) starts recording on subsequent device-pointer dspb_process calls;
 * dspb_profile_read synchronises, returns for each step i < cap the summed milliseconds and the
 * number of launches-rounds measured, and clears the record.  Returns the number of steps. */
int dspb_profile_enable(dspb_engine* e, int on);
int dspb_profile_read(dspb_engine* e, double* ms_total, int64_t* rounds, int cap);

/* Human-readable schedule (segments, ops, buffers) for DESIGN/profiling; returns bytes needed. */
int64_t dspb_describe_plan(dspb_engine* e, char* buf, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* DSPB200_H */
