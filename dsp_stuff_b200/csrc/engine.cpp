// engine.cpp — host side of the B200 batch engine: node registry, graph model, topological
// scheduler that lowers the graph to fused device programs + FIR steps, state/ring/FIR memory, and
// the C ABI declared in include/dspb200.h.
//
// Replaces (reference paths relative to dsp-stuff/src):
//   nodes/mod.rs:65-123 (type registry)            -> kNodeTypes
//   dsp-stuff-derive/src/lib.rs:163-231 (defaults, port order) -> NodeType tables
//   runtime.rs:125-224, 646-732 (links, per-port link vectors, task loops) -> Engine::compile / process
//   node.rs:162-194, 267-352 (fan-in average, per-block wrapper) -> lowering in Lowerer
// There is no CPU execution path in this file: every dspb_process ends in CUDA launches.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <vector>

#include "../../include/dspb200.h"
#include "json_min.h"
#include "plan.h"

using namespace dspb;

namespace {

thread_local std::string g_err;
int fail(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CUDA_TRY(expr)                                                                        \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) return fail(DSPB_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

// ---- node registry: verbatim mirror of the #[dsp(...)] blocks (SURVEY.md Appendix A) -------------------
enum TypeId { T_GAIN, T_DISTORT, T_OVERDRIVE, T_CHEBY, T_BIQUAD, T_LOWPASS, T_HIGHPASS, T_REVERB, T_FIR,
              T_ADD, T_MIX, T_MUX, T_DEMUX, T_ENVELOPE, T_SIGGEN, T_GATE, T_INPUT, T_OUTPUT, T_COUNT };

struct ParamDef {
    const char* name;
    float def, lo, hi;
    int ctl_port;  // input-port index of the same-named control port (slider(as_input)), -1 if none
};
struct EnumDef {
    const char* name;
    std::vector<const char*> variants;
    int def;
};
struct NodeType {
    const char* cfg_name;
    std::vector<const char*> ins, outs;
    std::vector<ParamDef> params;
    std::vector<EnumDef> enums;
};

const NodeType kNodeTypes[T_COUNT] = {
    /* gain       nodes/gain.rs:5-23      */ {"gain", {"in", "level"}, {"out"}, {{"level", 1.0f, 0.f, 10.f, 1}}, {}},
    /* distort    nodes/distort.rs:18-51  */
    {"distort", {"in", "level"}, {"out"}, {{"level", 0.0f, 0.f, 30.f, 1}},
     {{"mode", {"HardClip", "SoftClip", "Tanh", "RecipSoftClip", "Fuzz", "Sin", "Atan", "Square", "Chebyshev4"}, 1}}},
    /* overdrive  nodes/overdrive.rs:5-29 */
    {"overdrive", {"in", "boost", "drive", "level"}, {"out"},
     {{"boost", 0.f, 0.f, 30.f, 1}, {"drive", 0.f, 0.f, 1.f, 2}, {"level", 0.f, 0.f, 1.f, 3}}, {}},
    /* chebyshev  nodes/chebyshev.rs:5-26 */
    {"chebyshev", {"in"}, {"out"}, {{"level_pos", 0.f, 0.f, 50.f, -1}, {"level_neg", 0.f, 0.f, 50.f, -1}}, {}},
    /* biquad     nodes/biquad.rs:8-45    */
    {"biquad", {"in"}, {"out"},
     {{"a0", 1.0f, -10.f, 10.f, -1}, {"a1", -0.24f, -10.f, 10.f, -1}, {"a2", 0.f, -10.f, 10.f, -1},
      {"b0", 0.758f, -10.f, 10.f, -1}, {"b1", 0.f, -10.f, 10.f, -1}, {"b2", 0.f, -10.f, 10.f, -1}}, {}},
    /* low_pass   nodes/low_pass.rs:4-24 (its cfg_name() says "high_pass"; RESTORE key is low_pass) */
    {"low_pass", {"in"}, {"out"}, {{"ratio", 0.5f, 0.f, 1.f, -1}}, {}},
    /* high_pass  nodes/high_pass.rs:4-24 */ {"high_pass", {"in"}, {"out"}, {{"ratio", 0.5f, 0.f, 1.f, -1}}, {}},
    /* reverb     nodes/reverb.rs:12-42   */
    {"reverb", {"in"}, {"out"}, {{"seconds", 0.5f, 0.f, 1.f, -1}, {"decay", 0.5f, 0.f, 1.f, -1}}, {}},
    /* fir        nodes/fir.rs:19-66      */ {"fir", {"in"}, {"out"}, {}, {{"mode", {"Average", "Balanced"}, 1}}},
    /* add        nodes/add.rs:4-20       */ {"add", {"a", "b"}, {"out"}, {}, {}},
    /* mix        nodes/mix.rs:5-29       */ {"mix", {"a", "b", "ratio"}, {"out"}, {{"ratio", 0.5f, 0.f, 1.f, 2}}, {}},
    /* mux        nodes/mux.rs:5-41       */ {"mux", {"a", "b"}, {"out"}, {}, {{"in_port", {"A", "B"}, 0}}},
    /* demux      nodes/demux.rs:5-41     */ {"demux", {"in"}, {"a", "b"}, {}, {{"out_port", {"A", "B"}, 0}}},
    /* envelope   nodes/envelope.rs:9-32  */
    {"envelope", {"in"}, {"out"}, {{"attack", 0.f, 0.f, 1000.f, -1}, {"release", 0.f, 0.f, 1000.f, -1}}, {}},
    /* signal_gen nodes/signal_gen.rs:6-53 */
    {"signal_gen", {"amplitude", "frequency"}, {"out"},
     {{"amplitude", 0.5f, -1.f, 1.f, 0}, {"frequency", 100.0f, 0.1f, 20000.f, 1}},
     {{"mode", {"Sine", "Triangle", "Square", "Constant"}, 0}}},
    /* gate       EXTENSION, not a reference node (SURVEY.md: north_star names a noise gate, the reference has none):
                  out = envelope(in) >= threshold ? in : 0 with nodes/envelope.rs's detector (attack / release in frames) */
    {"gate", {"in"}, {"out"}, {{"threshold", 0.f, 0.f, 1.f, -1}, {"attack", 0.f, 0.f, 1000.f, -1}, {"release", 0.f, 0.f, 1000.f, -1}}, {}},
    /* input      nodes/input.rs:12-22    */ {"input", {}, {"out"}, {}, {}},
    /* output     nodes/output.rs:12-22   */ {"output", {"in"}, {}, {}, {}},
};

// Planning-only engines (device == -1: build and describe schedules, nothing can run) are a PER-ENGINE property:
// a planning engine and a real engine may live in one process, on different threads.
struct DevBuf {  // owning device allocation
    float* p = nullptr;
    size_t bytes = 0;
    bool fake = false;
    ~DevBuf() { if (p && !fake) cudaFree(p); }
    int alloc(size_t n_bytes, bool zero, bool plan_only) {
        if (p && !fake) cudaFree(p);
        p = nullptr;
        bytes = 0;
        if (n_bytes == 0) return DSPB_OK;
        if (plan_only) { fake = true; p = reinterpret_cast<float*>(uintptr_t(16)); bytes = n_bytes; return DSPB_OK; }
        cudaError_t e = cudaMalloc(&p, n_bytes);
        if (e != cudaSuccess) { p = nullptr; return fail(DSPB_ERR_NOMEM, "cudaMalloc(%zu): %s", n_bytes, cudaGetErrorString(e)); }
        bytes = n_bytes;
        if (zero) {
            e = cudaMemset(p, 0, n_bytes);
            if (e != cudaSuccess) return fail(DSPB_ERR_CUDA, "cudaMemset: %s", cudaGetErrorString(e));
        }
        return DSPB_OK;
    }
};

struct Node {
    int64_t id;
    int type;
    std::vector<float> f32;   // by ParamDef index
    std::vector<std::vector<float>> f32_pc;  // by ParamDef index: per-channel values (dspb_node_set_f32_channels), empty = shared;
                                             // f32 then holds channel 0's value
    std::vector<int> enums;   // by EnumDef index
    // biquad: normalised coefficients (regenerate_filter, nodes/biquad.rs:62-76)
    float bq[5] = {0.758f, 0.f, 0.f, -0.24f, 0.f};  // b0 b1 b2 a1 a2 (initial_filter, biquad.rs:48-55)
    // reverb
    int64_t D = 0, pos = 0;
    DevBuf ring;
    bool ring_dirty = true;
    // stateful recurrences
    DevBuf state;  // [C x 4] f32
    // fir
    std::vector<double> taps{1.0};  // reversed, nodes/fir.rs:61
    DevBuf U;                       // [C x u_ring] input rings: a call's sample i sits at slot (u_pos + i) mod u_ring, the
                                    // previous hist_pad samples right behind it -- history carries over without a copy
    int u_ring = 0, u_pos = 0;      // u_ring = round_up(hist_pad + max_samples, 128)
    DevBuf Y;                       // [C x max_samples]
    std::vector<std::unique_ptr<DevBuf>> fft_work;  // persistent FFT kernels: work counters, one set per launch lane
    DevBuf fdl;                     // short calls (UPC kernel): frequency-domain delay line, [pairs][P][2048] complex
    bool fdl_valid = false;         // the previous call was a UPC call: the FDL holds the P-1 previous block spectra
    bool upc_this_call = false;
    int64_t upc_ctr = 0;            // running block counter (FDL slot = counter mod P)
    DevBuf H, taps_dev;
    DevBuf toep_tiles, toep_split;  // FIR_TOEPLITZ: Toeplitz tiles of the taps, hi/lo bf16 split of U
    int hist_pad = 0;
    int64_t started = 0;            // samples this node has consumed since reset
    bool fir_dirty = true;
    // Per-channel impulse responses (dspb_node_set_taps_channels); all empty when the taps are shared.  `taps` then holds
    // set 0 (channel 0's), so taps.size() is the one tap count of every set.
    std::vector<double> fir_bank;   // [K x N] reversed taps of the K distinct sets, in order of first use by a channel
    std::vector<int32_t> fir_set;   // [C] set of each channel
    std::vector<int4> fir_xf;       // transform table {chA, chB or -1, set, 0}, see fir_transforms
    std::vector<int> fir_xf_group;  // [ceil(C / 32) + 1] index of each 32-channel group's first transform
    int fir_xf_single = 0;          // transforms that carry one channel
    DevBuf set_dev, xf_dev;         // fir_set and fir_xf on the device
    bool fir_pc() const { return !fir_set.empty(); }
};

// Transform table of per-channel impulse responses.  Two channels share one complex transform only when they use the same set.
// Transforms are formed inside each aligned group of 32 channels: the group's channels are sorted stably by set (sets in order
// of first appearance in the group), consecutive channels of one set are paired, and an odd one left over runs alone (B mirrors
// A and is never stored).  Every launch range [c_begin, c_end) starts on a multiple of 32 and ends on one or at C, so it
// covers one contiguous slice of the table, the same slice on every call.
void fir_transforms(Node& n, int C) {
    n.fir_xf.clear();
    n.fir_xf_group.clear();
    n.fir_xf_single = 0;
    for (int g0 = 0; g0 < C; g0 += 32) {
        n.fir_xf_group.push_back((int)n.fir_xf.size());
        const int g1 = std::min(C, g0 + 32);
        std::vector<int> order;   // sets of the group in order of first appearance
        for (int c = g0; c < g1; c++)
            if (std::find(order.begin(), order.end(), n.fir_set[c]) == order.end()) order.push_back(n.fir_set[c]);
        for (int k : order) {
            int pending = -1;
            for (int c = g0; c < g1; c++) {
                if (n.fir_set[c] != k) continue;
                if (pending < 0) {
                    pending = c;
                } else {
                    n.fir_xf.push_back(make_int4(pending, c, k, 0));
                    pending = -1;
                }
            }
            if (pending >= 0) {
                n.fir_xf.push_back(make_int4(pending, -1, k, 0));
                n.fir_xf_single++;
            }
        }
    }
    n.fir_xf_group.push_back((int)n.fir_xf.size());
}

void copy_fir_pc(Node& dst, const Node& src) {  // dspb_node_process: per-channel impulse responses carry over to the sub-engine
    dst.fir_bank = src.fir_bank;
    dst.fir_set = src.fir_set;
    dst.fir_xf = src.fir_xf;
    dst.fir_xf_group = src.fir_xf_group;
    dst.fir_xf_single = src.fir_xf_single;
}

struct Link { int src, sport, dst, dport; };

enum StepKind { STEP_FUSED, STEP_FIR };
struct Step {
    StepKind kind;
    Program prog;   // STEP_FUSED
    int G = 1;
    int fir_node = -1;
    int fir_out_term = -1;   // >= 0: the FIR kernel applies the sink's fan-in average and writes output terminal t directly
    float fir_post_nf = 0.0f;
    // which prog.bufs entries are rebound per call: ext input terminal t (>=0), ext output terminal t, scratch, fir U/Y
    struct Bind { int kind; int idx; };  // kind 0 ext-in, 1 ext-out, 2 scratch, 3 fir U (idx=node), 4 fir Y (idx=node)
    std::vector<Bind> binds;             // parallel to prog.bufs
    std::vector<int> ring_nodes;         // parallel to prog.rings
    std::vector<int> nodes;              // STEP_FUSED: the nodes (engine indices) whose ops this segment holds, in order
    std::vector<float> pc_host;          // STEP_FUSED: per-channel parameter table [C x pc_k] (plan.h Program::pc), or empty
    int pc_k = 0;
    std::string text;                    // human-readable listing
};

}  // namespace

struct dspb_engine {
    dspb_config cfg{};
    std::vector<std::unique_ptr<Node>> nodes;
    std::vector<Link> links;
    bool compiled = false;
    bool lowered = false;
    std::vector<int> order, in_terms, out_terms;
    std::vector<std::vector<std::vector<int>>> in_links, out_links;
    std::vector<Step> steps;
    std::vector<std::unique_ptr<DevBuf>> scratch;  // [C x max_samples] intermediates crossing steps
    std::vector<std::unique_ptr<DevBuf>> pc_tabs;  // per step: its per-channel parameter table on the device (or null)
    // host-memory mode staging
    std::vector<std::unique_ptr<DevBuf>> h_in, h_out;
    cudaStream_t s_h2d = nullptr, s_cmp = nullptr, s_d2h = nullptr;
    std::vector<cudaEvent_t> ev_pool;
    int64_t last_launches = 0;
    int force_G = 0;
    int dev_chunks = 1;      // device-pointer mode: channel chunks run on separate streams so kernels of different steps overlap
    std::vector<cudaStream_t> chunk_streams;
    std::vector<cudaEvent_t> chunk_events;
    bool raw_ports = false;  // sub-engine of dspb_node_process: ports carry pre-averaged buffers, no fan-in division
    struct NodeEngine { dspb_engine* e = nullptr; uint32_t present_mask = 0; };
    std::map<int64_t, NodeEngine> node_engines;
    bool prof_on = false;
    struct ProfRec { int step; cudaEvent_t a, b; };
    std::vector<ProfRec> prof;
    bool plan_only = false;
    bool host_inflight = false;   // a DSPB_MEM_HOST_ASYNC call may still be running on the internal streams
    int64_t host_last_n = 0;
    // playback-side sample-rate converter (dspb_resample_dup_stereo): dasp Converter state shared by all channels + the
    // last 16 pushed frames of every channel
    struct Resampler {
        double target_hz = 0.0, value = 0.0;   // Converter::interpolation_value
        int idx = 0;                           // Sinc::idx (saturates at depth = 8)
        int cur = 0;
        DevBuf hist[2];                        // [C x 16] f32, double-buffered
        DevBuf meta, w;                        // per-call plan on the device
        size_t cap = 0;
    } rs;

    int find(int64_t id) const {
        for (size_t i = 0; i < nodes.size(); i++)
            if (nodes[i]->id == id) return (int)i;
        return -1;
    }
    ~dspb_engine() {
        for (auto& kv : node_engines) delete kv.second.e;
        for (auto& r : prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
        for (auto e : ev_pool) cudaEventDestroy(e);
        for (auto e : chunk_events) cudaEventDestroy(e);
        for (auto st : chunk_streams) cudaStreamDestroy(st);
        if (s_h2d) cudaStreamDestroy(s_h2d);
        if (s_cmp) cudaStreamDestroy(s_cmp);
        if (s_d2h) cudaStreamDestroy(s_d2h);
    }
};

namespace {

int param_index(const NodeType& nt, const char* name) {
    for (size_t i = 0; i < nt.params.size(); i++)
        if (!strcmp(nt.params[i].name, name)) return (int)i;
    return -1;
}
int port_index(const std::vector<const char*>& v, const char* name) {
    for (size_t i = 0; i < v.size(); i++)
        if (!strcmp(v[i], name)) return (int)i;
    return -1;
}

int64_t round_up(int64_t n, int64_t g) { return g <= 1 ? n : (n + g - 1) / g * g; }

// Host side of exact_math.cuh's div_const.  The 3-instruction sequence is NOT exact for every divisor
// (measured: 0.3, 29.99, ... have millions of wrong quotients), so a divisor gets the fast path only
// after the device has enumerated all 2^32 dividends against IEEE division with zero mismatches
// (verify_const_div, a few ms, cached per process).  Everything else takes __fdiv_rn.
bool div_const_ok(float b, bool plan_only) {
    if (!(b > 0.0f) || !std::isfinite(b) || b < 1e-30f || b > 1e30f) return false;
    if (plan_only) return true;  // nothing runs in planning-only mode; show the optimistic schedule
    // the verdict is IEEE arithmetic, identical on every device: one process-wide cache, serialised (engines on
    // different threads compile concurrently; the enumeration itself runs on the calling engine's device)
    static std::mutex mu;
    static std::map<uint32_t, bool> cache;
    uint32_t bits;
    memcpy(&bits, &b, 4);
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(bits);
    if (it != cache.end()) return it->second;
    bool ok = false;
    unsigned long long mism = 1;
    if (verify_const_div(b, 1.0f / b, &mism) == 0) ok = mism == 0;
    cache[bits] = ok;
    return ok;
}
void set_const_div(Op& op, int p_b, int p_r, float b, bool plan_only) {
    const bool ok = div_const_ok(b, plan_only);
    op.p[p_b] = b;
    op.p[p_r] = ok ? 1.0f / b : 0.0f;
    op.pad = ok ? 1 : 0;
}

// ---- opt-in time-parallel recurrences (dspb_config::iir_mode = 1) ---------------------------------------------------
// ScanTab for y[n] = p[n] - a1 y[n-1] - a2 y[n-2]: powers of A = [[-a1, -a2], [1, 0]] in f64, rounded to f32.
ScanTab make_scan_tab(float a1, float a2) {
    ScanTab t;
    memset(&t, 0, sizeof t);
    t.a1 = a1;
    t.a2 = a2;
    double M[4] = {-(double)a1, -(double)a2, 1.0, 0.0}, R[4] = {1, 0, 0, 1};
    auto mul2 = [](const double* a, const double* b, double* o) {
        double r[4] = {a[0] * b[0] + a[1] * b[2], a[0] * b[1] + a[1] * b[3], a[2] * b[0] + a[3] * b[2], a[2] * b[1] + a[3] * b[3]};
        memcpy(o, r, sizeof r);
    };
    for (int i = 0; i < 3; i++) mul2(M, M, M);  // A^8
    memcpy(R, M, sizeof R);
    for (int i = 0; i < 6; i++) {               // A^(8 * 2^i)
        for (int k = 0; k < 4; k++) t.P[i][k] = R[k];
        mul2(R, R, R);
    }
    return t;
}
// Verdict for one coefficient set: scan mode only if the device probe (fused_chain.cu measure_scan_error) stays below
// half of the 1e-5 parity bar.  Cached per process (IEEE arithmetic: the same on every device).
constexpr float kScanGate = 5e-6f;  // half of the 1e-5 parity bar: the probe sees ONE filter, a graph may chain several
bool scan_qualifies(const Op& op, ScanTab& tab, bool plan_only) {
    if (plan_only) { tab.probe_err = 0.0f; return true; }  // nothing runs in planning mode: show the optimistic schedule
    static std::mutex mu;
    static std::map<std::vector<uint32_t>, float> cache;
    std::vector<uint32_t> key{op.code};
    for (int i = 0; i < 4; i++) { uint32_t b; memcpy(&b, &op.p[i], 4); key.push_back(b); }
    { uint32_t b; memcpy(&b, &op.a2, 4); key.push_back(b); }
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    float err = 1.0f;
    if (it != cache.end()) err = it->second;
    else {
        if (measure_scan_error(op, tab, &err) != 0) err = 1.0f;
        cache[key] = err;
    }
    tab.probe_err = err;
    return err <= kScanGate;
}

// Reverb::refresh_seconds, nodes/reverb.rs:55-71.  Integer work: must match the reference exactly.
int64_t reverb_delay(float seconds, int sample_rate, int granule) {
    float prod = seconds * (float)sample_rate;
    int64_t num = 0;  // `as usize`: NaN/negative -> 0, truncating, saturating
    if (prod > 0.0f) num = prod >= 9.0e18f ? (INT64_MAX / 2) : (int64_t)prod;
    num = std::max<int64_t>(num, 128);
    return round_up(num, granule);
}

// BiQuad::regenerate_filter, nodes/biquad.rs:62-76 (f32 divisions): sliders a0 a1 a2 b0 b1 b2 -> bq = b0 b1 b2 a1 a2
void biquad_coefs(const float* f, float* bq) {
    const float a0 = f[0];
    bq[3] = f[1] / a0;  // a1
    bq[4] = f[2] / a0;  // a2
    bq[0] = f[3] / a0;  // b0
    bq[1] = f[4] / a0;  // b1
    bq[2] = f[5] / a0;  // b2
}
void biquad_regenerate(Node& n) { biquad_coefs(n.f32.data(), n.bq); }
float calc_gain(float frames) { return frames == 0.0f ? 0.0f : std::exp(-1.0f / frames); }  // dasp calc_gain

// The values op `which` of a node of type `type` reads, in plan.h op_pc_cols order (p[0], p[1], ...; the biquad's a2 last),
// from the node's slider values f (ParamDef order) with the reference's host arithmetic.  Both the shared Op fields and every
// row of a per-channel table come from here.  which: 0, or the gate's second op (1: the compare).
void op_values(int type, int which, const float* f, float* v) {
    switch (type) {
        case T_GAIN: case T_DISTORT: case T_MIX: v[0] = f[0]; break;
        case T_OVERDRIVE: v[0] = f[0]; v[1] = f[1]; v[2] = f[2]; break;
        case T_CHEBY:  // level.tanh(): libm tanhf, as the reference host would
            v[0] = f[0]; v[1] = f[1]; v[2] = std::tanh(f[0]); v[3] = std::tanh(f[1]); break;
        case T_BIQUAD: biquad_coefs(f, v); break;
        case T_LOWPASS: case T_HIGHPASS: v[0] = f[0]; v[1] = 1.0f - f[0]; break;
        case T_REVERB: v[0] = f[1]; break;  // decay (seconds sets the ring length: shared)
        case T_ENVELOPE: v[0] = calc_gain(f[0]); v[1] = calc_gain(f[1]); break;
        case T_SIGGEN: v[0] = f[0]; v[1] = f[1]; break;
        case T_GATE:
            if (which == 0) { v[0] = calc_gain(f[1]); v[1] = calc_gain(f[2]); }
            else v[0] = f[0];
            break;
    }
}
// op_values into the shared Op fields
void set_op_values(Op& op, const float* v) {
    const int n = op_pc_cols(op.code);
    for (int k = 0; k < n && k < 4; k++) op.p[k] = v[k];
    if (n > 4) op.a2 = v[4];
}

bool is_stateful(int type) {
    return type == T_BIQUAD || type == T_LOWPASS || type == T_HIGHPASS || type == T_ENVELOPE || type == T_SIGGEN || type == T_GATE;
}

int clear_node_state(dspb_engine* e, Node& n) {
    if (n.state.p) CUDA_TRY(cudaMemset(n.state.p, 0, n.state.bytes));
    if (n.ring.p) CUDA_TRY(cudaMemset(n.ring.p, 0, n.ring.bytes));
    n.pos = 0;
    if (n.U.p) CUDA_TRY(cudaMemset(n.U.p, 0, n.U.bytes));
    n.started = 0;
    n.u_pos = 0;
    n.fdl_valid = false;
    n.upc_ctr = 0;
    (void)e;
    return DSPB_OK;
}

// ---- lowering ------------------------------------------------------------------------------------------------
// A value is what one node output port carries for the current tile.
struct Value {
    enum Where { NONE, VREG, GLOBAL, ZERO } where = NONE;
    int id = -1;      // virtual vreg id or prog buffer kind key
    int bind_kind = 0, bind_idx = 0;  // for GLOBAL
    int def_step = -1;
};

struct Lowerer {
    dspb_engine& e;
    std::vector<Step> steps;
    Step cur{};
    std::vector<Op> ops;           // ops of the current fused step (virtual vreg ids)
    std::vector<std::string> txt;
    int next_vreg = 0;
    int n_scratch = 0;
    std::map<std::pair<int, int>, Value> values;  // (node, out port) -> value
    std::map<std::pair<int, int>, int> use_step;  // last step that uses the value
    std::vector<int> node_step;                   // step index in which a node's ops are emitted
    std::set<int> fused_sinks;                    // output terminals written directly by a FIR step
    std::vector<ScanTab> scan_tabs;               // scan tables of the current fused step (Op::mode = index + 1)
    std::vector<std::vector<float>> pc_cols;      // per-channel table of the current fused step, column by column
    std::string err;
    // A graph region between two FIR nodes normally becomes ONE fused segment.  When it exceeds what one Program holds
    // (ops, global buffers, states, rings, virtual vregs, shared memory) the segment is closed in front of a node and the
    // rest starts a new one; values that cross the cut travel through global scratch like values that cross a FIR step.
    // lower_graph() retries with one more cut until every segment fits.
    std::set<int> split_before;                   // nodes in front of which the open segment is closed
    int want_split = -1;                          // set with `err` when one more cut would help
    std::vector<int> cur_nodes;                   // nodes that emitted ops into the open segment
    int cur_node = -1;

    explicit Lowerer(dspb_engine& en) : e(en) {}

    // A per-segment limit was hit while lowering `cur_node`: everything before it fitted, so cut in front of it.
    void overflow(const char* what) {
        if (!err.empty()) return;
        err = what;
        if (!cur_nodes.empty() && cur_nodes.front() != cur_node) want_split = cur_node;
    }
    int buf_slot(int kind, int idx) {
        for (size_t i = 0; i < cur.binds.size(); i++)
            if (cur.binds[i].kind == kind && cur.binds[i].idx == idx) return (int)i;
        if ((int)cur.binds.size() >= kMaxBufs) { overflow("segment uses too many global buffers"); return 0; }
        cur.binds.push_back({kind, idx});
        return (int)cur.binds.size() - 1;
    }
    int new_vreg() {
        if (next_vreg >= 0xFF) { overflow("segment has too many intermediate values"); return 0; }  // 0xFF names the accumulator
        return next_vreg++;
    }
    void emit(Op op, const std::string& s) {
        // bound on the UNFOLDED listing only (finish_vregs folds the fan-in prologues, typically 2-3 ops into one); the
        // limit that matters, kMaxOps of the folded Program, is checked in close_fused
        if ((int)ops.size() >= 4 * kMaxOps) { overflow("segment has too many ops"); return; }
        ops.push_back(op);
        txt.push_back(s);
    }
    static Op mk(uint8_t code) {
        Op o;
        memset(&o, 0, sizeof o);
        o.code = code;
        return o;
    }
    // acc = value (first term: 0.0 + v) or acc += value
    void emit_term(const Value& v, bool first, const std::string& what) {
        if (e.raw_ports && first && (v.where == Value::VREG || v.where == Value::GLOBAL)) {  // pre-averaged buffer: plain copy
            Op o = mk(v.where == Value::VREG ? OP_COPYV : OP_COPYG);
            if (v.where == Value::VREG) o.vreg = (uint8_t)v.id;
            else o.buf = (uint8_t)buf_slot(v.bind_kind, v.bind_idx);
            emit(o, "acc = port buffer            ; " + what);
            return;
        }
        if (v.where == Value::ZERO || v.where == Value::NONE) {
            if (first) {
                emit(mk(OP_ZERO), "acc = 0                      ; " + what);
            } else {  // acc + 0.0 only turns a -0.0 sum into +0.0; kept so that the sign of a zero matches node.rs:181-183
                Op z = mk(OP_LOADV);
                z.vreg = 0xFF;
                emit(z, "acc = 0.0 + acc              ; " + what + " (all-zero link)");
            }
            return;
        }
        if (v.where == Value::VREG) {
            Op o = mk(first ? OP_LOADV : OP_ADDV);
            o.vreg = (uint8_t)v.id;
            emit(o, std::string(first ? "acc = 0.0 + v" : "acc += v") + std::to_string(v.id) + "           ; " + what);
        } else {
            Op o = mk(first ? OP_LOADG : OP_ADDG);
            o.buf = (uint8_t)buf_slot(v.bind_kind, v.bind_idx);
            emit(o, std::string(first ? "acc = 0.0 + G" : "acc += G") + std::to_string(o.buf) + "           ; " + what);
        }
    }
    // collect_and_average (node.rs:162-194) for input port p of node ni; result in acc.
    bool emit_avg(int ni, int p) {
        const auto& ls = e.in_links[ni][p];
        if (ls.empty()) {
            emit(mk(OP_ZERO), "acc = 0                      ; unconnected port (0/0.0001)");
            return false;
        }
        float nf = 0.0001f;
        bool first = true;
        for (int l : ls) {
            const Link& k = e.links[l];
            nf += 1.0f;
            emit_term(values[{k.src, k.sport}], first,
                      std::string("link ") + kNodeTypes[e.nodes[k.src]->type].cfg_name + "#" + std::to_string(e.nodes[k.src]->id));
            first = false;
        }
        if (e.raw_ports) return true;  // dspb_node_process: inputs are already averaged (node.rs:217-222)
        Op d = mk(OP_DIVC);
        set_const_div(d, 0, 1, nf, e.plan_only);
        char b[96];
        snprintf(b, sizeof b, "acc /= %.9g           ; fan-in average of %zu link(s)", nf, ls.size());
        emit(d, b);
        return true;
    }
    // Scratch buffers ([C x max_samples] each) are reused: a buffer whose last reader ran in an EARLIER step than the one
    // that defines the new value is free (steps are kernels in stream order; within one step a tile-by-tile writer could
    // overtake a reader of the same buffer, hence strictly earlier).
    std::vector<int> scratch_last_read;           // per scratch buffer: the last logical step that reads its current value
    int alloc_scratch(int def_step, int last_use_step) {
        for (size_t i = 0; i < scratch_last_read.size(); i++)
            if (scratch_last_read[i] < def_step) { scratch_last_read[i] = last_use_step; return (int)i; }
        scratch_last_read.push_back(last_use_step);
        n_scratch = (int)scratch_last_read.size();
        return n_scratch - 1;
    }
    int temp_save(const std::string& what) {
        int id = new_vreg();
        Op o = mk(OP_SAVEV);
        o.vreg = (uint8_t)id;
        emit(o, "v" + std::to_string(id) + " = acc                    ; " + what);
        return id;
    }
    // Per-channel parameters of the op node `ni` is about to emit: when one of `fields` (a bitmask over its ParamDef indices)
    // holds per-channel values that no linked control port overrides (lib.rs:122-161), the op gets op_pc_cols columns in
    // this segment's table, row c = op_values of channel c's sliders -- the function that gave the op its shared values.
    // Returns the listing marker ("" = shared parameters).
    std::string per_channel(Op& op, int ni, int which, unsigned fields) {
        const Node& nd = *e.nodes[ni];
        const NodeType& nt = kNodeTypes[nd.type];
        std::string names;
        for (size_t p = 0; p < nt.params.size(); p++) {
            if (!((fields >> p) & 1) || nd.f32_pc[p].empty()) continue;
            const int port = nt.params[p].ctl_port;
            if (port >= 0 && !e.in_links[ni][port].empty()) continue;
            names += std::string(names.empty() ? "" : ",") + nt.params[p].name;
        }
        if (names.empty()) return "";
        const int k = op_pc_cols(op.code), col = (int)pc_cols.size();
        if (col + k > kMaxPcCols) { overflow("segment has more per-channel parameters than one table holds"); return ""; }
        const int C = e.cfg.channels;
        pc_cols.resize(col + k, std::vector<float>(C));
        std::vector<float> f(nd.f32);
        float v[5] = {0, 0, 0, 0, 0};
        for (int c = 0; c < C; c++) {
            for (size_t p = 0; p < f.size(); p++) f[p] = nd.f32_pc[p].empty() ? nd.f32[p] : nd.f32_pc[p][c];
            op_values(nd.type, which, f.data(), v);
            for (int q = 0; q < k; q++) pc_cols[col + q][c] = v[q];
        }
        op.pad = (uint8_t)((op.pad & 1) | ((col + 1) << 1));
        return " per-channel[" + names + "]";
    }
    void close_fused();
    int lower();
    int finish_vregs(Step& st, std::vector<Op>& o, std::vector<std::string>& t);
};

// Ops whose `vreg` field names a shared-memory vreg they READ (one predicate for liveness, remapping and the kernels'
// op_reads_vreg: a code missing from one of those lists reads a slot that was never allocated).
bool reads_vreg_operand(int code) { return op_reads_vreg_field(code); }

// Peephole + vreg allocation for one fused step.  Virtual vregs -> shared-memory slots by liveness.
int Lowerer::finish_vregs(Step& st, std::vector<Op>& o, std::vector<std::string>& t) {
    auto reads = [](const Op& op, int v) {
        if (reads_vreg_operand(op.code) && op.vreg == v) return true;
        for (int i = 0; i < 3; i++)
            if ((op.pflags & (1 << i)) && op.pv[i] == v) return true;
        return false;
    };
    // peephole: "vK = acc ; acc = 0.0 + vK" with vK used nowhere else -> "acc = 0.0 + acc"
    for (size_t i = 0; i + 1 < o.size();) {
        if (o[i].code == OP_SAVEV && o[i + 1].code == OP_LOADV && o[i + 1].vreg == o[i].vreg) {
            int v = o[i].vreg, uses = 0;
            for (size_t k = 0; k < o.size(); k++)
                if (reads(o[k], v)) uses++;
            if (uses == 1) {
                Op z = mk(OP_LOADV);
                z.vreg = 0xFF;  // acc itself
                o[i] = z;
                t[i] = "acc = 0.0 + acc              ; value stays in registers";
                o.erase(o.begin() + i + 1);
                t.erase(t.begin() + i + 1);
                continue;
            }
        }
        i++;
    }
    // fold the fan-in prologue ("acc = 0.0 + acc", "acc /= nf") into the op that consumes it
    auto consumes_acc = [](int c) {
        return c == OP_GAIN || c == OP_DISTORT || c == OP_OVERDRIVE || c == OP_CHEBY || c == OP_COMB || c == OP_BIQUAD ||
               c == OP_LP1 || c == OP_HP1 || c == OP_ENVELOPE || c == OP_STOREG || c == OP_SAVEV || c == OP_MODMAP ||
               c == OP_ADD || c == OP_MIX;
    };
    for (size_t i = 0; i < o.size(); i++) {
        int pre = 0;
        size_t k = i;
        if (o[k].code == OP_LOADV && o[k].vreg == 0xFF) { pre |= 1; k++; }
        if (k < o.size() && o[k].code == OP_DIVC) {
            pre |= 2 | (o[k].pad ? 4 : 0);
            const float nf = o[k].p[0], r = o[k].p[1];
            k++;
            Op host;
            std::string host_txt;
            if (k < o.size() && consumes_acc(o[k].code) && o[k].pre == 0) { host = o[k]; host_txt = t[k]; k++; }
            else { host = mk(OP_NOP); host_txt = "(fan-in prologue only)"; }
            host.pre = (uint8_t)pre;
            host.p[4] = nf;
            host.p[5] = r;
            char b[64];
            snprintf(b, sizeof b, "[%sacc /= %.9g] ", (pre & 1) ? "acc = 0.0 + acc; " : "", nf);
            o[i] = host;
            t[i] = std::string(b) + host_txt;
            o.erase(o.begin() + i + 1, o.begin() + k);
            t.erase(t.begin() + i + 1, t.begin() + k);
        } else if (pre) {  // "acc = 0.0 + acc" without a division cannot occur; keep it as a NOP prologue
            Op host = mk(OP_NOP);
            host.pre = 1;
            o[i] = host;
        }
    }
    // liveness
    std::map<int, std::pair<int, int>> live;  // virtual id -> [def, last use]
    for (size_t i = 0; i < o.size(); i++) {
        if (o[i].code == OP_SAVEV) {
            if (!live.count(o[i].vreg)) live[o[i].vreg] = {(int)i, (int)i};
        }
        for (auto& kv : live)
            if (reads(o[i], kv.first)) kv.second.second = (int)i;
    }
    std::map<int, int> phys;
    std::vector<int> slot_free_at;  // op index after which the slot is free
    for (size_t i = 0; i < o.size(); i++) {
        if (o[i].code != OP_SAVEV || phys.count(o[i].vreg)) continue;
        int v = o[i].vreg, s = -1;
        for (size_t k = 0; k < slot_free_at.size(); k++)
            if (slot_free_at[k] < (int)i) { s = (int)k; break; }
        if (s < 0) { slot_free_at.push_back(0); s = (int)slot_free_at.size() - 1; }
        slot_free_at[s] = live[v].second;
        phys[v] = s;
    }
    for (auto& op : o) {
        if ((reads_vreg_operand(op.code) || op.code == OP_SAVEV) && op.vreg != 0xFF)
            op.vreg = (uint8_t)phys[op.vreg];
        for (int i = 0; i < 3; i++)
            if (op.pflags & (1 << i)) op.pv[i] = (uint8_t)phys[op.pv[i]];
    }
    st.prog.n_vregs = (int)slot_free_at.size();
    return DSPB_OK;
}

void Lowerer::close_fused() {
    if (ops.empty() || !err.empty()) { cur = Step(); ops.clear(); txt.clear(); cur_nodes.clear(); pc_cols.clear(); next_vreg = 0; return; }
    cur.kind = STEP_FUSED;
    finish_vregs(cur, ops, txt);
    if ((int)ops.size() > kMaxOps - 1) {  // the folded program does not fit: cut the segment in the middle and lower again
        err = "segment has too many ops";
        if (cur_nodes.size() >= 2) want_split = cur_nodes[cur_nodes.size() / 2];
        return;
    }
    cur.nodes = cur_nodes;
    cur_nodes.clear();
    Program& P = cur.prog;
    P.n_ops = (int)ops.size();
    P.needs_tile = 0;
    int64_t min_ring = INT64_MAX;
    bool has_rec = false, has_scan = false;
    auto is_lin_rec = [](int c) { return c == OP_BIQUAD || c == OP_LP1 || c == OP_HP1; };
    // Scan mode pays only when NO sequential recurrence is left in the segment (one exact chain bounds the kernel anyway,
    // and the pipelined warp-specialised kernels only take exact recurrences): all or nothing per segment.
    bool any_exact = false;
    for (auto& o : ops) any_exact = any_exact || o.code == OP_ENVELOPE || (is_lin_rec(o.code) && o.mode == 0);
    if (any_exact)
        for (size_t i = 0; i < ops.size(); i++)
            if (is_lin_rec(ops[i].code) && ops[i].mode != 0) {
                ops[i].mode = 0;
                txt[i] += "  [exact after all: another recurrence of this segment stays sequential]";
            }
    P.n_scan = 0;
    for (int i = 0; i < P.n_ops; i++) {
        P.ops[i] = ops[i];
        const int c = ops[i].code;
        if (is_lin_rec(c) && ops[i].mode != 0) {
            has_scan = true;
            P.scan[P.n_scan] = scan_tabs[ops[i].mode - 1];
            P.ops[i].mode = (uint8_t)(++P.n_scan);
        } else if (c == OP_BIQUAD || c == OP_LP1 || c == OP_HP1 || c == OP_ENVELOPE) {
            P.needs_tile = 1;
            has_rec = true;
        }
        if (c == OP_COMB) min_ring = std::min(min_ring, e.nodes[cur.ring_nodes[ops[i].aux & 0xff]]->D);
    }
    scan_tabs.clear();
    cur.pc_k = (int)pc_cols.size();
    if (cur.pc_k) {  // row-major [C x K]: row = absolute channel
        const int C = e.cfg.channels;
        cur.pc_host.assign((size_t)C * cur.pc_k, 0.0f);
        for (int k = 0; k < cur.pc_k; k++)
            for (int c = 0; c < C; c++) cur.pc_host[(size_t)c * cur.pc_k + k] = pc_cols[k][c];
    }
    pc_cols.clear();
    // Tile geometry: G channels x S = 4096/G samples per CTA.  S may not exceed the shortest comb
    // delay (a tile must never read a ring slot it writes itself); recurrences run lane = channel,
    // so they want G large, but the grid wants >= ~1.7 CTAs per SM (148 SMs).
    const int C = e.cfg.channels;
    int G = 1;
    if (has_rec) {
        if (C <= 2048 && P.n_vregs == 0 && P.n_ops <= 8) {
            // few channels per SM and a light chain: the kernel is bound by the sequential recurrence chain, not by
            // elementwise work (measured: heavier graphs such as config 5's 17-op segment with shared-memory vregs are
            // better off with 256 CTAs at two per SM).
            // One CTA per SM in one wave (<= 8 GPCs x 16 SMs = 128 CTAs) lets the warp-specialised kernel give the
            // recurrence warp an SM sub-partition of its own (fused_chain.cu, XR layout: 14 instead of ~35 cycles per step).
            // (Fatter CTAs with shorter tiles -- G = 8 for 256 channels -- were measured no faster: 0.155 vs 0.141 ms.)
            while (G < 32 && (C + G - 1) / G > 128) G <<= 1;
        } else {
            G = 32;
            while (G > 1 && (C + G - 1) / G < 256) G >>= 1;
        }
    }
    if (has_scan && !has_rec) {
        // every thread works time-parallel: fill the machine with CTAs (about two per SM), channels per CTA as needed
        G = 1;
        while (G < 32 && (C + G - 1) / G > 296) G <<= 1;
    }
    while ((int64_t)kTile / G > min_ring && G < 32) G <<= 1;
    if (e.force_G) G = e.force_G;
    if ((int64_t)kTile / G > min_ring) G = 32;
    cur.G = G;
    // Register prefetch (one tile ahead): slot 0 = the first streamed global read, slot 1 = the first comb ring
    // whose geometry allows it (16-aligned slots; the next tile must not read what this tile writes: D >= 2S).
    const int S = kTile / G;
    P.n_prefetch = 0;
    for (int k = 0; k < kMaxPrefetch; k++) P.pf_buf[k] = P.pf_ring[k] = -1;
    static const bool in_prefetch = !(getenv("DSPB_IN_PREFETCH") && atoi(getenv("DSPB_IN_PREFETCH")) == 0);
    for (int i = 0; i < P.n_ops && in_prefetch; i++)
        if (P.ops[i].code == OP_LOADG) {
            // A buffer this very program stores earlier (a source value spilled for a later step AND consumed again in
            // this one) must not be read one tile ahead: the prefetch would see the previous call's scratch.
            bool stored_here = false;
            for (int k = 0; k < i; k++) stored_here = stored_here || (P.ops[k].code == OP_STOREG && P.ops[k].buf == P.ops[i].buf);
            if (stored_here) continue;
            P.pf_buf[0] = P.ops[i].buf;
            P.ops[i].aux = 1;
            P.n_prefetch++;
            break;
        }
    P.st_buf = -1;
    for (int i = 0; i < P.n_ops; i++)
        if (P.ops[i].code == OP_STOREG) {
            P.st_buf = P.ops[i].buf;
            P.ops[i].aux = 1;
            break;
        }
    static const bool ring_prefetch = !(getenv("DSPB_RING_PREFETCH") && atoi(getenv("DSPB_RING_PREFETCH")) == 0);
    for (int i = 0; i < P.n_ops && ring_prefetch; i++)
        if (P.ops[i].code == OP_COMB) {
            const Node& rn = *e.nodes[cur.ring_nodes[P.ops[i].aux & 0xff]];
            if ((rn.D & (kChunk - 1)) == 0 && rn.D >= 2 * (int64_t)S) {
                P.pf_ring[1] = (int16_t)(P.ops[i].aux & 0xff);
                P.ops[i].aux = (uint16_t)((P.ops[i].aux & 0xff) | (1 << 8));
                P.n_prefetch++;
            }
            break;
        }
    int alg = 0;  // ALGORITHMIC bytes per channel-sample of this kernel: 4 per global f32 read/write, 8 per ring
    for (int i = 0; i < P.n_ops; i++) {
        const int c = P.ops[i].code;
        if (c == OP_LOADG || c == OP_ADDG || c == OP_COPYG || c == OP_STOREG) alg += 4;
        if (c == OP_COMB) alg += 8;
    }
    char hdr[200];
    snprintf(hdr, sizeof hdr, "fused segment: G=%d channels x S=%d samples per CTA, %d ops, %d smem vregs, %d prefetch slots, alg_bytes=%d\n", G,
             S, P.n_ops, P.n_vregs, P.n_prefetch, alg);
    cur.text = hdr;
    if (cur.pc_k) {
        cur.text.pop_back();
        cur.text += ", per-channel table " + std::to_string(cur.pc_k) + " column(s)\n";
    }
    for (size_t i = 0; i < txt.size(); i++) cur.text += "    " + txt[i] + "\n";
    {   // the lowered program as the kernel sees it (physical shared-memory slots, prefetch flags): "op<code>:..." per op
        std::string m = "    lowered:";
        for (int i = 0; i < P.n_ops; i++) {
            const Op& o = P.ops[i];
            char b[96];
            int k = snprintf(b, sizeof b, " %d", (int)o.code);
            if (op_reads_vreg_field(o.code) || o.code == OP_SAVEV) k += snprintf(b + k, sizeof b - k, ":v%d", o.vreg == 0xFF ? -1 : (int)o.vreg);
            for (int q = 0; q < 3; q++)
                if (o.pflags & (1 << q)) k += snprintf(b + k, sizeof b - k, ":p%d=v%d", q, (int)o.pv[q]);
            if (op_pc_col(o) >= 0) k += snprintf(b + k, sizeof b - k, ":c%d", op_pc_col(o));  // per-channel table column
            if (o.code == OP_LOADG || o.code == OP_ADDG || o.code == OP_COPYG || o.code == OP_STOREG) k += snprintf(b + k, sizeof b - k, ":g%d%s", (int)o.buf, o.aux ? "*" : "");
            m += b;
        }
        cur.text += m + "\n";
        m = "    buffers:";   // what each g<slot> is bound to at launch: terminals, scratch between segments, a FIR node's input ring / output
        for (size_t i = 0; i < cur.binds.size(); i++) {
            static const char* kKind[] = {"in", "out", "scratch", "firU#", "firY#"};
            const int kind = cur.binds[i].kind, idx = cur.binds[i].idx;
            m += " g" + std::to_string(i) + "=" + kKind[kind] + std::to_string(kind >= 3 ? (long long)e.nodes[idx]->id : (long long)idx);
        }
        cur.text += m + "\n";
    }
    steps.push_back(cur);
    cur = Step();
    ops.clear();
    txt.clear();
    next_vreg = 0;
}

int Lowerer::lower() {
    const int N = (int)e.nodes.size();
    // step assignment: ops of a node are emitted in the fused step open when it is visited; a Fir
    // node closes that step (its input average is stored there) and gets its own step.
    node_step.assign(N, 0);
    {
        int s = 0;
        for (int ni : e.order) {
            if (split_before.count(ni)) s += 1;      // a cut: this node opens a new fused step
            node_step[ni] = s;
            if (e.nodes[ni]->type == T_FIR) s += 2;  // fused step s, FIR step s+1, next fused s+2
        }
        // NOTE: empty fused steps are still numbered; only relative order matters here.
        for (int ni : e.order)
            for (size_t p = 0; p < e.in_links[ni].size(); p++)
                for (int l : e.in_links[ni][p]) {
                    auto key = std::make_pair(e.links[l].src, e.links[l].sport);
                    use_step[key] = std::max(use_step.count(key) ? use_step[key] : -1, node_step[ni]);
                }
    }
    int state_slot = 0;
    // `steps.size()` is not the step number used above (empty steps are dropped), so track it separately.
    int logical_step = 0;
    auto def_step_of = [&](int) { return logical_step; };
    (void)def_step_of;
    for (int ni : e.order) {
        Node& nd = *e.nodes[ni];
        const NodeType& nt = kNodeTypes[nd.type];
        const std::string tag = std::string(nt.cfg_name) + "#" + std::to_string(nd.id);
        if (split_before.count(ni)) {
            close_fused();
            if (!err.empty()) return DSPB_ERR_INVALID;
            logical_step += 1;
            state_slot = 0;
        }
        cur_node = ni;
        const size_t ops_before = ops.size();
        if (nd.type != T_FIR) cur_nodes.push_back(ni);   // dropped again below if the node emits nothing
        auto out_value = [&](int port) {
            Value v;
            auto key = std::make_pair(ni, port);
            const int us = use_step.count(key) ? use_step[key] : -1;
            if (us < 0) { v.where = Value::NONE; return v; }
            if (us != logical_step) {
                v.where = Value::GLOBAL;
                v.bind_kind = 2;
                v.bind_idx = alloc_scratch(logical_step, us);
                Op o = mk(OP_STOREG);
                o.buf = (uint8_t)buf_slot(2, v.bind_idx);
                emit(o, "G" + std::to_string(o.buf) + " = acc                    ; " + tag + " (used in a later step)");
            } else {
                v.where = Value::VREG;
                v.id = next_vreg++;
                Op o = mk(OP_SAVEV);
                o.vreg = (uint8_t)v.id;
                emit(o, "v" + std::to_string(v.id) + " = acc                    ; " + tag + ".out");
            }
            return v;
        };
        auto ctl_param = [&](Op& op, int which, int pidx) {
            // derive helper <field>_input (lib.rs:122-161): connected control port overrides the scalar
            const ParamDef& pd = nt.params[pidx];
            op.p[which] = nd.f32[pidx];
            if (pd.ctl_port >= 0 && !e.in_links[ni][pd.ctl_port].empty()) {
                emit_avg(ni, pd.ctl_port);
                Op m = mk(OP_MODMAP);
                m.p[0] = pd.lo;
                m.p[1] = pd.hi;
                emit(m, std::string("acc = map(acc, ") + std::to_string(pd.lo) + ", " + std::to_string(pd.hi) + ") ; " + tag + "." + pd.name + " control port");
                int v = temp_save(tag + "." + pd.name);
                op.pflags |= (1 << which);
                op.pv[which] = (uint8_t)v;
            }
        };
        auto alloc_state = [&](Op& op) -> int {
            if (state_slot >= kMaxStates) { overflow("too many stateful nodes in one segment"); return -1; }
            op.aux = (uint16_t)state_slot;
            cur.prog.states[state_slot] = nd.state.p;
            return state_slot++;
        };
        switch (nd.type) {
            case T_INPUT: {
                int t = (int)(std::find(e.in_terms.begin(), e.in_terms.end(), ni) - e.in_terms.begin());
                Value v;
                v.where = Value::GLOBAL;
                v.bind_kind = 0;
                v.bind_idx = t;
                values[{ni, 0}] = v;
            } break;
            case T_OUTPUT: {
                if (fused_sinks.count(ni)) break;
                int t = (int)(std::find(e.out_terms.begin(), e.out_terms.end(), ni) - e.out_terms.begin());
                emit_avg(ni, 0);  // nodes/output.rs:223
                Op o = mk(OP_STOREG);
                o.buf = (uint8_t)buf_slot(1, t);
                emit(o, "G" + std::to_string(o.buf) + " = acc                    ; output terminal " + std::to_string(t));
            } break;
            case T_FIR: {
                cur_nodes.push_back(ni);
                emit_avg(ni, 0);
                Op o = mk(OP_STOREG);
                o.buf = (uint8_t)buf_slot(3, ni);
                emit(o, "G" + std::to_string(o.buf) + " = acc                    ; " + tag + " input (+history)");
                if (!err.empty()) return DSPB_ERR_INVALID;
                close_fused();
                if (!err.empty()) return DSPB_ERR_INVALID;
                Step fs;
                fs.kind = STEP_FIR;
                fs.fir_node = ni;
                // A sink fed only by this node: fold its fan-in average into the FIR epilogue
                if (e.out_links[ni][0].size() == 1 && !e.raw_ports) {
                    const int dst = e.links[e.out_links[ni][0][0]].dst;
                    if (e.nodes[dst]->type == T_OUTPUT && e.in_links[dst][0].size() == 1) {
                        fs.fir_out_term = (int)(std::find(e.out_terms.begin(), e.out_terms.end(), dst) - e.out_terms.begin());
                        fs.fir_post_nf = 0.0001f + 1.0f;
                        fused_sinks.insert(dst);
                    }
                }
                char b[200];
                if (e.cfg.fir_mode == FIR_FFT || e.cfg.fir_mode == FIR_FFT_PACKED)
                    snprintf(b, sizeof b, "fir step: %s, %zu taps, overlap-save FFT 2^%d%s, two channels per transform, alg_bytes=8\n", tag.c_str(),
                             nd.taps.size(), e.cfg.fir_fft_log2,
                             e.cfg.fir_mode == FIR_FFT_PACKED ? " (packed f32x2 variant)" : " (+ 2^14 double segments in one piece, persistent CTAs)");
                else if (e.cfg.fir_mode == FIR_TOEPLITZ)
                    snprintf(b, sizeof b, "fir step: %s, %zu taps, Toeplitz-tiled tcgen05 GEMM 128x256x32, split bf16 (3 MMAs per K step), alg_bytes=8\n",
                             tag.c_str(), nd.taps.size());
                else
                    snprintf(b, sizeof b, "fir step: %s, %zu taps, direct f64 sum in reference order, alg_bytes=8\n", tag.c_str(), nd.taps.size());
                fs.text = b;
                if (nd.fir_pc()) {
                    fs.text.pop_back();
                    const int K = (int)(nd.fir_bank.size() / nd.taps.size());
                    if (e.cfg.fir_mode == FIR_FFT && (int)nd.taps.size() <= fir_fft_max_taps())   // fir_mode 2 / 3 hold no per-channel taps
                        snprintf(b, sizeof b, ", per-channel taps: %d sets, %zu transforms (%d single-channel)\n", K, nd.fir_xf.size(),
                                 nd.fir_xf_single);
                    else
                        snprintf(b, sizeof b, ", per-channel taps: %d sets\n", K);
                    fs.text += b;
                }
                if (fs.fir_out_term >= 0) {
                    fs.text.pop_back();
                    fs.text += ", epilogue (0.0 + y)/1.00010002 -> output terminal " + std::to_string(fs.fir_out_term) + "\n";
                }
                steps.push_back(fs);
                logical_step += 2;
                state_slot = 0;
                memset(cur.prog.states, 0, sizeof cur.prog.states);
                Value v;
                v.where = Value::GLOBAL;
                v.bind_kind = 4;
                v.bind_idx = ni;
                values[{ni, 0}] = v;
            } break;
            case T_MUX: {  // nodes/mux.rs:45-55: copy the selected (averaged) input
                emit_avg(ni, nd.enums[0]);
                values[{ni, 0}] = out_value(0);
            } break;
            case T_DEMUX: {  // nodes/demux.rs:45-58: the other output keeps its zero-init (node.rs:272)
                const int sel = nd.enums[0];
                Value z;
                z.where = Value::ZERO;
                values[{ni, 1 - sel}] = z;
                if (use_step.count({ni, sel})) {
                    emit_avg(ni, 0);
                    values[{ni, sel}] = out_value(sel);
                } else {
                    values[{ni, sel}] = z;
                }
            } break;
            case T_ADD:
            case T_MIX: {
                emit_avg(ni, 1);
                int vb = temp_save(tag + ".b");
                Op op = mk(nd.type == T_ADD ? OP_ADD : OP_MIX);
                std::string pcm;
                if (nd.type == T_MIX) {
                    ctl_param(op, 0, 0);
                    pcm = per_channel(op, ni, 0, 1u);
                }
                emit_avg(ni, 0);
                op.vreg = (uint8_t)vb;
                emit(op, nd.type == T_ADD ? "acc = acc + v" + std::to_string(vb) + "            ; " + tag
                                          : "acc = v" + std::to_string(vb) + "*r + acc*(1-r)" + pcm + "      ; " + tag);
                values[{ni, 0}] = out_value(0);
            } break;
            case T_GATE: {  // extension: x -> vreg, envelope(x) (nodes/envelope.rs arithmetic) -> compare -> select
                emit_avg(ni, 0);
                const int vx = temp_save(tag + ".x");
                Op env = mk(OP_ENVELOPE);
                float v[5];
                op_values(T_GATE, 0, nd.f32.data(), v);
                set_op_values(env, v);
                const std::string pce = per_channel(env, ni, 0, 6u);
                if (alloc_state(env) < 0) return DSPB_ERR_INVALID;
                char b[200];
                snprintf(b, sizeof b, "acc = envelope(acc; ga=%g gr=%g) exact, lane=channel%s  ; %s", env.p[0], env.p[1], pce.c_str(), tag.c_str());
                emit(env, b);
                Op g = mk(OP_GATE);
                g.vreg = (uint8_t)vx;
                op_values(T_GATE, 1, nd.f32.data(), v);
                set_op_values(g, v);
                const std::string pcg = per_channel(g, ni, 1, 1u);
                snprintf(b, sizeof b, "acc = acc >= %g ? v%d : 0%s     ; %s (extension)", nd.f32[0], vx, pcg.c_str(), tag.c_str());
                emit(g, b);
                values[{ni, 0}] = out_value(0);
            } break;
            case T_SIGGEN: {  // nodes/signal_gen.rs:111-130: no signal input, two control ports
                Op op = mk(OP_SIGGEN);
                op.mode = (uint8_t)nd.enums[0];
                ctl_param(op, 0, 0);  // amplitude
                ctl_param(op, 1, 1);  // frequency
                op.p[2] = (float)e.cfg.sample_rate;
                const std::string pcm = per_channel(op, ni, 0, 3u);
                if (alloc_state(op) < 0) return DSPB_ERR_INVALID;
                char b[200];
                snprintf(b, sizeof b, "acc = signal_gen[%s](amp=%g, freq=%g)%s  ; %s", nt.enums[0].variants[nd.enums[0]], nd.f32[0], nd.f32[1],
                         pcm.c_str(), tag.c_str());
                emit(op, b);
                values[{ni, 0}] = out_value(0);
            } break;
            default: {  // single-input effect nodes
                Op op = mk(OP_END);
                std::string desc, pcm;
                char b[320];
                switch (nd.type) {
                    case T_GAIN:
                        op.code = OP_GAIN;
                        ctl_param(op, 0, 0);
                        pcm = per_channel(op, ni, 0, 1u);
                        snprintf(b, sizeof b, "acc *= level(%g)%s", nd.f32[0], pcm.c_str());
                        break;
                    case T_DISTORT:
                        op.code = OP_DISTORT;
                        op.mode = (uint8_t)nd.enums[0];
                        ctl_param(op, 0, 0);
                        pcm = per_channel(op, ni, 0, 1u);
                        // the exact fast division is verified per divisor: per-channel levels divide with IEEE division (dv)
                        if (pcm.empty()) set_const_div(op, 0, 1, nd.f32[0], e.plan_only);
                        snprintf(b, sizeof b, "acc = distort[%s](acc, %g)%s", nt.enums[0].variants[nd.enums[0]], nd.f32[0], pcm.c_str());
                        break;
                    case T_OVERDRIVE:
                        op.code = OP_OVERDRIVE;
                        ctl_param(op, 0, 0);
                        ctl_param(op, 1, 1);
                        ctl_param(op, 2, 2);
                        pcm = per_channel(op, ni, 0, 7u);
                        snprintf(b, sizeof b, "acc = overdrive(acc, %g, %g, %g)%s", nd.f32[0], nd.f32[1], nd.f32[2], pcm.c_str());
                        break;
                    case T_CHEBY: {
                        op.code = OP_CHEBY;
                        float v[5];
                        op_values(T_CHEBY, 0, nd.f32.data(), v);
                        set_op_values(op, v);
                        pcm = per_channel(op, ni, 0, 3u);
                        snprintf(b, sizeof b, "acc = chebyshev(acc, %g, %g)%s", nd.f32[0], nd.f32[1], pcm.c_str());
                    } break;
                    case T_BIQUAD:
                    case T_LOWPASS:
                    case T_HIGHPASS: {
                        ScanTab tab;
                        if (nd.type == T_BIQUAD) {
                            op.code = OP_BIQUAD;
                            set_op_values(op, nd.bq);  // regenerated by every setter (biquad_regenerate)
                            tab = make_scan_tab(nd.bq[3], nd.bq[4]);
                            pcm = per_channel(op, ni, 0, 63u);
                            snprintf(b, sizeof b, "acc = DF1(acc; b=%g,%g,%g a=%g,%g)", nd.bq[0], nd.bq[1], nd.bq[2], nd.bq[3], nd.bq[4]);
                        } else {
                            op.code = nd.type == T_LOWPASS ? OP_LP1 : OP_HP1;
                            float v[5];
                            op_values(nd.type, 0, nd.f32.data(), v);
                            set_op_values(op, v);
                            tab = make_scan_tab(-nd.f32[0], 0.0f);  // z[n] = xr[n] + ratio z[n-1]
                            pcm = per_channel(op, ni, 0, 1u);
                            snprintf(b, sizeof b, "acc = %s(acc; ratio=%g)", nt.cfg_name, nd.f32[0]);
                        }
                        std::string how = " exact, lane=channel";
                        if (!pcm.empty()) {
                            // one scan table per Program, not per channel: per-channel coefficients stay sequential (exact)
                            how = (e.cfg.iir_mode == 1 ? " exact (per-channel coefficients)" : how) + pcm;
                        } else if (e.cfg.iir_mode == 1) {
                            char v[96];
                            if (scan_qualifies(op, tab, e.plan_only)) {
                                // a Program holds kMaxScan scan tables; a fifth qualifying filter would stay sequential and
                                // (all or nothing, close_fused) demote the other four with it: cut the segment here instead
                                if ((int)scan_tabs.size() >= kMaxScan) {
                                    overflow("segment has more time-parallel recurrences than one Program holds");
                                    return DSPB_ERR_INVALID;
                                }
                                scan_tabs.push_back(tab);
                                op.mode = (uint8_t)scan_tabs.size();
                                snprintf(v, sizeof v, " time-parallel scan (probe error %.2g <= %.2g)", tab.probe_err, kScanGate);
                            } else {
                                snprintf(v, sizeof v, " exact, lane=channel (scan probe error %.2g > %.2g)", tab.probe_err, kScanGate);
                            }
                            how = v;
                        }
                        strncat(b, how.c_str(), sizeof b - strlen(b) - 1);
                    } break;
                    case T_ENVELOPE: {
                        op.code = OP_ENVELOPE;
                        float v[5];
                        op_values(T_ENVELOPE, 0, nd.f32.data(), v);
                        set_op_values(op, v);
                        pcm = per_channel(op, ni, 0, 3u);
                        snprintf(b, sizeof b, "acc = envelope(acc; ga=%g gr=%g) exact, lane=channel%s", op.p[0], op.p[1], pcm.c_str());
                    } break;
                    case T_REVERB:
                        op.code = OP_COMB;
                        op.p[0] = nd.f32[1];
                        if ((int)cur.ring_nodes.size() >= kMaxRings) { overflow("too many reverb nodes in one segment"); return DSPB_ERR_INVALID; }
                        pcm = per_channel(op, ni, 0, 2u);
                        op.aux = (uint16_t)cur.ring_nodes.size();
                        cur.ring_nodes.push_back(ni);
                        snprintf(b, sizeof b, "acc += ring*%g ; ring = acc   (D=%lld)%s", nd.f32[1], (long long)nd.D, pcm.c_str());
                        break;
                    default:
                        err = "unhandled node type";
                        return DSPB_ERR_INVALID;
                }
                emit_avg(ni, 0);
                if (is_stateful(nd.type) && alloc_state(op) < 0) return DSPB_ERR_INVALID;
                emit(op, std::string(b) + "  ; " + tag);
                values[{ni, 0}] = out_value(0);
            } break;
        }
        if (!err.empty()) return DSPB_ERR_INVALID;
        if (nd.type != T_FIR && ops.size() == ops_before && !cur_nodes.empty() && cur_nodes.back() == ni) cur_nodes.pop_back();
    }
    close_fused();
    return err.empty() ? DSPB_OK : DSPB_ERR_INVALID;
}

int ensure_resources(dspb_engine* e) {
    const int C = e->cfg.channels;
    const int64_t maxn = e->cfg.max_samples;
    for (auto& np : e->nodes) {
        Node& n = *np;
        if (is_stateful(n.type) && !n.state.p) {
            int r = n.state.alloc((size_t)C * 16, true, e->plan_only);
            if (r) return r;
        }
        if (n.type == T_REVERB && (n.ring_dirty || !n.ring.p)) {
            int r = n.ring.alloc((size_t)C * n.D * 4, true, e->plan_only);  // "full of zeros": reverb.rs:63-68
            if (r) return r;
            n.pos = 0;
            n.ring_dirty = false;
        }
        if (n.type == T_FIR && (n.fir_dirty || !n.Y.p)) {
            const int N = (int)n.taps.size();
            const int F = 1 << e->cfg.fir_fft_log2;
            // history kept in front of a call: N-1 samples; the UPC kernel re-primes its delay line from P whole blocks
            const int upc_P = e->cfg.fir_mode == FIR_FFT ? fir_upc_partitions(N) : 0;
            n.hist_pad = (int)round_up(std::max(std::max(N - 1, 4), upc_P * kUpcBlock), 4);
            if ((int64_t)n.hist_pad + maxn > (1ll << 30)) return fail(DSPB_ERR_INVALID, "max_samples too large for the FIR input ring");
            n.u_ring = (int)round_up(n.hist_pad + maxn, 128);
            int r = n.U.alloc((size_t)C * n.u_ring * 4, true, e->plan_only);
            if (r) return r;
            r = n.Y.alloc((size_t)C * maxn * 4, false, e->plan_only);
            if (r) return r;
            // per-channel impulse responses: K sets of spectra and taps, set k at H + k * fir_fft_spectrum_bytes()
            const bool pc = n.fir_pc();
            const int K = pc ? (int)(n.fir_bank.size() / N) : 1;
            const double* taps_host = pc ? n.fir_bank.data() : n.taps.data();
            r = n.H.alloc(K * fir_fft_spectrum_bytes(), false, e->plan_only);  // every spectrum table of the FFT kernels
            if (r) return r;
            (void)F;
            r = n.taps_dev.alloc((size_t)K * N * 8, false, e->plan_only);
            if (r) return r;
            r = n.set_dev.alloc(pc ? (size_t)C * 4 : 0, false, e->plan_only);
            if (r) return r;
            r = n.xf_dev.alloc(pc ? n.fir_xf.size() * sizeof(int4) : 0, false, e->plan_only);
            if (r) return r;
            if (upc_P) {  // one delay line per transform
                r = n.fdl.alloc(fir_upc_fdl_bytes(N, pc ? (int)n.fir_xf.size() : (C + 1) / 2), true, e->plan_only);
                if (r) return r;
            }
            n.fdl_valid = false;
            n.upc_ctr = 0;
            // work counters of the persistent FFT kernels, one set per launch lane: device-pointer chunk k runs on lane k,
            // an unchunked call and the host path on lane 0
            n.fft_work.clear();
            for (int lane = 0; e->cfg.fir_mode == FIR_FFT && lane < std::max(1, e->dev_chunks); lane++) {
                n.fft_work.push_back(std::make_unique<DevBuf>());
                r = n.fft_work.back()->alloc(fir_fft_work_bytes(), true, e->plan_only);
                if (r) return r;
            }
            const bool toep = e->cfg.fir_mode == FIR_TOEPLITZ && N <= fir_toeplitz_max_taps();
            if (toep) {
                r = n.toep_tiles.alloc(fir_toeplitz_tiles_bytes(N), false, e->plan_only);
                if (r) return r;
                r = n.toep_split.alloc(fir_toeplitz_split_bytes(N, C, maxn), true, e->plan_only);  // rows beyond C stay zero
                if (r) return r;
            }
            if (!e->plan_only) {
                CUDA_TRY(cudaMemcpy(n.taps_dev.p, taps_host, (size_t)K * N * 8, cudaMemcpyHostToDevice));
                if (pc) {
                    CUDA_TRY(cudaMemcpy(n.set_dev.p, n.fir_set.data(), (size_t)C * 4, cudaMemcpyHostToDevice));
                    CUDA_TRY(cudaMemcpy(n.xf_dev.p, n.fir_xf.data(), n.fir_xf.size() * sizeof(int4), cudaMemcpyHostToDevice));
                }
                if (toep) {
                    int rc = fir_toeplitz_prepare(reinterpret_cast<const double*>(n.taps_dev.p), N, n.toep_tiles.p, nullptr);
                    if (rc) return fail(DSPB_ERR_CUDA, "fir_toeplitz_prepare: %s", cudaGetErrorString((cudaError_t)rc));
                } else if (N <= fir_fft_max_taps()) {  // longer impulse responses run on the exact direct path
                    int rc = fir_prepare_spectrum(e->cfg.fir_fft_log2, reinterpret_cast<const double*>(n.taps_dev.p), N, K,
                                                  reinterpret_cast<float2*>(n.H.p), nullptr);
                    if (rc) return fail(DSPB_ERR_CUDA, "fir_prepare_spectrum: %s", cudaGetErrorString((cudaError_t)rc));
                }
                CUDA_TRY(cudaDeviceSynchronize());
            }
            n.started = 0;
            n.u_pos = 0;
            n.fir_dirty = false;
        }
    }
    return DSPB_OK;
}

int lower_graph(dspb_engine* e) {
    int r = ensure_resources(e);
    if (r) return r;
    // Lower; when a segment exceeds what one Program / one CTA holds, cut it in front of the node the Lowerer names and
    // lower again (each attempt adds one cut, so this ends after at most one attempt per node).
    std::set<int> cuts;
    int n_scratch = 0;
    for (;;) {
        Lowerer L(*e);
        L.split_before = cuts;
        r = L.lower();
        if (r) {
            if (L.want_split >= 0 && cuts.insert(L.want_split).second) continue;
            return fail(r, "lowering failed: %s", L.err.c_str());
        }
        int cut = -1;
        for (auto& st : L.steps)
            if (st.kind == STEP_FUSED && fused_smem_bytes(st.prog, st.G) > 200 * 1024) {
                if (st.nodes.size() < 2)
                    return fail(DSPB_ERR_INVALID, "fused segment needs %d B of shared memory (too many live values)", fused_smem_bytes(st.prog, st.G));
                cut = st.nodes[st.nodes.size() / 2];
                break;
            }
        if (cut >= 0) {
            if (cuts.insert(cut).second) continue;
            return fail(DSPB_ERR_INVALID, "fused segment does not fit in shared memory (too many live values)");
        }
        e->steps = std::move(L.steps);
        n_scratch = L.n_scratch;
        break;
    }
    // Per-channel parameter tables.  Rows up to C + 31 exist (zero) because the last CTA's lanes may run past C with
    // discarded results.  Lowering runs inside dspb_process, whose kernels go to non-blocking streams: the pageable copy
    // is waited for here (off the hot path), so a kernel never reads a table the DMA has not finished.
    e->pc_tabs.resize(e->steps.size());
    bool uploaded = false;
    for (size_t i = 0; i < e->steps.size(); i++) {
        Step& st = e->steps[i];
        if (st.pc_host.empty()) continue;
        if (!e->pc_tabs[i]) e->pc_tabs[i] = std::make_unique<DevBuf>();
        DevBuf& tb = *e->pc_tabs[i];
        r = tb.alloc(((size_t)e->cfg.channels + 31) * st.pc_k * 4, true, e->plan_only);
        if (r) return r;
        if (!e->plan_only) CUDA_TRY(cudaMemcpy(tb.p, st.pc_host.data(), st.pc_host.size() * 4, cudaMemcpyHostToDevice));
        st.prog.pc = tb.p;
        st.prog.pc_stride = st.pc_k;
        uploaded = true;
    }
    if (uploaded && !e->plan_only) CUDA_TRY(cudaDeviceSynchronize());
    while ((int)e->scratch.size() < n_scratch) {
        auto b = std::make_unique<DevBuf>();
        r = b->alloc((size_t)e->cfg.channels * e->cfg.max_samples * 4, false, e->plan_only);
        if (r) return r;
        e->scratch.push_back(std::move(b));
    }
    e->lowered = true;
    return DSPB_OK;
}

int topo_sort(dspb_engine* e) {
    const int N = (int)e->nodes.size();
    e->in_links.assign(N, {});
    e->out_links.assign(N, {});
    for (int i = 0; i < N; i++) {
        e->in_links[i].assign(kNodeTypes[e->nodes[i]->type].ins.size(), {});
        e->out_links[i].assign(kNodeTypes[e->nodes[i]->type].outs.size(), {});
    }
    std::vector<int> indeg(N, 0), nlinks(N, 0);
    for (size_t l = 0; l < e->links.size(); l++) {
        const Link& k = e->links[l];
        e->in_links[k.dst][k.dport].push_back((int)l);  // link-creation order (runtime.rs:125-134)
        e->out_links[k.src][k.sport].push_back((int)l);
        indeg[k.dst]++;
        nlinks[k.src]++;
        nlinks[k.dst]++;
    }
    e->in_terms.clear();
    e->out_terms.clear();
    for (int i = 0; i < N; i++) {
        if (e->nodes[i]->type == T_INPUT) e->in_terms.push_back(i);
        if (e->nodes[i]->type == T_OUTPUT) e->out_terms.push_back(i);
    }
    // Depth-first Kahn (LIFO ready list) keeps chains contiguous so values stay in registers;
    // nodes with no links at all never run (runtime.rs:661-668).
    e->order.clear();
    std::vector<int> ready;
    for (int i = N - 1; i >= 0; i--)
        if (indeg[i] == 0) ready.push_back(i);
    int seen = 0;
    while (!ready.empty()) {
        int n = ready.back();
        ready.pop_back();
        seen++;
        if (nlinks[n] > 0) e->order.push_back(n);
        for (int q = (int)e->out_links[n].size() - 1; q >= 0; q--)
            for (int li = (int)e->out_links[n][q].size() - 1; li >= 0; li--) {
                int d = e->links[e->out_links[n][q][li]].dst;
                if (--indeg[d] == 0) ready.push_back(d);
            }
    }
    if (seen != N) return fail(DSPB_ERR_GRAPH, "graph has a cycle (the reference would deadlock: every link ring starts empty, runtime.rs:568)");
    return DSPB_OK;
}

// Bind per-call pointers and launch every step for channels [c0, c1).
// `lane`: index of the concurrent launch lane (device-pointer chunks run on their own streams), selects per-lane scratch.
int run_steps(dspb_engine* e, const float* const* d_in, float* const* d_out, int64_t n, int c0, int c1, cudaStream_t st, int lane = 0) {
    int step_idx = -1;
    for (auto& s : e->steps) {
        step_idx++;
        struct ProfScope {  // CUDA events around this step on the launching stream
            dspb_engine* e; cudaStream_t st; bool on; cudaEvent_t a{}, b{}; int idx;
            ProfScope(dspb_engine* e_, cudaStream_t st_, int idx_) : e(e_), st(st_), on(e_->prof_on && e_->prof.size() < 16384), idx(idx_) {
                if (on) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, st); }
            }
            ~ProfScope() { if (on) { cudaEventRecord(b, st); e->prof.push_back({idx, a, b}); } }
        } prof_scope(e, st, step_idx);
        if (s.kind == STEP_FUSED) {
            Program& P = s.prog;
            for (size_t b = 0; b < s.binds.size(); b++) {
                BufDesc& d = P.bufs[b];
                d.ring_len = 0;
                d.ring_pos = 0;
                switch (s.binds[b].kind) {
                    case 0: d.base = const_cast<float*>(d_in[s.binds[b].idx]); d.row_stride = n; break;
                    case 1: d.base = d_out[s.binds[b].idx]; d.row_stride = n; break;
                    case 2: d.base = e->scratch[s.binds[b].idx]->p; d.row_stride = e->cfg.max_samples; break;
                    case 3: {  // FIR input ring
                        Node& f = *e->nodes[s.binds[b].idx];
                        d.row_stride = f.u_ring;
                        d.base = f.U.p;
                        d.ring_len = f.u_ring;
                        d.ring_pos = f.u_pos;
                    } break;
                    case 4: {
                        Node& f = *e->nodes[s.binds[b].idx];
                        d.base = f.Y.p;
                        d.row_stride = e->cfg.max_samples;
                    } break;
                }
            }
            for (size_t r = 0; r < s.ring_nodes.size(); r++) {
                Node& rn = *e->nodes[s.ring_nodes[r]];
                P.rings[r].base = rn.ring.p;
                P.rings[r].D = rn.D;
                P.rings[r].pos = rn.pos;
            }
            int rc = launch_fused(P, s.G, c0, c1, n, st);
            if (rc) return fail(DSPB_ERR_CUDA, "fused kernel launch: %s", cudaGetErrorString((cudaError_t)rc));
            e->last_launches++;
        } else {
            Node& f = *e->nodes[s.fir_node];
            FirPlan fp;
            fp.mode = e->cfg.fir_mode;
            if (fp.mode == FIR_TOEPLITZ && (int)f.taps.size() > fir_toeplitz_max_taps()) fp.mode = FIR_DIRECT;
            if ((fp.mode == FIR_FFT || fp.mode == FIR_FFT_PACKED) && (int)f.taps.size() > fir_fft_max_taps()) fp.mode = FIR_DIRECT;  // long IRs: exact path
            fp.toep_tiles = f.toep_tiles.p;
            fp.toep_split = f.toep_split.p;
            fp.toep_max_samples = e->cfg.max_samples;
            fp.log2F = e->cfg.fir_fft_log2;
            fp.n_taps = (int)f.taps.size();
            fp.hist_pad = f.hist_pad;
            fp.H = reinterpret_cast<const float2*>(f.H.p);
            fp.taps = reinterpret_cast<const double*>(f.taps_dev.p);
            fp.divisor = f.enums[0] == 0 ? 1.0f / (float)f.taps.size() : 1.0f;  // fir.rs:187-190
            fp.post_nf = s.fir_post_nf;
            fp.u_ring = f.u_ring;
            fp.u_pos = f.u_pos;
            // work counters of the persistent FFT kernels: lanes run concurrently on their own streams
            fp.fft_work = fp.mode == FIR_FFT ? f.fft_work[lane]->p : nullptr;
            if (f.fir_pc()) {  // per-channel impulse responses: the transform-table slice of channels [c0, c1)
                if (c0 % 32 || (c1 % 32 && c1 != e->cfg.channels))
                    return fail(DSPB_ERR_INVALID, "per-channel taps: launch range [%d, %d) is not aligned to 32 channels", c0, c1);
                const int x0 = f.fir_xf_group[c0 / 32], x1 = f.fir_xf_group[(c1 + 31) / 32];
                fp.set_index = reinterpret_cast<const int*>(f.set_dev.p);
                fp.xf = reinterpret_cast<const int4*>(f.xf_dev.p) + x0;
                fp.n_xf = x1 - x0;
                fp.xf0 = x0;
                fp.h_stride = (int64_t)(fir_fft_spectrum_bytes() / sizeof(float2));
            }
            // short calls (1 or 2 blocks of 1024): uniformly partitioned convolution with a frequency-domain delay line.  Measured
            // at 4096 channels: 62 / 101 / 141 us for 1 / 2 / 3 blocks against 92 - 104 us for the one 8192-point window the
            // segment kernel needs for any call of up to 4096 samples.
            constexpr int kUpcMaxBlocks = 2;
            const int upc_P = fir_upc_partitions(fp.n_taps);
            f.upc_this_call = fp.mode == FIR_FFT && upc_P > 0 && f.fdl.p && n % kUpcBlock == 0 && n / kUpcBlock <= kUpcMaxBlocks;
            if (f.upc_this_call) {
                fp.upc_fdl = f.fdl.p;
                fp.upc_prime = f.fdl_valid ? 0 : upc_P - 1;
                fp.upc_block0 = f.upc_ctr;
            }
            int nl = 0;
            float* yp = s.fir_out_term >= 0 ? d_out[s.fir_out_term] : f.Y.p;
            const int64_t ys = s.fir_out_term >= 0 ? n : e->cfg.max_samples;
            int rc = launch_fir(fp, f.U.p, f.u_ring, yp, ys, c0, c1, n, f.started, st, &nl);
            if (rc) return fail(DSPB_ERR_CUDA, "fir kernel launch: %s", cudaGetErrorString((cudaError_t)rc));
            e->last_launches += nl;
        }
    }
    return DSPB_OK;
}

void advance_state(dspb_engine* e, int64_t n) {
    for (auto& np : e->nodes) {
        Node& nd = *np;
        if (nd.type == T_REVERB && nd.D > 0) nd.pos = (nd.pos + n) % nd.D;
        if (nd.type == T_FIR) {
            nd.started += n;
            nd.u_pos = (int)((nd.u_pos + n) % nd.u_ring);
            nd.fdl_valid = nd.upc_this_call;   // a call through the segment kernels leaves the delay line stale
            if (nd.upc_this_call) nd.upc_ctr += n / kUpcBlock;
            nd.upc_this_call = false;
        }
    }
}

int check_ready(dspb_engine* e, int64_t n) {
    if (!e->compiled) return fail(DSPB_ERR_GRAPH, "graph not compiled (call dspb_compile after structural changes)");
    if (n <= 0 || n % e->cfg.ref_block) return fail(DSPB_ERR_INVALID, "n_samples must be a positive multiple of %d", e->cfg.ref_block);
    if (n > e->cfg.max_samples) return fail(DSPB_ERR_INVALID, "n_samples %lld exceeds max_samples %lld", (long long)n, (long long)e->cfg.max_samples);
    if (!e->lowered) {
        int r = lower_graph(e);
        if (r) return r;
    }
    return DSPB_OK;
}

// after_settings_change (lib.rs:560-568) of a slider store, shared or per channel
int after_settings_change(dspb_engine* e, Node& n) {
    if (!e->plan_only) CUDA_TRY(cudaSetDevice(e->cfg.device));
    if (n.type == T_BIQUAD) {  // regenerate_filter: new coefficients + reset_state (per-channel ones: at lowering, op_values)
        biquad_regenerate(n);
        if (n.state.p && !e->plan_only) CUDA_TRY(cudaMemsetAsync(n.state.p, 0, n.state.bytes, nullptr));
    }
    if (n.type == T_REVERB) {  // refresh_seconds on ANY slider of the node
        n.D = reverb_delay(n.f32[0], e->cfg.sample_rate, e->cfg.ring_granule);
        n.ring_dirty = true;
    }
    e->lowered = false;
    return DSPB_OK;
}

}  // namespace

// =================================================== C ABI =====================================================
extern "C" {

const char* dspb_last_error(void) { return g_err.c_str(); }
int dspb_sync(dspb_engine* e);
// parameter / structure changes touch state the asynchronous host calls still use: finish those first
#define DSPB_QUIESCE(e)                                   \
    do {                                                  \
        if ((e)->host_inflight) {                         \
            int _q = dspb_sync(e);                        \
            if (_q) return _q;                            \
        }                                                 \
    } while (0)
int dspb_abi_version(void) { return DSPB_ABI_VERSION; }

int dspb_engine_create(const dspb_config* cfg, dspb_engine** out) {
    if (!cfg || !out) return fail(DSPB_ERR_INVALID, "null argument");
    if (cfg->channels <= 0) return fail(DSPB_ERR_INVALID, "channels must be > 0");
    const bool plan_only = cfg->device == -1;  // schedules can be built and described, nothing can run
    if (!plan_only) {
        int ndev = 0;
        cudaError_t ce = cudaGetDeviceCount(&ndev);
        if (ce != cudaSuccess || ndev == 0)
            return fail(DSPB_ERR_CUDA, "no usable CUDA device (%s); this engine has no CPU fallback", ce == cudaSuccess ? "device count 0" : cudaGetErrorString(ce));
        if (cfg->device < 0 || cfg->device >= ndev) return fail(DSPB_ERR_INVALID, "device %d out of range (have %d)", cfg->device, ndev);
        CUDA_TRY(cudaSetDevice(cfg->device));
        cudaDeviceProp prop;
        CUDA_TRY(cudaGetDeviceProperties(&prop, cfg->device));
        if (prop.major < 10) return fail(DSPB_ERR_CUDA, "device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
    }
    auto* e = new dspb_engine();
    e->plan_only = plan_only;
    e->cfg = *cfg;
    if (e->cfg.sample_rate <= 0) e->cfg.sample_rate = 48000;
    if (e->cfg.ref_block <= 0) e->cfg.ref_block = kRefBlock;
    if (e->cfg.ref_block != kRefBlock) { delete e; return fail(DSPB_ERR_INVALID, "ref_block must be 128 (node.rs:257)"); }
    if (e->cfg.block <= 0) e->cfg.block = kRefBlock;
    if (e->cfg.block % kRefBlock) { delete e; return fail(DSPB_ERR_INVALID, "block must be a multiple of 128"); }
    if (e->cfg.ring_granule <= 0) e->cfg.ring_granule = 1024;
    if (e->cfg.max_samples <= 0) e->cfg.max_samples = 64 * (int64_t)e->cfg.block;
    e->cfg.max_samples = round_up(e->cfg.max_samples, kRefBlock);
    if (e->cfg.fir_fft_log2 <= 0) e->cfg.fir_fft_log2 = 13;
    if (e->cfg.fir_fft_log2 != 13) { delete e; return fail(DSPB_ERR_INVALID, "fir_fft_log2 must be 13 in this build"); }
    if (e->cfg.fir_mode < FIR_FFT || e->cfg.fir_mode > FIR_FFT_PACKED) {
        delete e;
        return fail(DSPB_ERR_INVALID, "fir_mode must be 0 (FFT), 1 (direct), 2 (Toeplitz tensor-core) or 3 (packed FFT)");
    }
    if (e->cfg.iir_mode < 0 || e->cfg.iir_mode > 1) {
        delete e;
        return fail(DSPB_ERR_INVALID, "iir_mode must be 0 (exact recurrences) or 1 (time-parallel scan where the measured error allows)");
    }
    if (const char* g = getenv("DSPB_FORCE_G")) e->force_G = atoi(g);
    if (const char* g = getenv("DSPB_CHUNKS")) e->dev_chunks = std::max(1, std::min(8, atoi(g)));
    *out = e;
    return DSPB_OK;
}

void dspb_engine_destroy(dspb_engine* e) {
    if (!e) return;
    if (!e->plan_only) {
        cudaSetDevice(e->cfg.device);
        cudaDeviceSynchronize();
    }
    delete e;
}

int dspb_node_add(dspb_engine* e, const char* cfg_name, int64_t node_id) {
    if (!e || !cfg_name) return fail(DSPB_ERR_INVALID, "null argument");
    if (e->find(node_id) >= 0) return fail(DSPB_ERR_INVALID, "duplicate node id %lld", (long long)node_id);
    int type = -1;
    for (int t = 0; t < T_COUNT; t++)
        if (!strcmp(kNodeTypes[t].cfg_name, cfg_name)) type = t;
    if (type < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown typename '%s' (reference: panic in NodeInstance::restore, runtime.rs:634-637)", cfg_name);
    auto n = std::make_unique<Node>();
    n->id = node_id;
    n->type = type;
    for (auto& p : kNodeTypes[type].params) n->f32.push_back(p.def);
    n->f32_pc.resize(n->f32.size());
    for (auto& en : kNodeTypes[type].enums) n->enums.push_back(en.def);
    if (type == T_REVERB) n->D = round_up(128, e->cfg.ring_granule);  // make_buffer(): circular_buffer(128), reverb.rs:44-52
    e->nodes.push_back(std::move(n));
    e->compiled = e->lowered = false;
    return DSPB_OK;
}

int dspb_node_set_f32(dspb_engine* e, int64_t node_id, const char* field, float value) {
    if (!e || !field) return fail(DSPB_ERR_INVALID, "null argument");
    int i = e->find(node_id);
    if (i < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown node id %lld", (long long)node_id);
    Node& n = *e->nodes[i];
    int p = param_index(kNodeTypes[n.type], field);
    if (p < 0) return fail(DSPB_ERR_UNKNOWN_PORT, "node type '%s' has no f32 field '%s'", kNodeTypes[n.type].cfg_name, field);
    DSPB_QUIESCE(e);
    n.f32[p] = value;
    n.f32_pc[p].clear();  // shared again
    return after_settings_change(e, n);
}

int dspb_node_set_f32_channels(dspb_engine* e, int64_t node_id, const char* field, const float* values, int64_t n_values) {
    if (!e || !field || !values) return fail(DSPB_ERR_INVALID, "null argument");
    int i = e->find(node_id);
    if (i < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown node id %lld", (long long)node_id);
    Node& n = *e->nodes[i];
    int p = param_index(kNodeTypes[n.type], field);
    if (p < 0) return fail(DSPB_ERR_UNKNOWN_PORT, "node type '%s' has no f32 field '%s'", kNodeTypes[n.type].cfg_name, field);
    if (n.type == T_REVERB && p == 0)
        return fail(DSPB_ERR_INVALID, "reverb.seconds cannot vary per channel: it sets the ring length D, and the ring is one "
                                      "[C x D] array with one D for every channel (use dspb_node_set_f32)");
    if (n_values != e->cfg.channels)
        return fail(DSPB_ERR_INVALID, "n_values %lld != channels %d", (long long)n_values, e->cfg.channels);
    bool same = true;  // bit for bit: NaN payloads and the sign of zero count
    for (int64_t c = 1; c < n_values && same; c++) same = memcmp(&values[c], &values[0], 4) == 0;
    if (same) return dspb_node_set_f32(e, node_id, field, values[0]);
    DSPB_QUIESCE(e);
    n.f32_pc[p].assign(values, values + n_values);
    n.f32[p] = values[0];
    return after_settings_change(e, n);
}

int dspb_node_set_enum(dspb_engine* e, int64_t node_id, const char* field, const char* variant) {
    if (!e || !field || !variant) return fail(DSPB_ERR_INVALID, "null argument");
    int i = e->find(node_id);
    if (i < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown node id %lld", (long long)node_id);
    Node& n = *e->nodes[i];
    const NodeType& nt = kNodeTypes[n.type];
    for (size_t k = 0; k < nt.enums.size(); k++)
        if (!strcmp(nt.enums[k].name, field)) {
            for (size_t v = 0; v < nt.enums[k].variants.size(); v++)
                if (!strcmp(nt.enums[k].variants[v], variant)) {
                    DSPB_QUIESCE(e);
                    n.enums[k] = (int)v;
                    e->lowered = false;
                    return DSPB_OK;
                }
            return fail(DSPB_ERR_UNKNOWN_PORT, "enum field '%s' has no variant '%s'", field, variant);
        }
    return fail(DSPB_ERR_UNKNOWN_PORT, "node type '%s' has no enum field '%s'", nt.cfg_name, field);
}

int dspb_node_set_taps(dspb_engine* e, int64_t node_id, const double* taps, int64_t n_taps) {
    if (!e || !taps || n_taps <= 0) return fail(DSPB_ERR_INVALID, "bad taps");
    int i = e->find(node_id);
    if (i < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown node id %lld", (long long)node_id);
    Node& n = *e->nodes[i];
    if (n.type != T_FIR) return fail(DSPB_ERR_INVALID, "node %lld is not a fir", (long long)node_id);
    DSPB_QUIESCE(e);
    n.taps.assign(taps, taps + n_taps);
    n.fir_bank.clear();  // shared again
    n.fir_set.clear();
    n.fir_xf.clear();
    n.fir_xf_group.clear();
    n.fir_xf_single = 0;
    n.fir_dirty = true;
    e->lowered = false;
    return DSPB_OK;
}

int dspb_node_set_impulse_response(dspb_engine* e, int64_t node_id, const double* h, int64_t n) {
    if (!h || n <= 0) return fail(DSPB_ERR_INVALID, "bad impulse response");
    std::vector<double> rev(h, h + n);
    std::reverse(rev.begin(), rev.end());  // taps.reverse(), nodes/fir.rs:163-168
    return dspb_node_set_taps(e, node_id, rev.data(), n);
}

int dspb_node_set_taps_channels(dspb_engine* e, int64_t node_id, const double* taps, int64_t n_sets, int64_t n_taps,
                                const int32_t* set_index, int64_t n_channels) {
    if (!e) return fail(DSPB_ERR_INVALID, "null engine");
    int i = e->find(node_id);
    if (i < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown node id %lld", (long long)node_id);
    Node& n = *e->nodes[i];
    if (n.type != T_FIR) return fail(DSPB_ERR_INVALID, "node %lld is not a fir", (long long)node_id);
    if (!taps || !set_index) return fail(DSPB_ERR_INVALID, "null argument");
    if (n_sets < 1 || n_taps < 1) return fail(DSPB_ERR_INVALID, "n_sets %lld and n_taps %lld must be >= 1", (long long)n_sets, (long long)n_taps);
    const int C = e->cfg.channels;
    if (n_channels != C) return fail(DSPB_ERR_INVALID, "n_channels %lld != channels %d", (long long)n_channels, C);
    for (int c = 0; c < C; c++)
        if (set_index[c] < 0 || set_index[c] >= n_sets)
            return fail(DSPB_ERR_INVALID, "set_index[%d] = %d is outside [0, %lld)", c, (int)set_index[c], (long long)n_sets);
    // Deduplicate: bit-identical rows (memcmp) are one set, unused rows are dropped, sets are numbered in order of first use.
    const size_t row_bytes = (size_t)n_taps * sizeof(double);
    std::vector<int32_t> remap(n_sets, -1), set(C);
    std::vector<int64_t> kept;                          // original row of each set
    std::map<uint64_t, std::vector<int>> by_hash;       // FNV-1a of a row's bytes -> sets with that hash
    for (int c = 0; c < C; c++) {
        const int32_t s = set_index[c];
        if (remap[s] < 0) {
            const unsigned char* row = reinterpret_cast<const unsigned char*>(taps + (size_t)s * n_taps);
            uint64_t h = 1469598103934665603ull;
            for (size_t b = 0; b < row_bytes; b++) h = (h ^ row[b]) * 1099511628211ull;
            auto& cand = by_hash[h];
            for (int k : cand)
                if (!memcmp(row, taps + (size_t)kept[k] * n_taps, row_bytes)) { remap[s] = k; break; }
            if (remap[s] < 0) {
                remap[s] = (int32_t)kept.size();
                cand.push_back(remap[s]);
                kept.push_back(s);
            }
        }
        set[c] = remap[s];
    }
    if (kept.size() == 1) return dspb_node_set_taps(e, node_id, taps + (size_t)kept[0] * n_taps, n_taps);  // every channel alike
    if (e->cfg.fir_mode != FIR_FFT && e->cfg.fir_mode != FIR_DIRECT)
        return fail(DSPB_ERR_INVALID, "per-channel taps need fir_mode 0 or 1 (FFT or direct); this engine has fir_mode %d", e->cfg.fir_mode);
    DSPB_QUIESCE(e);
    n.fir_bank.resize(kept.size() * (size_t)n_taps);
    for (size_t k = 0; k < kept.size(); k++) memcpy(n.fir_bank.data() + k * n_taps, taps + (size_t)kept[k] * n_taps, row_bytes);
    n.taps.assign(n.fir_bank.begin(), n.fir_bank.begin() + n_taps);
    n.fir_set = std::move(set);
    fir_transforms(n, C);
    n.fir_dirty = true;
    e->lowered = false;
    return DSPB_OK;
}

int dspb_node_set_impulse_response_channels(dspb_engine* e, int64_t node_id, const double* h, int64_t n_sets, int64_t n_taps,
                                            const int32_t* set_index, int64_t n_channels) {
    if (!h || n_sets < 1 || n_taps < 1) return fail(DSPB_ERR_INVALID, "bad impulse responses");
    std::vector<double> rev(h, h + n_sets * n_taps);
    for (int64_t k = 0; k < n_sets; k++) std::reverse(rev.begin() + k * n_taps, rev.begin() + (k + 1) * n_taps);  // per row, like the WAV loader
    return dspb_node_set_taps_channels(e, node_id, rev.data(), n_sets, n_taps, set_index, n_channels);
}

int dspb_link(dspb_engine* e, int64_t src_node, const char* out_port, int64_t dst_node, const char* in_port) {
    if (!e || !out_port || !in_port) return fail(DSPB_ERR_INVALID, "null argument");
    int s = e->find(src_node), d = e->find(dst_node);
    if (s < 0 || d < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown node id in link %lld -> %lld", (long long)src_node, (long long)dst_node);
    int sp = port_index(kNodeTypes[e->nodes[s]->type].outs, out_port);
    int dp = port_index(kNodeTypes[e->nodes[d]->type].ins, in_port);
    if (sp < 0) return fail(DSPB_ERR_UNKNOWN_PORT, "node type '%s' has no output port '%s'", kNodeTypes[e->nodes[s]->type].cfg_name, out_port);
    if (dp < 0) return fail(DSPB_ERR_UNKNOWN_PORT, "node type '%s' has no input port '%s'", kNodeTypes[e->nodes[d]->type].cfg_name, in_port);
    e->links.push_back(Link{s, sp, d, dp});
    e->compiled = e->lowered = false;
    return DSPB_OK;
}

int dspb_compile(dspb_engine* e) {
    if (!e) return fail(DSPB_ERR_INVALID, "null engine");
    DSPB_QUIESCE(e);
    if (!e->plan_only) CUDA_TRY(cudaSetDevice(e->cfg.device));
    int r = topo_sort(e);
    if (r) return r;
    e->compiled = true;
    e->lowered = false;
    return lower_graph(e);
}

int dspb_reset_state(dspb_engine* e) {
    if (!e) return fail(DSPB_ERR_INVALID, "null engine");
    if (e->plan_only) return fail(DSPB_ERR_CUDA, "planning-only engine (device -1) holds no state");
    CUDA_TRY(cudaSetDevice(e->cfg.device));
    CUDA_TRY(cudaDeviceSynchronize());
    e->host_inflight = false;
    for (auto& n : e->nodes) {
        int r = clear_node_state(e, *n);
        if (r) return r;
    }
    e->rs.target_hz = 0.0;  // the next dspb_resample_dup_stereo call builds a fresh converter
    return DSPB_OK;
}

int dspb_process(dspb_engine* e, const float* const* inputs, float* const* outputs, int64_t n, int mem_kind, void* stream) {
    if (!e) return fail(DSPB_ERR_INVALID, "null engine");
    if (e->plan_only) return fail(DSPB_ERR_CUDA, "planning-only engine (device -1) cannot process: there is no CPU fallback");
    CUDA_TRY(cudaSetDevice(e->cfg.device));
    int r = check_ready(e, n);
    if (r) return r;
    const int C = e->cfg.channels;
    const size_t n_in = e->in_terms.size(), n_out = e->out_terms.size();
    if ((n_in && !inputs) || (n_out && !outputs)) return fail(DSPB_ERR_INVALID, "null buffer table");
    for (size_t i = 0; i < n_in; i++)
        if (!inputs[i]) return fail(DSPB_ERR_INVALID, "null input buffer %zu", i);
    for (size_t i = 0; i < n_out; i++)
        if (!outputs[i]) return fail(DSPB_ERR_INVALID, "null output buffer %zu", i);
    e->last_launches = 0;
    if (mem_kind == DSPB_MEM_DEVICE && e->host_inflight) {  // state is shared: finish the asynchronous host calls first
        int rs = dspb_sync(e);
        if (rs) return rs;
    }
    if (mem_kind == DSPB_MEM_DEVICE) {
        for (size_t i = 0; i < n_in; i++)
            if ((uintptr_t)inputs[i] & 15) return fail(DSPB_ERR_INVALID, "device buffers must be 16-byte aligned");
        for (size_t i = 0; i < n_out; i++)
            if ((uintptr_t)outputs[i] & 15) return fail(DSPB_ERR_INVALID, "device buffers must be 16-byte aligned");
        int chunks = e->dev_chunks;
        if (e->steps.size() < 2 || C < 64 * chunks) chunks = 1;
        if (chunks <= 1) {
            r = run_steps(e, inputs, outputs, n, 0, C, (cudaStream_t)stream);
            if (r) return r;
        } else {
            // fork: every chunk's step chain runs on its own stream, so the FIR kernel of chunk k overlaps the
            // fused kernel of chunk k+1 (both are latency-limited on their own); join back on the caller's stream
            cudaStream_t cs = (cudaStream_t)stream;
            while ((int)e->chunk_streams.size() < chunks) {
                cudaStream_t st2;
                CUDA_TRY(cudaStreamCreateWithFlags(&st2, cudaStreamNonBlocking));
                e->chunk_streams.push_back(st2);
            }
            while ((int)e->chunk_events.size() < chunks + 1) {
                cudaEvent_t ev;
                CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
                e->chunk_events.push_back(ev);
            }
            CUDA_TRY(cudaEventRecord(e->chunk_events[chunks], cs));
            int per = ((C + chunks - 1) / chunks + 31) / 32 * 32;
            for (int k = 0; k < chunks; k++) {
                const int c0 = k * per, c1 = std::min(C, c0 + per);
                if (c0 >= c1) break;
                CUDA_TRY(cudaStreamWaitEvent(e->chunk_streams[k], e->chunk_events[chunks], 0));
                r = run_steps(e, inputs, outputs, n, c0, c1, e->chunk_streams[k], k);
                if (r) return r;
                CUDA_TRY(cudaEventRecord(e->chunk_events[k], e->chunk_streams[k]));
                CUDA_TRY(cudaStreamWaitEvent(cs, e->chunk_events[k], 0));
            }
        }
        advance_state(e, n);
        return DSPB_OK;
    }
    if (mem_kind != DSPB_MEM_HOST && mem_kind != DSPB_MEM_HOST_ASYNC)
        return fail(DSPB_ERR_INVALID, "mem_kind must be DSPB_MEM_DEVICE, DSPB_MEM_HOST or DSPB_MEM_HOST_ASYNC");
    // Host buffers: channel ranges are independent, so H2D / kernels / D2H of successive channel
    // chunks overlap on three streams.  DSPB_MEM_HOST_ASYNC returns without waiting: the next call's H2D then runs next
    // to this call's D2H (PCIe is full duplex); chunk k of a call waits for chunk k of the previous one wherever the two
    // share a staging region (events below), which needs the same n and chunking -- otherwise the calls are serialised.
    if (e->host_inflight && (e->host_last_n != n)) {
        CUDA_TRY(cudaStreamSynchronize(e->s_d2h));
        CUDA_TRY(cudaStreamSynchronize(e->s_cmp));
        e->host_inflight = false;
    }
    if (!e->s_cmp) {
        CUDA_TRY(cudaStreamCreateWithFlags(&e->s_h2d, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&e->s_cmp, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&e->s_d2h, cudaStreamNonBlocking));
    }
    while (e->h_in.size() < n_in) {
        auto b = std::make_unique<DevBuf>();
        r = b->alloc((size_t)C * e->cfg.max_samples * 4, false, e->plan_only);
        if (r) return r;
        e->h_in.push_back(std::move(b));
    }
    while (e->h_out.size() < n_out) {
        auto b = std::make_unique<DevBuf>();
        r = b->alloc((size_t)C * e->cfg.max_samples * 4, false, e->plan_only);
        if (r) return r;
        e->h_out.push_back(std::move(b));
    }
    std::vector<const float*> din(n_in);
    std::vector<float*> dout(n_out);
    for (size_t i = 0; i < n_in; i++) din[i] = e->h_in[i]->p;
    for (size_t i = 0; i < n_out; i++) dout[i] = e->h_out[i]->p;
    static const int host_chunks = getenv("DSPB_HOST_CHUNKS") ? std::max(1, std::min(64, atoi(getenv("DSPB_HOST_CHUNKS")))) : 16;
    int n_chunks = host_chunks;
    int per = (C + n_chunks - 1) / n_chunks;
    per = (per + 31) / 32 * 32;  // keep CTA channel groups intact
    n_chunks = (C + per - 1) / per;
    while ((int)e->ev_pool.size() < 3 * n_chunks) {
        cudaEvent_t ev;
        CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        e->ev_pool.push_back(ev);
    }
    for (int k = 0; k < n_chunks; k++) {
        const int c0 = k * per, c1 = std::min(C, c0 + per);
        cudaEvent_t ev_h2d = e->ev_pool[3 * k], ev_cmp = e->ev_pool[3 * k + 1], ev_d2h = e->ev_pool[3 * k + 2];
        // the previous (asynchronous) call's kernels of this chunk still read the staging region this copy overwrites
        if (e->host_inflight) CUDA_TRY(cudaStreamWaitEvent(e->s_h2d, ev_cmp, 0));
        for (size_t i = 0; i < n_in; i++)
            CUDA_TRY(cudaMemcpyAsync(e->h_in[i]->p + (size_t)c0 * n, inputs[i] + (size_t)c0 * n, (size_t)(c1 - c0) * n * 4, cudaMemcpyHostToDevice, e->s_h2d));
        CUDA_TRY(cudaEventRecord(ev_h2d, e->s_h2d));
        CUDA_TRY(cudaStreamWaitEvent(e->s_cmp, ev_h2d, 0));
        // ... and its D2H of this chunk still reads the output staging region these kernels overwrite
        if (e->host_inflight) CUDA_TRY(cudaStreamWaitEvent(e->s_cmp, ev_d2h, 0));
        r = run_steps(e, din.data(), dout.data(), n, c0, c1, e->s_cmp);
        if (r) return r;
        CUDA_TRY(cudaEventRecord(ev_cmp, e->s_cmp));
        CUDA_TRY(cudaStreamWaitEvent(e->s_d2h, ev_cmp, 0));
        for (size_t i = 0; i < n_out; i++)
            CUDA_TRY(cudaMemcpyAsync(outputs[i] + (size_t)c0 * n, e->h_out[i]->p + (size_t)c0 * n, (size_t)(c1 - c0) * n * 4, cudaMemcpyDeviceToHost, e->s_d2h));
        CUDA_TRY(cudaEventRecord(ev_d2h, e->s_d2h));
    }
    advance_state(e, n);
    e->host_last_n = n;
    if (mem_kind == DSPB_MEM_HOST_ASYNC) {
        e->host_inflight = true;
        return DSPB_OK;
    }
    CUDA_TRY(cudaStreamSynchronize(e->s_d2h));
    CUDA_TRY(cudaStreamSynchronize(e->s_cmp));
    e->host_inflight = false;
    return DSPB_OK;
}

int dspb_sync(dspb_engine* e) {
    if (!e) return fail(DSPB_ERR_INVALID, "null engine");
    if (e->plan_only) return DSPB_OK;
    CUDA_TRY(cudaSetDevice(e->cfg.device));
    if (e->s_d2h) CUDA_TRY(cudaStreamSynchronize(e->s_d2h));
    if (e->s_cmp) CUDA_TRY(cudaStreamSynchronize(e->s_cmp));
    if (e->s_h2d) CUDA_TRY(cudaStreamSynchronize(e->s_h2d));
    e->host_inflight = false;
    return DSPB_OK;
}

// ---- device-boundary format steps (boundary.cu) ----------------------------------------------------------
static int boundary_step(dspb_engine* e, const float* src, float* dst, int64_t n_frames, int mem_kind, void* stream, bool fold) {
    if (!e || (n_frames > 0 && (!src || !dst))) return fail(DSPB_ERR_INVALID, "null argument");
    if (n_frames < 0) return fail(DSPB_ERR_INVALID, "n_frames must be >= 0");
    if (e->plan_only) return fail(DSPB_ERR_CUDA, "engine was created with device = -1 (planning only): no CUDA device, no CPU fallback");
    if (n_frames == 0) return DSPB_OK;
    CUDA_TRY(cudaSetDevice(e->cfg.device));
    const long long total = (long long)e->cfg.channels * n_frames;
    const size_t in_bytes = (size_t)total * (fold ? 8 : 4), out_bytes = (size_t)total * (fold ? 4 : 8);
    cudaStream_t st = (cudaStream_t)stream;
    if (mem_kind == DSPB_MEM_DEVICE) {
        int rc = fold ? dspb::launch_fold_stereo(src, dst, total, st) : dspb::launch_dup_stereo(src, dst, total, st);
        if (rc) return fail(DSPB_ERR_CUDA, "boundary kernel launch: %s", cudaGetErrorString((cudaError_t)rc));
        return DSPB_OK;
    }
    if (mem_kind != DSPB_MEM_HOST) return fail(DSPB_ERR_INVALID, "mem_kind must be DSPB_MEM_DEVICE or DSPB_MEM_HOST");
    float *din = nullptr, *dout = nullptr;
    CUDA_TRY(cudaMallocAsync(&din, in_bytes, st));
    CUDA_TRY(cudaMallocAsync(&dout, out_bytes, st));
    CUDA_TRY(cudaMemcpyAsync(din, src, in_bytes, cudaMemcpyHostToDevice, st));
    int rc = fold ? dspb::launch_fold_stereo(din, dout, total, st) : dspb::launch_dup_stereo(din, dout, total, st);
    if (rc) return fail(DSPB_ERR_CUDA, "boundary kernel launch: %s", cudaGetErrorString((cudaError_t)rc));
    CUDA_TRY(cudaMemcpyAsync(dst, dout, out_bytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaFreeAsync(din, st));
    CUDA_TRY(cudaFreeAsync(dout, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return DSPB_OK;
}
// ---- 48 kHz -> device-rate converter + duplicate (devices.rs:443-500, 550-556; dasp Converter + Sinc<[f32; 16]>) -------------
int dspb_resample_dup_stereo(dspb_engine* e, const float* mono, float* interleaved, int64_t n_in, int64_t n_out, double target_hz,
                             int mem_kind, void* cuda_stream, int64_t* consumed) {
    if (!e || (n_in > 0 && !mono) || (n_out > 0 && !interleaved)) return fail(DSPB_ERR_INVALID, "null argument");
    if (n_in < 0 || n_out < 0 || !(target_hz > 0.0)) return fail(DSPB_ERR_INVALID, "n_in, n_out must be >= 0 and target_hz > 0");
    if (n_out > (1ll << 30) || n_in > (1ll << 30)) return fail(DSPB_ERR_INVALID, "call too long");
    if (e->plan_only) return fail(DSPB_ERR_CUDA, "engine was created with device = -1 (planning only): no CUDA device, no CPU fallback");
    CUDA_TRY(cudaSetDevice(e->cfg.device));
    auto& rs = e->rs;
    const int C = e->cfg.channels;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (!rs.hist[0].p || rs.target_hz != target_hz) {  // a fresh Converter: value 0, ring of zeros, idx 0 (devices.rs:550-556)
        for (auto& h : rs.hist) {
            int r = h.alloc((size_t)C * 16 * 4, true, false);
            if (r) return r;
        }
        rs.target_hz = target_hz;
        rs.value = 0.0;
        rs.idx = 0;
        rs.cur = 0;
    }
    // Converter::next control flow, once for all channels (f64, the arithmetic of dasp_signal 0.11.0 interpolate.rs)
    const double ratio = (double)e->cfg.sample_rate / target_hz;  // from_hz_to_hz: source_hz / target_hz
    std::vector<int32_t> meta((size_t)n_out * 2);
    std::vector<double> w((size_t)n_out * 16);
    int64_t pushed = 0;
    double value = rs.value;
    int idx = rs.idx;
    for (int64_t m = 0; m < n_out; m++) {
        while (value >= 1.0) {
            pushed++;
            if (idx < 8) idx++;
            value -= 1.0;
        }
        meta[2 * m] = (int32_t)pushed;
        meta[2 * m + 1] = idx;
        const double phil = value, phir = 1.0 - value;
        for (int n = 0; n < 8; n++) {  // Sinc::interpolate's window: sinc(a) * (0.5 + 0.5 cos(a / depth)), depth = 8
            double a = M_PI * (phil + (double)n);
            w[16 * m + 2 * n] = (a == 0.0 ? 1.0 : std::sin(a) / a) * (0.5 + 0.5 * std::cos(a / 8.0));
            a = M_PI * (phir + (double)n);
            w[16 * m + 2 * n + 1] = (a == 0.0 ? 1.0 : std::sin(a) / a) * (0.5 + 0.5 * std::cos(a / 8.0));
        }
        value += ratio;
    }
    if (pushed > (1ll << 30)) return fail(DSPB_ERR_INVALID, "call too long");
    if ((size_t)n_out > rs.cap) {
        int r = rs.meta.alloc((size_t)n_out * 8, false, false);
        if (r) return r;
        r = rs.w.alloc((size_t)n_out * 128, false, false);
        if (r) return r;
        rs.cap = (size_t)n_out;
    }
    const float* din = mono;
    float* dout = interleaved;
    float *tin = nullptr, *tout = nullptr;
    if (mem_kind == DSPB_MEM_HOST) {
        if (n_in) CUDA_TRY(cudaMallocAsync(&tin, (size_t)C * n_in * 4, st));
        if (n_out) CUDA_TRY(cudaMallocAsync(&tout, (size_t)C * n_out * 8, st));
        if (n_in) CUDA_TRY(cudaMemcpyAsync(tin, mono, (size_t)C * n_in * 4, cudaMemcpyHostToDevice, st));
        din = tin;
        dout = tout;
    } else if (mem_kind != DSPB_MEM_DEVICE) {
        return fail(DSPB_ERR_INVALID, "mem_kind must be DSPB_MEM_DEVICE or DSPB_MEM_HOST");
    }
    if (n_out) {
        // the plan arrays are pageable: these copies return once the data is staged, so the vectors may die with this call
        CUDA_TRY(cudaMemcpyAsync(rs.meta.p, meta.data(), (size_t)n_out * 8, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(rs.w.p, w.data(), (size_t)n_out * 128, cudaMemcpyHostToDevice, st));
    }
    int rc = dspb::launch_resample_dup(din, n_in, rs.hist[rs.cur].p, rs.hist[rs.cur ^ 1].p, rs.meta.p, reinterpret_cast<const double*>(rs.w.p),
                                       dout, n_out, pushed, C, st);
    if (rc) return fail(DSPB_ERR_CUDA, "resampler kernel launch: %s", cudaGetErrorString((cudaError_t)rc));
    if (mem_kind == DSPB_MEM_HOST) {
        if (n_out) CUDA_TRY(cudaMemcpyAsync(interleaved, tout, (size_t)C * n_out * 8, cudaMemcpyDeviceToHost, st));
        if (tin) CUDA_TRY(cudaFreeAsync(tin, st));
        if (tout) CUDA_TRY(cudaFreeAsync(tout, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    rs.cur ^= 1;
    rs.value = value;
    rs.idx = idx;
    if (consumed) *consumed = std::min<int64_t>(pushed, n_in);  // CountingSignal::index stops at the end of its buffer
    return DSPB_OK;
}

int dspb_fold_stereo(dspb_engine* e, const float* interleaved, float* mono, int64_t n_frames, int mem_kind, void* cuda_stream) {
    return boundary_step(e, interleaved, mono, n_frames, mem_kind, cuda_stream, true);
}
int dspb_dup_stereo(dspb_engine* e, const float* mono, float* interleaved, int64_t n_frames, int mem_kind, void* cuda_stream) {
    return boundary_step(e, mono, interleaved, n_frames, mem_kind, cuda_stream, false);
}

int dspb_node_get_i64(dspb_engine* e, int64_t node_id, const char* key, int64_t* out) {
    if (!e || !key || !out) return fail(DSPB_ERR_INVALID, "null argument");
    if (!strcmp(key, "kernel_launches")) { *out = e->last_launches; return DSPB_OK; }
    if (!strcmp(key, "n_segments")) { *out = (int64_t)e->steps.size(); return DSPB_OK; }
    int i = e->find(node_id);
    if (i < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown node id %lld", (long long)node_id);
    Node& n = *e->nodes[i];
    if (!strcmp(key, "n_inputs")) { *out = (int64_t)kNodeTypes[n.type].ins.size(); return DSPB_OK; }
    if (!strcmp(key, "n_outputs")) { *out = (int64_t)kNodeTypes[n.type].outs.size(); return DSPB_OK; }
    if (!strcmp(key, "delay_samples") && n.type == T_REVERB) { *out = n.D; return DSPB_OK; }
    if (!strcmp(key, "ring_pos") && n.type == T_REVERB) { *out = n.pos; return DSPB_OK; }
    if (!strcmp(key, "n_taps") && n.type == T_FIR) { *out = (int64_t)n.taps.size(); return DSPB_OK; }
    return fail(DSPB_ERR_UNKNOWN_PORT, "node type '%s' has no key '%s'", kNodeTypes[n.type].cfg_name, key);
}

int dspb_node_port_index(dspb_engine* e, int64_t node_id, const char* port, int is_output, int32_t* out) {
    if (!e || !port || !out) return fail(DSPB_ERR_INVALID, "null argument");
    int i = e->find(node_id);
    if (i < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown node id %lld", (long long)node_id);
    const NodeType& nt = kNodeTypes[e->nodes[i]->type];
    int p = port_index(is_output ? nt.outs : nt.ins, port);
    if (p < 0) return fail(DSPB_ERR_UNKNOWN_PORT, "node type '%s' has no %s port '%s'", nt.cfg_name, is_output ? "output" : "input", port);
    *out = p;
    return DSPB_OK;
}

int dspb_profile_enable(dspb_engine* e, int on) {
    if (!e) return fail(DSPB_ERR_INVALID, "null engine");
    e->prof_on = on != 0;
    return DSPB_OK;
}

int dspb_profile_read(dspb_engine* e, double* ms_total, int64_t* rounds, int cap) {
    if (!e) return fail(DSPB_ERR_INVALID, "null engine");
    if (!e->plan_only) CUDA_TRY(cudaDeviceSynchronize());
    for (int i = 0; i < cap; i++) {
        if (ms_total) ms_total[i] = 0.0;
        if (rounds) rounds[i] = 0;
    }
    for (auto& r : e->prof) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, r.a, r.b);
        if (r.step < cap) {
            if (ms_total) ms_total[r.step] += ms;
            if (rounds) rounds[r.step] += 1;
        }
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    e->prof.clear();
    return (int)e->steps.size();
}

// debug aid (not part of the public header): phase timing of the warp-specialised kernel, see fused_chain.cu
int dspb_debug_ws_timing(long long* out8, int clear) { return dspb::ws_timing_read(out8, clear != 0); }

int64_t dspb_describe_plan(dspb_engine* e, char* buf, int64_t cap) {
    if (!e) return 0;
    std::string s;
    char b[128];
    snprintf(b, sizeof b, "plan: %d channels, %zu step(s)\n", e->cfg.channels, e->steps.size());
    s += b;
    int k = 0;
    for (auto& st : e->steps) {
        snprintf(b, sizeof b, "[%d] ", k++);
        s += b;
        s += st.text;
    }
    if (buf && cap > 0) {
        size_t n = std::min<size_t>(s.size(), (size_t)cap - 1);
        memcpy(buf, s.data(), n);
        buf[n] = 0;
    }
    return (int64_t)s.size() + 1;
}

// ---- single-node call: SimpleNode::process on pre-averaged port buffers ----------------------------------------
// Implemented with a cached one-node sub-engine lowered in "raw ports" mode (no fan-in arithmetic): the node
// keeps its own state across dspb_node_process calls, independent of the graph-level dspb_process state.
int dspb_node_process(dspb_engine* e, int64_t node_id, const float* const* port_inputs, const uint8_t* present,
                      float* const* port_outputs, int64_t n, int mem_kind, void* stream) {
    if (!e || !port_outputs) return fail(DSPB_ERR_INVALID, "null argument");
    if (e->plan_only) return fail(DSPB_ERR_CUDA, "planning-only engine (device -1) cannot process: there is no CPU fallback");
    const int i = e->find(node_id);
    if (i < 0) return fail(DSPB_ERR_UNKNOWN_NODE, "unknown node id %lld", (long long)node_id);
    Node& src = *e->nodes[i];
    const NodeType& nt = kNodeTypes[src.type];
    if (src.type == T_INPUT || src.type == T_OUTPUT) return fail(DSPB_ERR_INVALID, "terminals have no process()");
    const int n_in = (int)nt.ins.size(), n_out = (int)nt.outs.size();
    uint32_t mask = 0;
    for (int p = 0; p < n_in; p++)
        if (port_inputs && port_inputs[p] && (!present || present[p])) mask |= 1u << p;
    for (int q = 0; q < n_out; q++)
        if (!port_outputs[q]) return fail(DSPB_ERR_INVALID, "null output buffer for port '%s'", nt.outs[q]);
    auto& ne = e->node_engines[node_id];
    if (!ne.e || ne.present_mask != mask) {
        delete ne.e;
        ne.e = nullptr;
        dspb_engine* sub = nullptr;
        int r = dspb_engine_create(&e->cfg, &sub);
        if (r) return r;
        sub->raw_ports = true;
        ne.e = sub;
        ne.present_mask = mask;
        if ((r = dspb_node_add(sub, nt.cfg_name, 0))) return r;
        for (int p = 0; p < n_in; p++)
            if (mask & (1u << p)) {
                if ((r = dspb_node_add(sub, "input", 1000 + p))) return r;
                if ((r = dspb_link(sub, 1000 + p, "out", 0, nt.ins[p]))) return r;
            }
        for (int q = 0; q < n_out; q++) {
            if ((r = dspb_node_add(sub, "output", 2000 + q))) return r;
            if ((r = dspb_link(sub, 0, nt.outs[q], 2000 + q, "in"))) return r;
        }
        Node& dst = *sub->nodes[0];
        dst.f32 = src.f32; dst.f32_pc = src.f32_pc; dst.enums = src.enums; dst.taps = src.taps; dst.D = src.D;
        copy_fir_pc(dst, src);
        memcpy(dst.bq, src.bq, sizeof dst.bq);
        if ((r = dspb_compile(sub))) return r;
    }
    dspb_engine* sub = ne.e;
    Node& dst = *sub->nodes[0];
    // setters on the parent node since the last call: same side effects as on the parent (after_settings_change)
    const bool taps_changed = dst.taps != src.taps || dst.fir_bank != src.fir_bank || dst.fir_set != src.fir_set;
    if (dst.f32 != src.f32 || dst.f32_pc != src.f32_pc || dst.enums != src.enums || taps_changed || dst.D != src.D) {
        const bool f32_changed = dst.f32 != src.f32 || dst.f32_pc != src.f32_pc || dst.D != src.D;
        dst.f32 = src.f32; dst.f32_pc = src.f32_pc; dst.enums = src.enums; dst.taps = src.taps; dst.D = src.D;
        copy_fir_pc(dst, src);
        memcpy(dst.bq, src.bq, sizeof dst.bq);
        CUDA_TRY(cudaSetDevice(e->cfg.device));
        if (f32_changed && dst.type == T_BIQUAD && dst.state.p) CUDA_TRY(cudaMemset(dst.state.p, 0, dst.state.bytes));
        if (f32_changed && dst.type == T_REVERB) dst.ring_dirty = true;
        if (taps_changed) dst.fir_dirty = true;
        sub->lowered = false;
    }
    std::vector<const float*> ins;
    for (int p = 0; p < n_in; p++)
        if (mask & (1u << p)) ins.push_back(port_inputs[p]);
    return dspb_process(sub, ins.data(), port_outputs, n, mem_kind, stream);
}

// ---- saved-graph JSON (runtime.rs:44-48, 94-123, 560-564, 606-612; lib.rs:266-340) ------------------------------
int dspb_load_graph_json(dspb_engine* e, const char* text) {
    if (!e || !text) return fail(DSPB_ERR_INVALID, "null argument");
    if (!e->nodes.empty()) return fail(DSPB_ERR_GRAPH, "dspb_load_graph_json needs an empty engine");
    jsonmin::Value doc;
    std::string perr;
    if (!jsonmin::parse(text, doc, perr)) return fail(DSPB_ERR_PARSE, "graph JSON: %s", perr.c_str());
    const jsonmin::Value* nodes = doc.get("nodes");
    const jsonmin::Value* links = doc.get("links");
    if (!nodes || !nodes->is_array() || !links || !links->is_array()) return fail(DSPB_ERR_PARSE, "graph JSON: need 'nodes' and 'links' arrays");
    std::map<std::pair<int64_t, int64_t>, std::pair<std::string, bool>> port_names;  // (node, PortId) -> (name, is_output)
    // GUI-only sinks (nodes/mod.rs:111-122: oscilloscope, spectrogram, pitch read-out): no output port, no effect on any
    // audio value.  They are dropped together with the links into them, so a graph saved with a scope attached loads.
    std::set<int64_t> dropped_sinks;
    auto is_gui_sink = [](const std::string& t) { return t == "wave_view" || t == "spectrogram" || t == "pitch"; };
    for (const auto& nv : nodes->arr) {
        const jsonmin::Value* id = nv.get("id");
        const jsonmin::Value* tn = nv.get("typename");
        const jsonmin::Value* cfg = nv.get("cfg");
        if (!id || !id->is_number() || !tn || !tn->is_string() || !cfg || !cfg->is_object()) return fail(DSPB_ERR_PARSE, "graph JSON: malformed node entry");
        const int64_t nid = (int64_t)id->num;
        if (is_gui_sink(tn->str)) { dropped_sinks.insert(nid); continue; }
        if (tn->str == "muff")
            return fail(DSPB_ERR_UNKNOWN_NODE, "typename 'muff' (nodes/muff.rs) is not supported: its arithmetic lives in the private "
                                               "GPL crate dsp-stuff-gpl@170f168, which is not part of the reference tree");
        int r = dspb_node_add(e, tn->str.c_str(), nid);
        if (r) return r;
        Node& n = *e->nodes.back();
        const bool terminal = n.type == T_INPUT || n.type == T_OUTPUT;
        for (const auto& kv : cfg->obj) {
            const std::string& k = kv.first;
            const jsonmin::Value& v = kv.second;
            if (k == "id" || k == "file_name") continue;
            // InputConfig / OutputConfig (nodes/input.rs:33-38, nodes/output.rs:33-38): the cpal host and device names.
            // The engine's terminals bind to dspb_process buffers instead of audio devices.
            if (terminal && (k == "selected_host" || k == "selected_device")) continue;
            if (k == "inputs" || k == "outputs") {
                if (!v.is_object()) return fail(DSPB_ERR_PARSE, "graph JSON: '%s' must be a name -> PortId map", k.c_str());
                for (const auto& pv : v.obj) port_names[{nid, (int64_t)pv.second.num}] = {pv.first, k == "outputs"};
                continue;
            }
            if (k == "taps") {
                if (!v.is_array()) return fail(DSPB_ERR_PARSE, "graph JSON: taps must be an array");
                std::vector<double> t;
                for (const auto& x : v.arr) t.push_back(x.num);
                r = dspb_node_set_taps(e, nid, t.data(), (int64_t)t.size());
            } else if (v.is_string()) {
                r = dspb_node_set_enum(e, nid, k.c_str(), v.str.c_str());
            } else if (v.is_number()) {
                r = dspb_node_set_f32(e, nid, k.c_str(), (float)v.num);
            } else {
                continue;
            }
            if (r) return r;
        }
        // restore() runs after_settings_change unconditionally (lib.rs:319-336)
        if (n.type == T_REVERB) { n.D = reverb_delay(n.f32[0], e->cfg.sample_rate, e->cfg.ring_granule); n.ring_dirty = true; }
        if (n.type == T_BIQUAD) biquad_regenerate(n);
    }
    for (const auto& lv : links->arr) {
        const jsonmin::Value* lhs = lv.get("lhs");
        const jsonmin::Value* rhs = lv.get("rhs");
        if (!lhs || !rhs || !lhs->is_array() || !rhs->is_array() || lhs->arr.size() != 2 || rhs->arr.size() != 2)
            return fail(DSPB_ERR_PARSE, "graph JSON: malformed link entry");
        const int64_t sn = (int64_t)lhs->arr[0].num, sp = (int64_t)lhs->arr[1].num;
        const int64_t dn = (int64_t)rhs->arr[0].num, dp = (int64_t)rhs->arr[1].num;
        if (dropped_sinks.count(dn)) continue;  // link into a GUI sink
        auto a = port_names.find({sn, sp});
        auto b = port_names.find({dn, dp});
        if (a == port_names.end() || b == port_names.end() || !a->second.second || b->second.second)
            return fail(DSPB_ERR_UNKNOWN_PORT, "graph JSON: link refers to an unknown PortId");
        int r = dspb_link(e, sn, a->second.first.c_str(), dn, b->second.first.c_str());
        if (r) return r;
    }
    return dspb_compile(e);
}

}  // extern "C"
