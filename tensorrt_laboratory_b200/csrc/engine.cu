// C ABI implementation (include/b200infer.h): plan loader, activation-arena planner, per-batch launch
// plans (TMA tensor maps, tile selection), CUDA-graph-cached enqueue.
//
// Reference counterparts: trtlab/tensorrt/src/runtime.cc:62-143 (deserialize + weight allocation through
// the IGpuAllocator hook), src/model.cc:76-116 (binding metadata), src/execution_context.cc:9-27,
// src/workspace.cc:36-57 (setDeviceMemory, enqueueV2, graph capture).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200infer.h"
#include "kernels.h"
#include "plan_format.h"

#include "b2_internal.h"

namespace b2i {
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
}  // namespace b2i

namespace {
using b2i::fail;
using b2i::g_err;

#define B2_CUDA(expr)                                                                         \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return fail(B2_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)

// ---- driver entry points for tensor-map encoding (no link-time libcuda dependency) ------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode_tiled = nullptr;
EncodeIm2colFn g_encode_im2col = nullptr;
int g_driver_version = 0;
std::once_flag g_driver_once;
int g_driver_status = 0;

int load_driver_entry_points() {
    std::call_once(g_driver_once, [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) {
            g_driver_status = 1;
            return;
        }
        g_encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
        fn = nullptr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q) != cudaSuccess || !fn) {
            g_driver_status = 2;
            return;
        }
        g_encode_im2col = reinterpret_cast<EncodeIm2colFn>(fn);
        cudaDriverGetVersion(&g_driver_version);
    });
    return g_driver_status;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
constexpr size_t kSplitWorkspaceBytes = 12u << 20;  // bounds tiles*splits*128*BN*4 (see pick_conv_config)
constexpr int kMaxSplitTiles = 4096;                 // tile counters per context

int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v ? atoi(v) : dflt;
}

struct Tensor {
    std::string name;
    uint32_t kind, h, w, c, c_phys;
    int binding;
    float scale = 0.f;      // > 0: int8 tensor (INT8 engines), real value = q * scale
    size_t item_bytes = 0;  // bytes per batch item
    size_t offset = 0;      // arena offset (binding < 0)
    int def = -1, last_use = -1;
};

struct Op {
    b2plan::OpRec r;
    std::string name;
    // >= 0: this op's only consumer is the residual input of op `side_join`, and nothing in between depends on it (the
    // shortcut convolution of a ResNet "a" block): it may run on a forked stream, concurrently with the ops up to there
    int side_join = -1;
    // conv geometry with the "0 = square" defaults resolved
    int kh() const { return int(r.k); }
    int kw() const { return int(r.kw ? r.kw : r.k); }
    int sh() const { return int(r.stride); }
    int sw() const { return int(r.kw ? r.stride_w : r.stride); }
    int ph() const { return int(r.pad_); }
    int pw_lo() const { return int(r.kw ? r.pad_w_lo : r.pad_); }
    int pw_hi() const { return int(r.kw ? r.pad_w_hi : r.pad_); }
    double algo_k() const { return r.ceil_mode ? double(r.ceil_mode) : double(r.cin) * r.taps; }
};

struct Binding {
    std::string name;
    bool is_input;
    int dtype;
    int tensor;
    int nd;
    int32_t dims[8];
    size_t item_bytes;
    b2k::U8Norm norm{};  // B2_DT_UINT8 input: source geometry, crop and normalisation (from the plan's InputNormRec)
};

enum LKind { L_INPUT_CAST, L_CONV_TC, L_CONV_SIMT, L_MAXPOOL, L_AVGPOOL, L_FC, L_SOFTMAX, L_OUTPUT_CAST, L_NET, L_TAIL, L_QUANTIZE, L_CONV_I8, L_AVGPOOL_I8, L_OUTPUT_CAST_I8 };

// A run of consecutive tcgen05 convolution layers executed by ONE persistent kernel (net_kernel.cu): device-side layer
// table, dependency ranges and arrival counters live in one allocation owned by the plan.
struct NetRun {
    b2k::NetArgs args{};
    int ctas = 0;
    int first_op = 0, last_op = 0;
    void* d_blob = nullptr;
    ~NetRun() {
        if (d_blob) cudaFree(d_blob);
    }
};

struct Launch {
    LKind kind;
    std::string name;
    double flops = 0, bytes = 0;
    b2k::ConvLaunch conv;
    b2k::SimtConvArgs simt;
    const void* in = nullptr;
    void* out = nullptr;
    const void* w = nullptr;
    const float* bias = nullptr;
    int in_binding = -1, out_binding = -1;
    int src_dtype = B2_DT_FLOAT;  // input cast: dtype of the binding (fp32, fp16 or uint8 HWC)
    b2k::U8Norm norm{};           // input cast of a uint8 binding: passed to the kernel by value
    int max_blocks = 0;     // input cast: grid cap (option input_ctas), 0 = one thread per element group
    int side_join = -1;     // see Op::side_join (launch index == op index)
    std::shared_ptr<NetRun> net;  // L_NET
    b2k::TailArgs tail{};         // L_TAIL: pool + fc + softmax in one launch (out = the output binding)
    b2k::I8ConvLaunch i8{};       // L_CONV_I8
    float qscale = 0.f;           // L_QUANTIZE: 1/s; L_AVGPOOL_I8: s/HW; L_OUTPUT_CAST_I8: s
    int C_in_phys = 0;            // L_QUANTIZE / L_AVGPOOL_I8: channel pitch of the source tensor
    bool net_member = false;      // L_CONV_TC that build_plan folds into an L_NET launch
    int N = 0, C = 0, H = 0, W = 0, C_phys = 0, Ho = 0, Wo = 0, k = 0, stride = 0, pad = 0, K = 0, Cout = 0;
};

// A maximal run of launches that touch no binding: captured ONCE per plan (= per context, arena and batch) into a CUDA
// graph that is valid for any binding pointers.  Launches that read or write a binding (the input cast, the classifier
// tail, output casts) are issued directly around it, so the engine never captures or instantiates per Buffers object.
struct Segment {
    int begin = 0, end = 0;  // [begin, end) launch indices
    bool graphable = false;
    cudaGraphExec_t exec = nullptr;
};
// One kernel node of the plan's graph that reads or writes a binding: its pointer argument is re-pointed at the caller's
// buffer before every launch (cudaGraphExecKernelNodeSetParams) -- the graph itself is captured and instantiated once.
struct BindPatch {
    int launch = -1;              // index into Plan::launches
    cudaGraphNode_t node = nullptr;
    cudaKernelNodeParams np{};    // func / grid / block / smem as captured
    std::vector<void*> params;    // argument pointer array handed to the driver (entries point into the graph's storage ...)
    int n_params = 0;
    int in_index = -1, out_index = -1;  // ... except these, which point at in_value / out_value below
    void* in_value = nullptr;
    void* out_value = nullptr;
    b2k::TailArgs tail{};         // fused tail: the whole argument struct is replaced (its `out` field is the binding)
    bool is_tail = false;
};
struct Plan {
    int batch = 0;
    bool has_net = false;  // contains a persistent network kernel: a handful of launches, replayed directly (no graph)
    std::vector<Launch> launches;
    std::vector<Segment> segments;   // graph mode 3: binding-free runs as graphs, binding-dependent launches direct
    bool graph_failed = false;       // the plan could not be captured as one patchable graph: segments instead
    cudaGraph_t graph = nullptr;     // graph mode 1 (default): the whole plan, binding arguments patched per launch
    cudaGraphExec_t exec = nullptr;
    std::vector<BindPatch> patches;
    ~Plan() {
        for (Segment& sg : segments)
            if (sg.exec) cudaGraphExecDestroy(sg.exec);
        if (exec) cudaGraphExecDestroy(exec);
        if (graph) cudaGraphDestroy(graph);
    }
};

}  // namespace

struct ConvConfig {
    int bn, stages, splits;
    double est_us;
    int sps = 1;  // 64-wide K sub-blocks per pipeline stage
    int ws = 0;   // > 0: persistent warp-specialised kernel with this many CTAs
    int cn = 1;   // CTAs per cluster along N sharing the activation tile by TMA multicast (1 = no cluster)
    int halo = 0; // 1: 3x3 halo kernel (input block resident in smem, taps = shifted views)
};
// A pipeline deeper than the K loop is pure shared-memory cost: admit depths up to the smallest instantiated one
// that covers the loop (or the deepest available when none does).
static bool stage_depth_useful(int bn, int kb, int st, int kpc) {
    const int stgs[4] = {1, 2, 4, 8};
    int cover = 0, deepest = 0;
    for (int s2 : stgs) {
        if (!b2k::conv_config_exists(bn, kb, s2)) continue;
        deepest = s2;
        if (!cover && s2 >= kpc) cover = s2;
    }
    return st <= (cover ? cover : deepest);
}


constexpr int kHaloStagesTag = 2;  // reported pipeline depth of the halo kernel (its A ring)

struct b2_runtime {
    b2_alloc_fn alloc = nullptr;
    b2_free_fn free_ = nullptr;
    void* user = nullptr;
};

struct b2_engine {
    b2_runtime* rt = nullptr;
    b2_alloc_fn alloc = nullptr;  // snapshot of the runtime's allocator at deserialize time
    b2_free_fn free_ = nullptr;
    void* alloc_user = nullptr;
    std::string name;
    int precision = 0, max_batch = 0;
    std::vector<Tensor> tensors;
    std::vector<Op> ops;
    std::vector<Binding> bindings;
    uint8_t* d_payload = nullptr;
    size_t payload_bytes = 0;
    size_t arena_bytes = 0;
    size_t act_bytes = 0;
    int device = -1;
    bool inspect_only = false;
    double flops_per_item = 0;
    std::mutex tune_mutex;
    std::mutex tune_run_mutex;  // serialises on-device tactic timing across contexts of this engine
    std::map<std::pair<int, int>, ConvConfig> tuned;  // (op index, batch) -> measured-best configuration
    bool tune_cache_loaded = false;
    std::map<int, float> requant_r;  // INT8 convs: op index -> r = fl(s_res / s_out) (read from the plan's requantisation block)
    bool tactics_from_plan = false;  // the blob carried a tactic table: nothing left to tune
    bool tuned_at_load = false;      // b2_engine_tune has run
    bool half() const { return precision != B2_PREC_FP32; }  // fp16 storage and kernels (INT8 engines: their fp16 part)
    bool int8() const { return precision == B2_PREC_INT8; }
};

struct b2_context {
    b2_engine* e = nullptr;
    uint8_t* scratch = nullptr;
    // Launch plans (TMA maps embed arena addresses) and their captured graph segments are cached PER SCRATCH pointer:
    // the reference pairs a pooled IExecutionContext with whichever pooled activation block the request drew
    // (inference_manager.cc:254-273), so the same context may see several scratch pointers over its life.
    struct ScratchState {
        std::map<int, std::unique_ptr<Plan>> plans;
    };
    std::map<uint8_t*, ScratchState> states;
    ScratchState* cur = nullptr;
    int* d_counters = nullptr;  // split-K tile arrival counters (always zero between launches)
    int use_graph = 1;
    int force_simt = 0;
    int force_im2col = 0;
    int force_bn = 0;
    int force_stages = 0;
    int force_splits = 0;
    int force_sps = 0;
    int force_halo = 0; // 1: the 3x3 halo kernel wherever it applies, -1: never
    int force_cn = 0;   // > 0: this cluster size wherever it divides the N-tile count, -1: never cluster
    int force_ws = 0;   // 1: only the persistent warp-specialised tactic where it applies, -1: never
    int pdl_trigger = 1;
    int no_pack = 0;    // reserved (packed plans cannot fall back to the tensor-map weight path)
    int no_fold = 0;    // 1: run the stem through the generic 8-channel tap path instead of the row-folded one
    int autotune = 4;  // 0 off (cost model), 1 latency mode, N>=2 throughput mode over N streams
    int fork = 0;      // 1: run side branches (Op::side_join) on a forked stream / a parallel graph branch.  Off by default:
                       // measured neutral on B200 (0.476 ms either way, 4-context throughput within noise) -- the fork and
                       // join turn the programmatic (PDL) edges around them into full dependencies, which eats the overlap
    int net = 0;       // 1: runs of 64-channel-block tcgen05 convolutions execute as ONE persistent kernel (net_kernel.cu).
                       // Opt-in: bit-identical, but measured slower than the per-layer kernels at batch 8 (profiles/README.md, r2a-c)
    int net_ctas = 0;  // CTAs of that kernel (0 = one per SM); a server running N contexts gives each about 148 / N
    int net_bn = 0;    // force its N tile (64 / 128); 0 = 128 wherever the channel count allows
    int net_stages = 0;  // force its shared-memory ring depth (2..4); 0 = the deepest that lets two CTAs share an SM
    int i8_bn = 0;       // INT8 convolutions: force the N tile (128 / 256); 0 = 128
    int i8_stages = 0;   // ... and the shared-memory ring depth (2..4); 0 = by rule
    int fuse_tail = 1;   // global average pool + FC + softmax as one launch (tail_f16_kernel)
    int input_ctas = 0;  // grid cap of the input cast (0 = none); set when the input binding is read over PCIe (zero-copy)
    int* d_tail_ctrl = nullptr;  // its ticket / arrival counters (zero between launches)
    cudaStream_t side = nullptr;
    cudaEvent_t fork_ev = nullptr, join_ev = nullptr;
};

namespace {

// ---- plan parsing -----------------------------------------------------------------------------
std::string fixed_str(const char* p, size_t n) {
    size_t len = 0;
    while (len < n && p[len]) ++len;
    return std::string(p, len);
}

int parse_blob(const void* blob, size_t nbytes, b2_engine* e, const uint8_t** payload) {
    using namespace b2plan;
    if (!blob || nbytes < sizeof(Header)) return fail(B2_EINVAL, "plan: blob too small (%zu bytes)", nbytes);
    const uint8_t* base = static_cast<const uint8_t*>(blob);
    Header h;
    memcpy(&h, base, sizeof h);
    if (memcmp(h.magic, kMagic, 8) != 0) return fail(B2_EINVAL, "plan: bad magic (not a B2ENGINE blob)");
    if (h.version != kVersion) return fail(B2_EINVAL, "plan: version %u, this library reads %u", h.version, kVersion);
    if (h.precision > 2) return fail(B2_EINVAL, "plan: unknown precision %u", h.precision);
    if (h.max_batch == 0 || h.max_batch > 4096) return fail(B2_EINVAL, "plan: bad max_batch %u", h.max_batch);
    const size_t tbl = sizeof(Header) + size_t(h.n_tensors) * sizeof(TensorRec) + size_t(h.n_ops) * sizeof(OpRec) +
                       size_t(h.n_bindings) * sizeof(BindingRec);
    // (overflow-safe: a > n || b > n - a instead of a + b > n)
    if (tbl > nbytes || h.payload_offset < tbl || h.payload_offset > nbytes || h.payload_bytes > nbytes - h.payload_offset)
        return fail(B2_EINVAL, "plan: truncated (tables %zu, payload %llu+%llu, blob %zu)", tbl,
                    (unsigned long long)h.payload_offset, (unsigned long long)h.payload_bytes, nbytes);
    e->name = fixed_str(h.name, 64);
    e->precision = h.precision;
    e->max_batch = h.max_batch;
    e->payload_bytes = h.payload_bytes;
    const size_t elt = h.precision == B2_PREC_FP32 ? 4 : 2;
    const uint8_t* p = base + sizeof(Header);
    for (uint32_t i = 0; i < h.n_tensors; ++i, p += sizeof(TensorRec)) {
        TensorRec r;
        memcpy(&r, p, sizeof r);
        Tensor t;
        t.name = fixed_str(r.name, 64);
        t.kind = r.kind;
        t.h = r.h, t.w = r.w, t.c = r.c, t.c_phys = r.c_phys;
        t.binding = r.binding;
        t.scale = h.precision == B2_PREC_INT8 ? r.scale : 0.f;
        if (!(t.scale >= 0.f) || (t.scale > 0.f && (r.kind != T_ACT || r.c_phys % 128)))
            return fail(B2_EINVAL, "plan: tensor %s has a bad INT8 scale / layout", t.name.c_str());
        if (r.kind == T_ACT) {
            if (r.c_phys < r.c || r.h == 0 || r.w == 0) return fail(B2_EINVAL, "plan: tensor %s has bad dims", t.name.c_str());
            t.item_bytes = size_t(r.h) * r.w * r.c_phys * (t.scale > 0.f ? 1 : elt);
        } else if (r.kind == T_VEC) {
            t.item_bytes = size_t(r.c) * 4;
        } else {
            return fail(B2_EINVAL, "plan: tensor %s has unknown kind %u", t.name.c_str(), r.kind);
        }
        if (t.binding >= int(h.n_bindings)) return fail(B2_EINVAL, "plan: tensor %s binding out of range", t.name.c_str());
        e->tensors.push_back(t);
    }
    auto tensor_ok = [&](int idx, bool optional) { return (optional && idx == -1) || (idx >= 0 && idx < int(h.n_tensors)); };
    for (uint32_t i = 0; i < h.n_ops; ++i, p += sizeof(OpRec)) {
        Op op;
        memcpy(&op.r, p, sizeof(OpRec));
        op.name = fixed_str(op.r.name, 64);
        const OpRec& r = op.r;
        if (r.type > OP_QUANTIZE) return fail(B2_EINVAL, "plan: op %s has unknown type %u", op.name.c_str(), r.type);
        const bool in_opt = r.type == OP_INPUT_CAST, out_opt = r.type == OP_OUTPUT_CAST;
        if (!tensor_ok(r.in, in_opt) || !tensor_ok(r.out, out_opt) || !tensor_ok(r.res, true))
            return fail(B2_EINVAL, "plan: op %s references a missing tensor", op.name.c_str());
        if ((r.type == OP_INPUT_CAST || r.type == OP_OUTPUT_CAST) && (r.binding < 0 || r.binding >= int(h.n_bindings)))
            return fail(B2_EINVAL, "plan: cast op %s has a bad binding", op.name.c_str());
        if (r.w_off > h.payload_bytes || r.w_bytes > h.payload_bytes - r.w_off || r.b_off > h.payload_bytes ||
            r.b_bytes > h.payload_bytes - r.b_off)
            return fail(B2_EINVAL, "plan: op %s weights outside payload", op.name.c_str());
        if ((r.type == OP_MAXPOOL || r.type == OP_AVGPOOL) && (r.k == 0 || r.stride == 0))
            return fail(B2_EINVAL, "plan: pool %s has a zero window or stride", op.name.c_str());
        if (r.type == OP_MAXPOOL) {
            const Tensor& ti = e->tensors[r.in];
            const Tensor& to = e->tensors[r.out];
            if (ti.kind != T_ACT || to.kind != T_ACT || ti.c_phys != to.c_phys || to.h == 0 || to.w == 0 ||
                uint64_t(to.h - 1) * r.stride >= uint64_t(ti.h) + r.pad_ || uint64_t(to.w - 1) * r.stride >= uint64_t(ti.w) + r.pad_)
                return fail(B2_EINVAL, "plan: pool %s output dims do not fit its input", op.name.c_str());
        }
        if (r.type == OP_INPUT_CAST || r.type == OP_OUTPUT_CAST) {  // the caller's Buffers are sized from the BINDING dims
            const Tensor& tt = e->tensors[r.type == OP_INPUT_CAST ? r.out : r.in];
            if (tt.kind != T_ACT) return fail(B2_EINVAL, "plan: cast op %s needs an activation tensor", op.name.c_str());
        }
        if (r.type == OP_QUANTIZE) {
            const Tensor& ti = e->tensors[r.in];
            const Tensor& to = e->tensors[r.out];
            if (h.precision != B2_PREC_INT8 || ti.scale > 0.f || !(to.scale > 0.f) || ti.h != to.h || ti.w != to.w || ti.c != to.c)
                return fail(B2_EINVAL, "plan: quantize %s needs an fp16 input and an int8 output of the same shape", op.name.c_str());
        }
        if (r.type == OP_CONV) {
            if (r.k == 0 || r.stride == 0 || int(r.taps) != op.kh() * op.kw() || r.taps_phys < r.taps || op.sw() == 0)
                return fail(B2_EINVAL, "plan: conv %s has bad geometry", op.name.c_str());
            const bool i8 = (r.relu & 4) != 0;
            if (i8) {
                const Tensor& qi = e->tensors[r.in];
                const Tensor& qo = e->tensors[r.out];
                if (h.precision != B2_PREC_INT8 || !(qi.scale > 0.f) || !(qo.scale > 0.f) || (r.res >= 0 && !(e->tensors[r.res].scale > 0.f)) ||
                    r.cin_phys % 128 || r.cout_phys % 128 || r.taps_phys != r.taps || r.kw != 0 || !(r.relu & 2))
                    return fail(B2_EINVAL, "plan: int8 conv %s: tensors must be int8 with 128-channel rows", op.name.c_str());
                if (r.w_bytes != size_t(r.cout_phys) * r.taps_phys * r.cin_phys || r.b_bytes != (size_t(r.cout_phys) * 2 + 4) * 4)
                    return fail(B2_EINVAL, "plan: int8 conv %s weight / requantisation size mismatch", op.name.c_str());
            } else if (r.w_bytes != size_t(r.cout_phys) * r.taps_phys * r.cin_phys * elt || r.b_bytes != size_t(r.cout_phys) * 4)
                return fail(B2_EINVAL, "plan: conv %s weight size mismatch", op.name.c_str());
            if (!i8 && (e->tensors[r.in].scale > 0.f || e->tensors[r.out].scale > 0.f))
                return fail(B2_EINVAL, "plan: fp16 conv %s touches an int8 tensor", op.name.c_str());
            const Tensor& ti = e->tensors[r.in];
            const Tensor& to = e->tensors[r.out];
            if (ti.c_phys != r.cin_phys || to.c_phys != r.cout_phys || ti.c != r.cin || to.c != r.cout)
                return fail(B2_EINVAL, "plan: conv %s channel mismatch with its tensors", op.name.c_str());
            if (uint64_t(ti.h) + 2 * uint64_t(r.pad_) < r.k || int64_t(ti.w) + op.pw_lo() + op.pw_hi() < op.kw())
                return fail(B2_EINVAL, "plan: conv %s window larger than its padded input", op.name.c_str());
            const uint32_t ho = (ti.h + 2 * r.pad_ - r.k) / r.stride + 1;
            const uint32_t wo = uint32_t((int(ti.w) + op.pw_lo() + op.pw_hi() - op.kw()) / op.sw() + 1);
            if (to.h != ho || to.w != wo) return fail(B2_EINVAL, "plan: conv %s output dims mismatch", op.name.c_str());
            e->flops_per_item += 2.0 * ho * wo * r.cout * op.algo_k();
        } else if (r.type == OP_FC) {
            const Tensor& ti = e->tensors[r.in];
            const size_t K = size_t(ti.h) * ti.w * ti.c_phys;
            if (r.w_bytes != size_t(r.cout) * K * elt || r.b_bytes != size_t(r.cout) * 4)
                return fail(B2_EINVAL, "plan: fc %s weight size mismatch", op.name.c_str());
            e->flops_per_item += 2.0 * ti.h * ti.w * ti.c * r.cout;
        }
        e->ops.push_back(op);
    }
    for (uint32_t i = 0; i < h.n_bindings; ++i, p += sizeof(BindingRec)) {
        BindingRec r;
        memcpy(&r, p, sizeof r);
        Binding b;
        b.name = fixed_str(r.name, 64);
        b.is_input = r.is_input != 0;
        b.dtype = r.dtype;
        b.tensor = r.tensor;
        b.nd = r.nd;
        if (r.nd == 0 || r.nd > 8) return fail(B2_EINVAL, "plan: binding %s has bad rank", b.name.c_str());
        // fp32 is the reference's binding contract; fp16 INPUT bindings are the secondary mode of fp16 engines, uint8 HWC
        // image inputs that of fp16 and INT8 engines (both have the fp16 stem)
        if (r.dtype != B2_DT_FLOAT && !(r.dtype == B2_DT_HALF && b.is_input && h.precision == B2_PREC_FP16) &&
            !(r.dtype == B2_DT_UINT8 && b.is_input && h.precision != B2_PREC_FP32))
            return fail(B2_EINVAL, "plan: binding %s: bindings are fp32 (inputs of fp16 engines may be fp16, of fp16 / INT8 "
                                   "engines uint8)", b.name.c_str());
        if (r.dtype == B2_DT_UINT8 && r.nd != 3) return fail(B2_EINVAL, "plan: uint8 binding %s is not {H, W, C}", b.name.c_str());
        size_t n = 1;
        for (uint32_t d = 0; d < 8; ++d) {
            b.dims[d] = d < r.nd ? r.dims[d] : 0;
            if (d < r.nd) n *= size_t(r.dims[d]);
        }
        b.item_bytes = n * (r.dtype == B2_DT_UINT8 ? 1 : r.dtype == B2_DT_HALF ? 2 : 4);
        e->bindings.push_back(b);
    }
    // cast ops move a binding <-> a tensor: the caller sizes its Buffers from the BINDING dims, so the two must agree
    for (const Op& op : e->ops) {
        const OpRec& r = op.r;
        if (r.type != OP_INPUT_CAST && r.type != OP_OUTPUT_CAST) continue;
        const Binding& b = e->bindings[size_t(r.binding)];
        const Tensor& t = e->tensors[size_t(r.type == OP_INPUT_CAST ? r.out : r.in)];
        size_t n = 1;
        for (int d = 0; d < b.nd; ++d) n *= size_t(b.dims[d] > 0 ? b.dims[d] : 0);
        const bool s2d = r.type == OP_INPUT_CAST && r.k == 2;  // (its geometry is re-checked when the launch plan is built)
        const bool u8 = b.dtype == B2_DT_UINT8;
        if (b.is_input != (r.type == OP_INPUT_CAST) || (!s2d && !u8 && n != size_t(t.c) * t.h * t.w))
            return fail(B2_EINVAL, "plan: cast op %s: binding %s and tensor %s disagree", op.name.c_str(), b.name.c_str(), t.name.c_str());
        if (r.type != OP_INPUT_CAST) continue;
        if (r.b_bytes != (u8 ? sizeof(InputNormRec) : 0))
            return fail(B2_EINVAL, "plan: input cast %s: %llu normalisation bytes for a %s binding", op.name.c_str(),
                        (unsigned long long)r.b_bytes, u8 ? "uint8" : "non-uint8");
        if (!u8) continue;
        // uint8 HWC image: {src_h, src_w, C} -> the tensor's H x W crop (s2d: the tensor holds W/2 + pad_l + pad_r pairs)
        InputNormRec nr;
        memcpy(&nr, base + h.payload_offset + r.b_off, sizeof nr);  // (inside the payload: checked with the op)
        const int64_t src_h = b.dims[0], src_w = b.dims[1], C = b.dims[2];
        const int64_t H = t.h, W = s2d ? 2 * (int64_t(t.w) - int64_t(r.pad_) - int64_t(r.stride)) : int64_t(t.w);
        if (src_h < 1 || src_w < 1 || C < 1 || C > 4 || (!s2d && int64_t(t.c) != C) || t.c_phys != 8 || W < 1)
            return fail(B2_EINVAL, "plan: uint8 binding %s {%lld, %lld, %lld} does not fit tensor %s", b.name.c_str(),
                        (long long)src_h, (long long)src_w, (long long)C, t.name.c_str());
        if (int64_t(nr.crop_top) + H > src_h || int64_t(nr.crop_left) + W > src_w)
            return fail(B2_EINVAL, "plan: uint8 binding %s: crop %lldx%lld at (%u, %u) outside the %lldx%lld source", b.name.c_str(),
                        (long long)H, (long long)W, nr.crop_top, nr.crop_left, (long long)src_h, (long long)src_w);
        unsigned seen = 0;
        for (int c = 0; c < C; ++c) {
            if (nr.perm[c] >= C || (seen & (1u << nr.perm[c])))
                return fail(B2_EINVAL, "plan: uint8 binding %s: channel order is not a permutation of 0..%lld", b.name.c_str(),
                            (long long)C - 1);
            seen |= 1u << nr.perm[c];
            if (!std::isfinite(nr.mean[c]) || !std::isfinite(nr.inv_std[c]) || nr.inv_std[c] == 0.f)
                return fail(B2_EINVAL, "plan: uint8 binding %s: mean / inv_std of channel %d not finite or inv_std 0", b.name.c_str(), c);
        }
        for (int c = int(C); c < 4; ++c)  // entries past C are 0: the record agrees with the binding's channel count
            if (nr.perm[c] != 0 || nr.mean[c] != 0.f || nr.inv_std[c] != 0.f)
                return fail(B2_EINVAL, "plan: uint8 binding %s: normalisation entry %d set for a %lld-channel image", b.name.c_str(), c,
                            (long long)C);
        Binding& bm = e->bindings[size_t(r.binding)];
        bm.norm.C = int(C), bm.norm.src_h = int(src_h), bm.norm.src_w = int(src_w);
        bm.norm.top = int(nr.crop_top), bm.norm.left = int(nr.crop_left);
        for (int c = 0; c < 4; ++c) {
            bm.norm.mean[c] = c < C ? nr.mean[c] : 0.f;
            bm.norm.inv_std[c] = c < C ? nr.inv_std[c] : 0.f;
            bm.norm.perm[c] = c < C ? int(nr.perm[c]) : 0;
        }
    }
    if (h.n_tactics) {  // tactic table written by an offline tuning run (b2_engine_get_tactics -> builder.attach_tactics)
        if (h.tactics_offset > nbytes || size_t(h.n_tactics) > (nbytes - h.tactics_offset) / sizeof(TacticRec))
            return fail(B2_EINVAL, "plan: tactic table outside the blob");
        for (uint32_t i = 0; i < h.n_tactics; ++i) {
            TacticRec t;
            memcpy(&t, base + h.tactics_offset + size_t(i) * sizeof(TacticRec), sizeof t);
            if (t.op >= h.n_ops || t.batch == 0 || t.batch > h.max_batch) return fail(B2_EINVAL, "plan: tactic %u out of range", i);
            ConvConfig cfg{int(t.bn), int(t.stages), int(t.splits), 0.0, int(t.sps), int(t.ws), int(t.cn)};
            cfg.halo = int(t.halo);
            e->tuned[{int(t.op), int(t.batch)}] = cfg;
        }
        e->tactics_from_plan = true;
    }
    *payload = base + h.payload_offset;
    return B2_OK;
}

// ---- activation arena: first-fit over live intervals ------------------------------------------
void plan_arena(b2_engine* e) {
    // side branches: a conv whose output is consumed exactly once, as the residual of a later op, with at least one
    // independent op in between.  Regions do not nest or overlap.
    int busy_until = -1;
    for (size_t i = 0; i < e->ops.size(); ++i) {
        Op& op = e->ops[i];
        op.side_join = -1;
        if (int(i) <= busy_until || op.r.type != b2plan::OP_CONV || op.r.out < 0 || e->tensors[op.r.out].binding >= 0) continue;
        int consumers = 0, join = -1;
        bool as_residual_only = true;
        for (size_t k = i + 1; k < e->ops.size(); ++k) {
            const auto& rk = e->ops[k].r;
            if (rk.in == op.r.out) ++consumers, as_residual_only = false;
            if (rk.res == op.r.out) ++consumers, join = int(k);
        }
        if (consumers == 1 && as_residual_only && join > int(i) + 1) {
            op.side_join = join;
            busy_until = join;
        }
    }
    for (size_t i = 0; i < e->ops.size(); ++i) {
        const auto& r = e->ops[i].r;
        if (r.out >= 0 && e->tensors[r.out].def < 0) e->tensors[r.out].def = int(i);
        for (int t : {r.in, r.res})
            if (t >= 0) e->tensors[t].last_use = std::max(e->tensors[t].last_use, int(i));
        // a side op may still be READING its input while the ops before the join run: keep that buffer until the join
        if (e->ops[i].side_join >= 0 && r.in >= 0) e->tensors[r.in].last_use = std::max(e->tensors[r.in].last_use, e->ops[i].side_join);
    }
    struct Live {
        size_t off, size;
        int last;
    };
    std::vector<Live> live;
    size_t top = 0;
    std::vector<int> order;
    for (size_t i = 0; i < e->tensors.size(); ++i)
        if (e->tensors[i].binding < 0 && e->tensors[i].def >= 0) order.push_back(int(i));
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return e->tensors[a].def < e->tensors[b].def; });
    for (int ti : order) {
        Tensor& t = e->tensors[ti];
        if (t.last_use < t.def) t.last_use = t.def;
        const size_t size = align_up(t.item_bytes * e->max_batch, 1024);
        // a buffer may be reused once its last reader has been launched BEFORE the new producer.  When the persistent
        // network kernel is requested (B2_NET=1) fp16 engines keep it two more ops: that kernel overlaps consecutive
        // layers tile by tile, and a recycled buffer makes its new producer wait for the COMPLETION of every earlier
        // layer that touched it -- with the slack those layers lie >= 3 ops back and are long finished when the
        // producer's first tile is due.  (Measured cost of the larger arena on the per-layer path: ~1 %, so it is opt-in.)
        const int slack = e->half() ? env_int("B2_ARENA_SLACK", env_int("B2_NET", 0) ? 2 : 0) : 0;
        live.erase(std::remove_if(live.begin(), live.end(), [&](const Live& l) { return l.last + slack < t.def; }), live.end());
        std::sort(live.begin(), live.end(), [](const Live& a, const Live& b) { return a.off < b.off; });
        size_t off = 0;
        for (const Live& l : live) {
            if (off + size <= l.off) break;
            off = std::max(off, l.off + l.size);
        }
        t.offset = off;
        live.push_back({off, size, t.last_use});
        top = std::max(top, off + size);
    }
    e->act_bytes = align_up(std::max<size_t>(top, 1024), 1024);
    // fp16 engines reserve a fixed split-K workspace behind the activations (partial fp32 tiles)
    e->arena_bytes = e->act_bytes + (e->half() ? kSplitWorkspaceBytes : 0);
}

// ---- tensor maps ------------------------------------------------------------------------------
int make_map_2d(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint32_t box_inner,
                uint32_t box_outer, CUtensorMapSwizzle swz, bool int8 = false) {
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {inner * (int8 ? 1u : 2u)};
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode_tiled(map, int8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box,
                                estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(B2_ECUDA, "cuTensorMapEncodeTiled failed (%d) dims=%llu,%llu box=%u,%u", int(r),
                    (unsigned long long)inner, (unsigned long long)outer, box_inner, box_outer);
    return B2_OK;
}

// NHWC activation tensor as a 4-D tiled map {C, W, H, N} with a {64 ch, box_w, box_h, 1} box (3x3 halo kernel)
int make_map_nhwc(CUtensorMap* map, const void* base, int C, int W, int H, int N, uint32_t box_w, uint32_t box_h) {
    cuuint64_t dims[4] = {cuuint64_t(C), cuuint64_t(W), cuuint64_t(H), cuuint64_t(N)};
    cuuint64_t strides[3] = {cuuint64_t(C) * 2, cuuint64_t(C) * 2 * W, cuuint64_t(C) * 2 * W * H};
    cuuint32_t box[4] = {64, box_w, box_h, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(B2_ECUDA, "cuTensorMapEncodeTiled(4-D) failed (%d) C=%d W=%d H=%d N=%d box=%u,%u", int(r), C, W, H, N, box_w, box_h);
    return B2_OK;
}

// `pix_bytes` / `row_bytes` / `img_bytes`: global strides of the W, H, N modes.  The row-folded stem passes a pixel
// stride SMALLER than the C extent (overlapping windows): each "pixel" of the map is then kw real pixels.
int make_map_im2col(CUtensorMap* map, const void* base, int C, int W, int H, int N, uint64_t pix_bytes,
                    uint64_t row_bytes, uint64_t img_bytes, int kh, int kw, int stride_h, int stride_w, int pad_h,
                    int pad_w_lo, int pad_w_hi, uint32_t channels_per_pixel, uint32_t pixels_per_column,
                    CUtensorMapSwizzle swz, bool int8 = false) {
    cuuint64_t dims[4] = {cuuint64_t(C), cuuint64_t(W), cuuint64_t(H), cuuint64_t(N)};
    cuuint64_t strides[3] = {pix_bytes, row_bytes, img_bytes};
    // fprop bounding box: base pixel positions run over [-pad, dim - 1 + pad - (k-1)] (dilation 1)
    int lower[2] = {-pad_w_lo, -pad_h};                            // (W, H) order
    int upper[2] = {pad_w_hi - (kw - 1), pad_h - (kh - 1)};
    cuuint32_t estr[4] = {1, cuuint32_t(stride_w), cuuint32_t(stride_h), 1};
    CUresult r = g_encode_im2col(map, int8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, lower,
                                 upper, channels_per_pixel, pixels_per_column, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(B2_ECUDA, "cuTensorMapEncodeIm2col failed (%d) C=%d W=%d H=%d N=%d k=%dx%d s=%dx%d p=%d,%d/%d", int(r), C,
                    W, H, N, kh, kw, stride_h, stride_w, pad_h, pad_w_lo, pad_w_hi);
    // Driver workaround mirrored from CUTLASS (cute/atom/copy_traits_sm90_im2col.hpp): drivers <= 13.1 set a
    // descriptor bit that misbehaves for tensors smaller than 128 KiB.
    if (g_driver_version <= 13010 && img_bytes * uint64_t(N) < 131072)
        reinterpret_cast<uint64_t*>(map)[1] &= ~(1ull << 21);
    return B2_OK;
}

// Analytic cost model (microseconds) over the instantiated (N tile, pipeline depth, split-K) space.  The
// constants are rough B200 figures: ~70 KB/us of L2->SM bandwidth per SM, ~1 us TMA round trip, ~5 TB/s of
// aggregate L2 bandwidth, ~2 us of fixed per-CTA cost.  It only has to rank configurations sensibly.
ConvConfig pick_conv_config(int M, int cout_phys, int kblocks, int kb, bool residual, const b2_context* c, bool honor_forced) {
    const int m_tiles = (M + 127) / 128;
    ConvConfig best{0, 0, 1, 1e30};
    const int bns[4] = {256, 128, 64, 32};
    const int stgs[4] = {1, 2, 4, 8};
    for (int bn : bns) {
        if (cout_phys % bn) continue;
        if (honor_forced && c->force_bn && bn != c->force_bn) continue;
        const int tiles = m_tiles * (cout_phys / bn);
        for (int splits = 1; splits <= 8; ++splits) {
            if (c->force_splits ? splits != c->force_splits : splits != 1) continue;  // split-K is opt-in (measured slower)
            if (splits > 1 && (kb != 64 || kblocks / splits < 4 || tiles * splits > 160 || tiles > kMaxSplitTiles ||
                               size_t(tiles) * splits * 128 * bn * 4 > kSplitWorkspaceBytes))
                continue;
            const int kpc = (kblocks + splits - 1) / splits;
            if (splits > 1 && (splits - 1) * kpc >= kblocks) continue;  // an empty split
            for (int st : stgs) {
                if (!b2k::conv_config_exists(bn, kb, st)) continue;
                if (b2k::conv_smem_bytes(bn, st, residual) > 227 * 1024) continue;
                if (honor_forced && c->force_stages && st != c->force_stages) continue;
                if (!(honor_forced && c->force_stages) && !stage_depth_useful(bn, kb, st, kpc)) continue;
                const double smem = b2k::conv_smem_bytes(bn, st, residual);
                int per_sm = int(227.0 * 1024 / smem);
                per_sm = std::min(per_sm, 512 / std::max(32, bn));
                per_sm = std::max(1, std::min(per_sm, 8));
                const int ctas = tiles * splits;
                const int waves = (ctas + 148 * per_sm - 1) / (148 * per_sm);
                const int sharing = std::max(1, std::min(per_sm, (ctas + 147) / 148));
                const double stage_bytes = 16384.0 + bn * 128.0;
                const double t_kb = std::max(stage_bytes / (70000.0 / sharing), 1.0 / st);
                double t_epi = 0.6 + bn / 64.0 * 0.4 + (residual ? 0.4 : 0.0);
                if (splits > 1) t_epi += 1.0 + 0.3 * splits;
                const double t_cta = 2.0 + kpc * t_kb + t_epi;
                double total = waves * t_cta;
                const double traffic = double(ctas) * kpc * stage_bytes;
                total = std::max(total, traffic / 5.0e6 + 2.0);
                if (total < best.est_us) best = ConvConfig{bn, st, splits, total};
            }
        }
    }
    return best;
}

// Row-folded stem: an 8-channel input whose kw taps are contiguous in memory (stride_w 1, no W padding left to
// resolve) is read as ONE 64-byte "pixel" per filter row through an overlapping pixel stride.
bool conv_is_row_folded(const b2_context* c, const Op& op) {
    const b2plan::OpRec& r = op.r;
    return !c->no_fold && r.cin_phys == 8 && op.kw() * 8 * 2 == 64 && op.sw() == 1 && op.pw_lo() == 0 && op.pw_hi() == 0;
}
int conv_kb(const b2_context* c, const Op& op) {
    if (op.r.cin_phys % 64 == 0) return 64;
    return conv_is_row_folded(c, op) ? 32 : 8;
}
int conv_num_kblocks(const b2_context* c, const Op& op) {
    const b2plan::OpRec& r = op.r;
    if (r.cin_phys % 64 == 0) return int(r.taps) * (int(r.cin_phys) / 64);
    if (conv_is_row_folded(c, op)) return (op.kh() + 1) / 2;  // two filter rows (2 x 32 K) per 64-wide k-block
    return (int(r.taps_phys) + 7) / 8;
}

// 3x3 / stride 1 / pad 1 on 64-channel blocks with packed weights and no fused residual: the halo kernel applies.
// Returns the rows per tile R (0 = not applicable).
int conv_halo_rows(const b2_context* c, const Op& op) {
    const b2plan::OpRec& r = op.r;
    const Tensor& ti = c->e->tensors[r.in];
    const Tensor& to = c->e->tensors[r.out];
    if (r.cin_phys % 64 || r.cout_phys % 64 || op.kh() != 3 || op.kw() != 3 || op.sh() != 1 || op.sw() != 1 || op.ph() != 1 ||
        op.pw_lo() != 1 || op.pw_hi() != 1 || r.res >= 0 || !(r.relu & 2) || c->no_pack || ti.h != to.h || ti.w != to.w)
        return 0;
    const int wp = int(to.w) + 2;
    if (wp > 128) return 0;
    return std::min(128 / wp, int(to.h));
}

// Fill a ConvLaunch (kernel arguments + TMA tensor maps) for one conv op under a given configuration.
int make_conv_launch(b2_context* c, const Op& op, int batch, const ConvConfig& cfg, b2k::ConvLaunch* out) {
    b2_engine* e = c->e;
    const b2plan::OpRec& r = op.r;
    const Tensor& ti = e->tensors[r.in];
    const Tensor& to = e->tensors[r.out];
    auto tptr = [&](int idx) -> uint8_t* { return c->scratch + e->tensors[idx].offset; };
    const uint8_t* w = e->d_payload + r.w_off;
    const int M = batch * int(to.h) * int(to.w);
    const bool kb64 = r.cin_phys % 64 == 0;
    const bool fold = conv_is_row_folded(c, op);
    b2k::ConvLaunch& cl = *out;
    memset(&cl, 0, sizeof cl);
    cl.kb = conv_kb(c, op);
    cl.grid_m = (M + 127) / 128;
    const int nkb = conv_num_kblocks(c, op);
    cl.bn = cfg.bn;
    cl.stages = cfg.stages;
    cl.sps = cfg.sps > 0 ? cfg.sps : 1;
    cl.grid_n = int(r.cout_phys) / cl.bn;
    cl.ws_ctas = cfg.ws;
    cl.cn = (cfg.cn > 1 && cfg.ws == 0 && cl.kb == 64 && cl.grid_n % cfg.cn == 0 &&
             b2k::conv_cluster_config_exists(cl.bn, cl.stages, cl.sps, cfg.cn)) ? cfg.cn : 1;
    cl.args.cn = cl.cn;
    cl.args.tiles_m = cl.grid_m;
    cl.args.tiles_n = cl.grid_n;
    b2k::ConvArgs& a = cl.args;
    a.splits = cfg.splits;
    a.kb_per_split = (nkb + cfg.splits - 1) / cfg.splits;
    a.workspace = reinterpret_cast<float*>(c->scratch + e->act_bytes);
    a.tile_counters = c->d_counters;
    a.pdl_trigger = c->pdl_trigger;
    a.bias = reinterpret_cast<const float*>(e->d_payload + r.b_off);
    a.residual = r.res >= 0 ? reinterpret_cast<const __half*>(tptr(r.res)) : nullptr;
    a.out = reinterpret_cast<__half*>(tptr(r.out));
    a.M = M;
    a.Cout = int(r.cout_phys);
    a.taps = fold ? op.kh() : int(r.taps);            // folded: one "tap" = one filter row of kw*8 K-elements
    a.taps_phys = fold ? op.kh() : int(r.taps_phys);
    a.kw = fold ? 1 : op.kw();
    a.cblocks = kb64 ? int(r.cin_phys) / 64 : 1;
    a.num_kblocks = nkb;
    a.HoWo = int(to.h * to.w);
    a.Wo = int(to.w);
    a.stride_h = op.sh();
    a.stride_w = op.sw();
    a.pad_h = op.ph();
    a.pad_w = op.pw_lo();
    a.relu = int(r.relu & 1);
    a.wpacked = (r.relu & 2) && !c->no_pack ? w : nullptr;
    const bool tiled = r.k == 1 && op.kw() == 1 && r.stride == 1 && op.sw() == 1 && r.pad_ == 0 && op.pw_lo() == 0 &&
                       op.pw_hi() == 0 && kb64 && !c->force_im2col;
    a.a_mode = tiled ? b2k::A_TILED : b2k::A_IM2COL;
    if (cfg.halo) {
        const int R = conv_halo_rows(c, op);
        if (!R || !b2k::conv_halo_config_exists(cl.bn) || int(r.cin_phys) / 64 > 8 || b2k::conv_halo_smem(cl.bn, int(to.w), R, int(r.cin_phys) / 64) > 227 * 1024)
            return fail(B2_EINVAL, "conv %s: the halo tactic does not apply", op.name.c_str());
        cl.halo = 1;
        cl.ws_ctas = 0, cl.cn = 1, a.cn = 1, a.splits = 1, cl.stages = kHaloStagesTag, cl.sps = 1;
        a.halo_rows = R;
        cl.grid_m = batch * ((int(to.h) + R - 1) / R);
        int rc = make_map_nhwc(&cl.mapA, tptr(r.in), int(r.cin_phys), int(ti.w), int(ti.h), batch, uint32_t(ti.w) + 2, uint32_t(R) + 2);
        if (rc) return rc;
        rc = make_map_nhwc(&cl.mapOut, tptr(r.out), int(r.cout_phys), int(to.w), int(to.h), batch, uint32_t(to.w) + 2, uint32_t(R));
        cl.mapB = cl.mapA, cl.mapRes = cl.mapOut;
        return rc;
    }
    const CUtensorMapSwizzle swz = kb64 ? CU_TENSOR_MAP_SWIZZLE_128B : (fold ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE);
    const uint64_t pix = uint64_t(r.cin_phys) * 2, rowb = uint64_t(ti.w) * pix, imgb = uint64_t(ti.h) * rowb;
    int rc;
    if (tiled)
        rc = make_map_2d(&cl.mapA, tptr(r.in), r.cin_phys, uint64_t(M), 64, uint32_t(128 / cl.cn), swz);
    else if (fold)  // kw pixels x 8 channels = 32 contiguous K-elements per window; windows advance by ONE pixel
        rc = make_map_im2col(&cl.mapA, tptr(r.in), int(r.cin_phys) * op.kw(), int(ti.w) - op.kw() + 1, int(ti.h), batch, pix,
                             rowb, imgb, op.kh(), 1, op.sh(), 1, op.ph(), 0, 0, 32, 128, swz);
    else
        rc = make_map_im2col(&cl.mapA, tptr(r.in), int(r.cin_phys), int(ti.w), int(ti.h), batch, pix, rowb, imgb, op.kh(),
                             op.kw(), op.sh(), op.sw(), op.ph(), op.pw_lo(), op.pw_hi(), uint32_t(cl.kb), uint32_t(128 / cl.cn), swz);
    if (rc) return rc;
    if (r.relu & 2)  // packed weights are not addressable as a [Cout][K] matrix; mapB stays a valid dummy
        cl.mapB = cl.mapA;
    else
        rc = make_map_2d(&cl.mapB, w, uint64_t(r.taps_phys) * r.cin_phys, r.cout_phys, uint32_t(cl.kb), uint32_t(cl.bn), swz);
    if (rc) return rc;
    // epilogue maps: 128-row x min(64, BN)-column boxes, 128B (or 64B for BN=32) swizzle = conflict-free staging
    const uint32_t ow = cl.bn >= 64 ? 64 : 32;
    const CUtensorMapSwizzle oswz = cl.bn >= 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    rc = make_map_2d(&cl.mapOut, tptr(r.out), r.cout_phys, uint64_t(M), ow, 128, oswz);
    if (rc) return rc;
    if (r.res >= 0) rc = make_map_2d(&cl.mapRes, tptr(r.res), r.cout_phys, uint64_t(M), ow, 128, oswz);
    else cl.mapRes = cl.mapOut;
    return rc;
}

// INT8 convolution launch (i8_kernels.cu): TMA maps over 1-byte tensors whose 128-byte rows hold 128 channels.
int make_i8_conv_launch(b2_context* c, const Op& op, int batch, int bn, int stages, b2k::I8ConvLaunch* out) {
    b2_engine* e = c->e;
    const b2plan::OpRec& r = op.r;
    const Tensor& ti = e->tensors[r.in];
    const Tensor& to = e->tensors[r.out];
    auto tptr = [&](int idx) -> uint8_t* { return c->scratch + e->tensors[idx].offset; };
    b2k::I8ConvLaunch& cl = *out;
    memset(&cl, 0, sizeof cl);
    const int M = batch * int(to.h) * int(to.w);
    cl.bn = bn, cl.stages = stages;
    cl.grid_m = (M + 127) / 128;
    cl.grid_n = int(r.cout_phys) / bn;
    b2k::I8ConvArgs& a = cl.args;
    a.wpacked = e->d_payload + r.w_off;
    const float* rq = reinterpret_cast<const float*>(e->d_payload + r.b_off);
    a.m = rq;
    a.b = rq + r.cout_phys;
    a.r = e->requant_r.at(int(&op - &e->ops[0]));
    a.has_res = r.res >= 0 ? 1 : 0;
    a.relu = int(r.relu & 1);
    a.M = M, a.Cout = int(r.cout_phys);
    a.cblocks = int(r.cin_phys) / 128;
    a.last_cb_mmas = (int(r.cin) % 128) ? (int(r.cin) % 128 + 31) / 32 : 4;
    a.cout_real = int(r.cout);
    a.num_kblocks = int(r.taps) * a.cblocks;
    a.kw = op.kw(), a.HoWo = int(to.h * to.w), a.Wo = int(to.w);
    a.stride_h = op.sh(), a.stride_w = op.sw(), a.pad_h = op.ph(), a.pad_w = op.pw_lo();
    const bool tiled = r.k == 1 && r.stride == 1 && r.pad_ == 0;
    a.a_mode = tiled ? b2k::A_TILED : b2k::A_IM2COL;
    int rc;
    if (tiled)
        rc = make_map_2d(&cl.mapA, tptr(r.in), r.cin_phys, uint64_t(M), 128, 128, CU_TENSOR_MAP_SWIZZLE_128B, true);
    else {
        const uint64_t pix = uint64_t(r.cin_phys), rowb = uint64_t(ti.w) * pix, imgb = uint64_t(ti.h) * rowb;
        rc = make_map_im2col(&cl.mapA, tptr(r.in), int(r.cin_phys), int(ti.w), int(ti.h), batch, pix, rowb, imgb, op.kh(), op.kw(), op.sh(),
                             op.sw(), op.ph(), op.pw_lo(), op.pw_hi(), 128, 128, CU_TENSOR_MAP_SWIZZLE_128B, true);
    }
    if (rc) return rc;
    rc = make_map_2d(&cl.mapOut, tptr(r.out), r.cout_phys, uint64_t(M), 128, 128, CU_TENSOR_MAP_SWIZZLE_128B, true);
    if (rc) return rc;
    if (r.res >= 0) rc = make_map_2d(&cl.mapRes, tptr(r.res), r.cout_phys, uint64_t(M), 128, 128, CU_TENSOR_MAP_SWIZZLE_128B, true);
    else cl.mapRes = cl.mapOut;
    return rc;
}

// Tactic selection, the role TensorRT's builder plays for the reference's engines: time every instantiated
// (N tile, pipeline depth) on THIS device with the layer's real shapes and keep the fastest.  Runs once per
// (engine, layer, batch); results are shared by all contexts of the engine.
// fixed_halo: -1 free choice, 0 never, 1 only the halo kernel (decided once at max batch: it changes the summation order)
int autotune_conv(b2_context* c, const Op& op, int batch, int fixed_splits, int fixed_halo, ConvConfig* best_out) {
    b2_engine* e = c->e;
    const b2plan::OpRec& r = op.r;
    const Tensor& to = e->tensors[r.out];
    const int M = batch * int(to.h) * int(to.w);
    const int kbsz = conv_kb(c, op);
    const int nkb = conv_num_kblocks(c, op);
    // c->autotune == 1: latency mode (one stream).  >= 2: throughput mode -- the candidate is launched on that
    // many streams at once, which is how the kernels meet each other when several ExecutionContexts overlap
    // (BASELINE config: 4 contexts); deep pipelines that win alone can lose here because they hog shared memory.
    const int ns = std::max(1, std::min(c->autotune, 8));
    std::vector<cudaStream_t> ss(ns, nullptr);
    std::vector<cudaEvent_t> done(ns, nullptr);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool ok = cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess;
    for (int i = 0; i < ns && ok; ++i)
        ok = cudaStreamCreateWithFlags(&ss[i], cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) == cudaSuccess;
    auto cleanup = [&] {
        for (auto s_ : ss)
            if (s_) cudaStreamDestroy(s_);
        for (auto d : done)
            if (d) cudaEventDestroy(d);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
    };
    if (!ok) {
        cudaGetLastError();
        cleanup();
        return fail(B2_ECUDA, "autotune: cannot create streams/events");
    }
    ConvConfig best = *best_out;
    double best_ms = 1e30;
    const int bns[4] = {256, 128, 64, 32};
    const int stgs[4] = {1, 2, 4, 8};
    int status = B2_OK;
    const int verbose = env_int("B2_TUNE_VERBOSE", 0);             // 1: the winner per layer, 2: every candidate
    const int iters = std::max(4, env_int("B2_TUNE_ITERS", 12));   // launches per stream and measurement
    const int reps = std::max(1, env_int("B2_TUNE_REPS", 2));      // measurements per candidate (the quietest counts)
    const int m_tiles = (M + 127) / 128;
    const int split_cands[4] = {1, 2, 4, 8};
    std::vector<ConvConfig> candidates;
    for (int bn : bns) {
        if (int(r.cout_phys) % bn) continue;
        const int tiles = m_tiles * (int(r.cout_phys) / bn);
        for (int ws = 0; ws <= 1; ++ws)
        for (int sp : split_cands)
        for (int sps = 1; sps <= 2; ++sps)
        for (int st : stgs) {
            if (fixed_splits > 0 && sp != fixed_splits) continue;
            if (ws) {  // persistent warp-specialised tactic: 64-wide K, packed weights, no split-K
                if (c->force_ws < 0 || kbsz != 64 || !(r.relu & 2) || sp != 1) continue;
                if (!b2k::conv_ws_config_exists(bn, st, sps) || b2k::conv_ws_smem(bn, st, sps, r.res >= 0) > 227 * 1024) continue;
                if (sps == 2 && nkb < 4) continue;
            } else {
            if (c->force_ws > 0 && kbsz == 64 && (r.relu & 2)) continue;
            if (!b2k::conv_config_exists(bn, kbsz, st, sps)) continue;
            if (b2k::conv_smem_bytes(bn, st, r.res >= 0, sps) > 227 * 1024) continue;
            }
            const int kpc = (nkb + sp - 1) / sp;
            if (ws) {
                candidates.push_back(ConvConfig{bn, st, 1, 0.0, sps, std::min(tiles, 148), 1});
                if (tiles > 74) candidates.push_back(ConvConfig{bn, st, 1, 0.0, sps, 74, 1});  // half the SMs per stream
                if (tiles >= 592 && b2k::conv_ws_smem(bn, st, sps, r.res >= 0) <= 113 * 1024)
                    candidates.push_back(ConvConfig{bn, st, 1, 0.0, sps, 296, 1});  // two co-resident CTAs per SM
                continue;
            }
            if (sps == 2 && kpc < 4) continue;  // double-width stages only pay on long K loops
            if (sps == 1 && !stage_depth_useful(bn, kbsz, st, kpc)) continue;
            if (sps == 2 && st * 2 > kpc + 2) continue;
            if (sp > 1 && (kbsz != 64 || tiles >= 100 || tiles > kMaxSplitTiles / 8 || kpc < 4 || tiles * sp > 160 ||
                           (sp - 1) * kpc >= nkb ||
                           size_t(tiles) * sp * 128 * bn * 4 > kSplitWorkspaceBytes))
                continue;  // split-K only where the plain grid leaves SMs idle
            const bool cn_forced_here = c->force_cn > 1 && kbsz == 64 && (int(r.cout_phys) / bn) % c->force_cn == 0 &&
                                        b2k::conv_cluster_config_exists(bn, st, sps, c->force_cn);
            if (!cn_forced_here) candidates.push_back(ConvConfig{bn, st, sp, 0.0, sps, 0, 1});
            // clusters along N that multicast the activation tile: never won a timing on B200 (the L2 read is shared but
            // every SM still ingests the whole tile, and the cluster barriers cost latency) -> tried only on request
            if (kbsz == 64 && c->force_cn > 0)
                for (int cn = 2; cn <= 4; cn *= 2)
                    if ((int(r.cout_phys) / bn) % cn == 0 && (!c->force_cn || cn == c->force_cn) &&
                        b2k::conv_cluster_config_exists(bn, st, sps, cn))
                        candidates.push_back(ConvConfig{bn, st, sp, 0.0, sps, 0, cn});
        }
    }
    if (fixed_halo != 0 && c->force_halo >= 0 && (fixed_splits <= 1)) {
        const int R = conv_halo_rows(c, op);
        std::vector<ConvConfig> halo_cands;
        if (R)
            for (int bn : bns)
                if (int(r.cout_phys) % bn == 0 && b2k::conv_halo_config_exists(bn) &&
                    int(r.cin_phys) / 64 <= 8 && b2k::conv_halo_smem(bn, int(to.w), R, int(r.cin_phys) / 64) <= 227 * 1024) {
                    ConvConfig hc{bn, kHaloStagesTag, 1, 0.0, 1, 0, 1};
                    hc.halo = 1;
                    halo_cands.push_back(hc);
                }
        if (!halo_cands.empty() && (c->force_halo > 0 || fixed_halo > 0)) candidates.clear();
        candidates.insert(candidates.end(), halo_cands.begin(), halo_cands.end());
    }
    std::vector<std::pair<ConvConfig, double>> timed;
    for (const ConvConfig& cand : candidates) {
        {
            const int bn = cand.bn, st = cand.stages, sp = cand.splits;
            const int tiles = m_tiles * (int(r.cout_phys) / bn);
            b2k::ConvLaunch cl0;
            if ((status = make_conv_launch(c, op, batch, cand, &cl0))) break;
            // concurrent split-K launches must not share arrival counters or partial-tile storage
            std::vector<b2k::ConvLaunch> cls(ns, cl0);
            void* tmp_ws = nullptr;
            if (sp > 1) {
                const size_t ws_bytes = size_t(tiles) * sp * 128 * bn * 4;
                if (cudaMalloc(&tmp_ws, ws_bytes * ns) != cudaSuccess) {
                    cudaGetLastError();
                    continue;
                }
                for (int k = 0; k < ns; ++k) {
                    cls[k].args.workspace = reinterpret_cast<float*>(static_cast<uint8_t*>(tmp_ws) + ws_bytes * k);
                    cls[k].args.tile_counters = c->d_counters + k * (kMaxSplitTiles / 8);
                }
            }
            int rc = 0;
            for (int i = 0; i < 2 && !rc; ++i)
                for (int k = 0; k < ns && !rc; ++k) rc = b2k::launch_conv_f16_tcgen05(cls[k], ss[k]);
            for (int k = 0; k < ns; ++k) cudaStreamSynchronize(ss[k]);
            float ms = 1e30f;
            cudaError_t se = cudaSuccess;
            for (int rep = 0; rep < reps && !rc && se == cudaSuccess; ++rep) {  // keep the quietest measurement
                cudaEventRecord(e0, ss[0]);
                for (int k = 1; k < ns; ++k) cudaStreamWaitEvent(ss[k], e0, 0);
                for (int i = 0; i < iters && !rc; ++i)
                    for (int k = 0; k < ns && !rc; ++k) rc = b2k::launch_conv_f16_tcgen05(cls[k], ss[k]);
                for (int k = 1; k < ns; ++k) {
                    cudaEventRecord(done[k], ss[k]);
                    cudaStreamWaitEvent(ss[0], done[k], 0);
                }
                cudaEventRecord(e1, ss[0]);
                se = cudaStreamSynchronize(ss[0]);
                float t = 0.f;
                if (se == cudaSuccess && cudaEventElapsedTime(&t, e0, e1) == cudaSuccess) ms = std::min(ms, t);
            }
            if (tmp_ws) cudaFree(tmp_ws);
            if (rc || se != cudaSuccess) {
                status = fail(B2_ECUDA, "autotune of %s (bn=%d st=%d) failed: %s", op.name.c_str(), bn, st,
                              cudaGetErrorString(rc ? cudaError_t(rc) : se));
                break;
            }
            if (verbose > 1)
                fprintf(stderr, "[b2 tune]   %s b=%d cand bn=%d st=%d sp=%d sps=%d ws=%d cn=%d halo=%d : %.3f us/launch\n", op.name.c_str(),
                        batch, cand.bn, cand.stages, cand.splits, cand.sps, cand.ws, cand.cn, cand.halo, ms * 1e3 / (iters * ns));
            timed.push_back({cand, double(ms)});
            if (ms < best_ms) best_ms = ms, best = cand;
        }
        if (status) break;
    }
    cleanup();
    if (status) return status;
    // B2_TUNE_TIE_PERMILLE = t > 0: among the one-tile tactics within t/1000 of the fastest, take the WIDEST N tile (fewest
    // CTAs, least L2->SM traffic per MAC): with several copies of one layer the timing cannot see the SMs a wide tile
    // leaves to the other contexts' layers.  0 (default) = fastest wins; measured neutral-to-negative, DESIGN.md.
    const int tie = env_int("B2_TUNE_TIE_PERMILLE", 0);
    if (tie > 0 && !best.ws && !best.halo && best.splits == 1) {
        for (const auto& t : timed)
            if (!t.first.ws && !t.first.halo && t.first.splits == 1 && t.first.cn == best.cn && t.second <= best_ms * (1.0 + tie / 1000.0) &&
                (t.first.bn > best.bn || (t.first.bn == best.bn && t.second < best_ms)))
                best = t.first, best_ms = std::min(best_ms, t.second);
    }
    best.est_us = best_ms * 1e3 / (iters * ns);
    if (verbose)
        fprintf(stderr, "[b2 tune] %s b=%d M=%d N=%d K=%d best bn=%d st=%d sp=%d sps=%d ws=%d cn=%d halo=%d : %.3f us/launch (%d streams)\n",
                op.name.c_str(), batch, M, int(r.cout_phys), nkb * kbsz, best.bn, best.stages, best.splits, best.sps, best.ws, best.cn,
                best.halo, best.est_us, ns);
    *best_out = best;
    (void)M;
    return B2_OK;
}

// ---- tactic cache file (B2_TUNE_CACHE=<path>): the analogue of a TensorRT timing cache.  One line per tuned conv:
//      <engine name> <op index> <batch> <bn> <stages> <splits> <sps> <persistent CTAs or 0> <cluster size> <halo 0/1>
void tune_cache_load(b2_engine* e) {
    if (e->tune_cache_loaded) return;
    e->tune_cache_loaded = true;
    const char* path = getenv("B2_TUNE_CACHE");
    if (!path) return;
    FILE* f = fopen(path, "r");
    if (!f) return;
    char name[128];
    int op, batch, bn, st, sp, sps, ws, cn, halo;
    while (fscanf(f, "%127s %d %d %d %d %d %d %d %d %d", name, &op, &batch, &bn, &st, &sp, &sps, &ws, &cn, &halo) == 10)
        if (e->name == name && op >= 0 && op < int(e->ops.size())) {
            ConvConfig cfg{bn, st, sp, 0.0, sps, ws, cn};
            cfg.halo = halo;
            e->tuned[{op, batch}] = cfg;
        }
    fclose(f);
}
void tune_cache_append(const b2_engine* e, int op, int batch, const ConvConfig& cfg) {
    const char* path = getenv("B2_TUNE_CACHE");
    if (!path) return;
    FILE* f = fopen(path, "a");
    if (!f) return;
    fprintf(f, "%s %d %d %d %d %d %d %d %d %d\n", e->name.c_str(), op, batch, cfg.bn, cfg.stages, cfg.splits, cfg.sps, cfg.ws, cfg.cn,
            cfg.halo);
    fclose(f);
}

// Can `cfg` (possibly measured at another batch size) run `op` at `batch`?
bool tactic_applies(const b2_context* c, const Op& op, int batch, const ConvConfig& cfg) {
    const b2plan::OpRec& r = op.r;
    if (cfg.bn <= 0 || int(r.cout_phys) % cfg.bn) return false;
    const int kbsz = conv_kb(c, op);
    if (cfg.halo) return conv_halo_rows(c, op) > 0 && b2k::conv_halo_config_exists(cfg.bn);
    if (cfg.ws) return kbsz == 64 && b2k::conv_ws_config_exists(cfg.bn, cfg.stages, cfg.sps);
    if (!b2k::conv_config_exists(cfg.bn, kbsz, cfg.stages, cfg.sps)) return false;
    if (cfg.splits > 1) {
        const int tiles = ((batch * int(c->e->tensors[r.out].h * c->e->tensors[r.out].w) + 127) / 128) * (int(r.cout_phys) / cfg.bn);
        if (tiles > kMaxSplitTiles || size_t(tiles) * cfg.splits * 128 * cfg.bn * 4 > kSplitWorkspaceBytes) return false;
    }
    return true;
}

// INT8 twin of autotune_conv: times every (N tile, ring depth) of conv_i8_tcgen05 on `c->autotune` concurrent streams.
int autotune_i8_conv(b2_context* c, const Op& op, int batch, ConvConfig* best_out) {
    const b2plan::OpRec& r = op.r;
    const int ns = std::max(1, std::min(c->autotune, 8));
    std::vector<cudaStream_t> ss(size_t(ns), nullptr);
    std::vector<cudaEvent_t> done(size_t(ns), nullptr);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool ok = cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess;
    for (int i = 0; i < ns && ok; ++i)
        ok = cudaStreamCreateWithFlags(&ss[size_t(i)], cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&done[size_t(i)], cudaEventDisableTiming) == cudaSuccess;
    auto cleanup = [&] {
        for (auto s_ : ss)
            if (s_) cudaStreamDestroy(s_);
        for (auto d : done)
            if (d) cudaEventDestroy(d);
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
    };
    if (!ok) {
        cudaGetLastError();
        cleanup();
        return fail(B2_ECUDA, "autotune: cannot create streams/events");
    }
    const int verbose = env_int("B2_TUNE_VERBOSE", 0);
    const int iters = std::max(4, env_int("B2_TUNE_ITERS", 12));
    const int reps = std::max(1, env_int("B2_TUNE_REPS", 2));
    double best_ms = 1e30;
    ConvConfig best = *best_out;
    int status = B2_OK;
    for (int bn : {128, 256}) {
        if (int(r.cout_phys) % bn) continue;
        for (int st = 1; st <= 4 && !status; ++st) {
            if (!b2k::conv_i8_config_exists(bn, st)) continue;
            b2k::I8ConvLaunch cl;
            if ((status = make_i8_conv_launch(c, op, batch, bn, st, &cl))) break;
            int rc = 0;
            for (int i = 0; i < 2 && !rc; ++i)
                for (int k = 0; k < ns && !rc; ++k) rc = b2k::launch_conv_i8_tcgen05(cl, ss[size_t(k)]);
            for (int k = 0; k < ns; ++k) cudaStreamSynchronize(ss[size_t(k)]);
            float ms = 1e30f;
            cudaError_t se = cudaSuccess;
            for (int rep = 0; rep < reps && !rc && se == cudaSuccess; ++rep) {
                cudaEventRecord(e0, ss[0]);
                for (int k = 1; k < ns; ++k) cudaStreamWaitEvent(ss[size_t(k)], e0, 0);
                for (int i = 0; i < iters && !rc; ++i)
                    for (int k = 0; k < ns && !rc; ++k) rc = b2k::launch_conv_i8_tcgen05(cl, ss[size_t(k)]);
                for (int k = 1; k < ns; ++k) {
                    cudaEventRecord(done[size_t(k)], ss[size_t(k)]);
                    cudaStreamWaitEvent(ss[0], done[size_t(k)], 0);
                }
                cudaEventRecord(e1, ss[0]);
                se = cudaStreamSynchronize(ss[0]);
                float t = 0.f;
                if (se == cudaSuccess && cudaEventElapsedTime(&t, e0, e1) == cudaSuccess) ms = std::min(ms, t);
            }
            if (rc || se != cudaSuccess) {
                status = fail(B2_ECUDA, "autotune of %s (int8 bn=%d st=%d) failed: %s", op.name.c_str(), bn, st,
                              cudaGetErrorString(rc ? cudaError_t(rc) : se));
                break;
            }
            if (verbose > 1)
                fprintf(stderr, "[b2 tune]   %s b=%d cand int8 bn=%d st=%d : %.3f us/launch\n", op.name.c_str(), batch, bn, st,
                        ms * 1e3 / (iters * ns));
            if (ms < best_ms) best_ms = ms, best = ConvConfig{bn, st, 1, 0.0, 1, 0, 1};
        }
    }
    cleanup();
    if (status) return status;
    best.est_us = best_ms * 1e3 / (iters * ns);
    if (verbose) {
        const Tensor& to = c->e->tensors[r.out];
        const long long M = (long long)batch * to.h * to.w, K = (long long)r.k * r.k * r.cin_phys;
        fprintf(stderr, "[b2 tune] %s b=%d M=%lld N=%d K=%lld best int8 bn=%d st=%d : %.3f us/launch (%d streams) %.0f TOP/s\n",
                op.name.c_str(), batch, M, int(r.cout_phys), K, best.bn, best.stages, best.est_us, ns,
                2.0 * M * r.cout_phys * K / best.est_us * 1e-6);
    }
    *best_out = best;
    return B2_OK;
}

// Times the tactics of every tcgen05 convolution of the engine at `batch` (and, first, at max batch: the split-K factor
// is chosen once there) on a context with a PRIVATE arena -- never on memory a request may be using.
int tune_engine_batch(b2_context* c, int batch) {
    b2_engine* e = c->e;
    for (size_t i = 0; i < e->ops.size(); ++i) {
        const Op& op = e->ops[i];
        const b2plan::OpRec& r = op.r;
        if (r.type != b2plan::OP_CONV || !e->half()) continue;
        if (r.relu & 4) {  // INT8 convolution: (N tile, ring depth)
            {
                std::lock_guard<std::mutex> lock(e->tune_mutex);
                if (e->tuned.count({int(i), batch})) continue;
            }
            ConvConfig cfg{128, 2, 1, 0.0, 1, 0, 1};
            int rc = autotune_i8_conv(c, op, batch, &cfg);
            if (rc) return rc;
            std::lock_guard<std::mutex> lock(e->tune_mutex);
            e->tuned[{int(i), batch}] = cfg;
            tune_cache_append(e, int(i), batch, cfg);
            continue;
        }
        const bool kb64 = r.cin_phys % 64 == 0, kb8 = r.cin_phys == 8;
        if (!((kb64 || kb8) && r.cout_phys % 32 == 0 && (kb64 || r.taps_phys % 2 == 0))) continue;
        {
            std::lock_guard<std::mutex> lock(e->tune_mutex);
            if (e->tuned.count({int(i), batch})) continue;
        }
        const Tensor& to = e->tensors[r.out];
        const int kbsz = conv_kb(c, op), nkb = conv_num_kblocks(c, op);
        const bool side = op.side_join >= 0;
        // Split-K is the ONE tactic that changes the fp32 summation order (every other one -- N tile, ring depth, halo,
        // persistent -- adds the same products in the same order), so letting the timing pick it would make the BITS of a
        // model depend on the load-time measurement of that process: seen once as a 4e-3 relative difference between a tuned
        // manager and an untuned session of the same plan.  It never won a serving-regime timing anyway (the closest
        // candidate is 40 % behind, profiles/tune_dump_r2_rn50_b8_4streams.log), so the tuner leaves it alone unless
        // B2_TUNE_SPLITK=1; `splits` stays available as an explicit option.
        static const bool tune_splitk = env_int("B2_TUNE_SPLITK", 0) != 0;
        int splits = (side || !tune_splitk) ? 1 : 0;
        if (batch != e->max_batch && !side && tune_splitk) {
            std::lock_guard<std::mutex> lock(e->tune_mutex);
            auto it = e->tuned.find({int(i), e->max_batch});
            if (it != e->tuned.end()) splits = it->second.splits;
        }
        ConvConfig cfg = pick_conv_config(batch * int(to.h) * int(to.w), int(r.cout_phys), nkb, kbsz, r.res >= 0, c, false);
        int rc = autotune_conv(c, op, batch, splits, -1, &cfg);
        if (rc) return rc;
        std::lock_guard<std::mutex> lock(e->tune_mutex);
        e->tuned[{int(i), batch}] = cfg;
        tune_cache_append(e, int(i), batch, cfg);
    }
    return B2_OK;
}

// ---- persistent-kernel runs ----------------------------------------------------------------------
// Folds every maximal run of consecutive `net_member` convolution launches (launch index == op index here) into one
// L_NET launch: layer table with the TMA maps already built by make_conv_launch, the input M-tile range every output
// M tile depends on, and the layers whose completion a recycled output buffer has to wait for.
int fuse_net_runs(b2_context* c, Plan* plan, int batch) {
    b2_engine* e = c->e;
    std::vector<Launch>& ls = plan->launches;
    bool any = false;
    for (const Launch& L : ls) any = any || L.net_member;
    if (!any) return B2_OK;
    std::vector<Launch> fused;
    size_t i = 0;
    while (i < ls.size()) {
        if (!ls[i].net_member) {
            fused.push_back(std::move(ls[i]));
            ++i;
            continue;
        }
        size_t j = i;
        while (j + 1 < ls.size() && ls[j + 1].net_member && int(j + 1 - i) < b2k::kNetMaxLayers - 1) ++j;
        const int n = int(j - i + 1);
        std::vector<b2k::NetLayer> layers(n);
        std::vector<short2> deps;
        std::map<int, int> producer;  // tensor index -> local layer
        int tile_cursor = 0, flag_cursor = 0;
        double flops = 0, bytes = 0;
        auto trange = [&](int ti, size_t* lo, size_t* hi) {
            const Tensor& t = e->tensors[ti];
            *lo = t.offset;
            *hi = t.offset + t.item_bytes * size_t(batch);
        };
        for (int l = 0; l < n; ++l) {
            const Op& op = e->ops[i + l];
            const b2plan::OpRec& r = op.r;
            const b2k::ConvLaunch& cl = ls[i + l].conv;
            const b2k::ConvArgs& a = cl.args;
            b2k::NetLayer& nl = layers[l];
            memset(&nl, 0, sizeof nl);
            nl.mapA = cl.mapA;
            b2k::NetLayerInfo& f = nl.info;
            f.wpacked = a.wpacked, f.bias = a.bias, f.out = a.out, f.residual = a.residual;
            f.M = a.M, f.Cout = a.Cout, f.num_kblocks = a.num_kblocks, f.cblocks = a.cblocks;
            f.kw = a.kw, f.HoWo = a.HoWo, f.Wo = a.Wo, f.stride_h = a.stride_h, f.stride_w = a.stride_w;
            f.pad_h = a.pad_h, f.pad_w = a.pad_w, f.relu = a.relu, f.a_mode = a.a_mode;
            f.bn = cl.bn, f.tiles_m = cl.grid_m, f.tiles_n = cl.grid_n;
            f.tile_begin = tile_cursor, f.total_tiles = cl.grid_m * cl.grid_n;
            tile_cursor += f.total_tiles;
            f.out_flag_off = flag_cursor;
            flag_cursor += f.tiles_m;
            f.in_flag_off = f.res_flag_off = -1;
            auto pin = producer.find(r.in);
            if (pin != producer.end()) f.in_flag_off = layers[pin->second].info.out_flag_off, f.in_need = layers[pin->second].info.tiles_n;
            if (r.res >= 0) {
                auto pres = producer.find(r.res);
                if (pres != producer.end())
                    f.res_flag_off = layers[pres->second].info.out_flag_off, f.res_need = layers[pres->second].info.tiles_n;
            }
            // input M tiles read by each output M tile (a superset: whole rows once the window is clipped)
            f.dep_off = int(deps.size());
            const Tensor& ti = e->tensors[r.in];
            const Tensor& to = e->tensors[r.out];
            const int Hin = int(ti.h), Win = int(ti.w), Wo = int(to.w), HoWo = int(to.h * to.w);
            const int in_tiles = (batch * Hin * Win + 127) / 128;
            for (int mt = 0; mt < f.tiles_m; ++mt) {
                const int m_lo = mt * 128, m_hi = std::min(m_lo + 127, f.M - 1);
                const int n0 = m_lo / HoWo, p0 = (m_lo % HoWo) / Wo, q0 = m_lo % Wo;
                const int n1 = m_hi / HoWo, p1 = (m_hi % HoWo) / Wo, q1 = m_hi % Wo;
                int lr = p0 * op.sh() - op.ph(), lc = q0 * op.sw() - op.pw_lo();
                if (lr < 0) lr = 0, lc = 0;
                if (lc < 0) lc = 0;
                int hr = p1 * op.sh() - op.ph() + op.kh() - 1, hc = q1 * op.sw() - op.pw_lo() + op.kw() - 1;
                if (hr > Hin - 1) hr = Hin - 1, hc = Win - 1;
                if (hc > Win - 1) hc = Win - 1;
                const int lo = (n0 * Hin * Win + lr * Win + lc) / 128;
                const int hi = std::min((n1 * Hin * Win + hr * Win + hc) / 128, in_tiles - 1);
                deps.push_back(make_short2(short(lo), short(std::max(lo, hi))));
            }
            // recycled arena memory: every earlier layer of the run that read or wrote bytes this layer will overwrite
            size_t olo, ohi;
            trange(r.out, &olo, &ohi);
            f.war_upto = -1;
            for (int q = 0; q < l; ++q) {
                const b2plan::OpRec& rq = e->ops[i + q].r;
                for (int u : {rq.in, rq.res, rq.out}) {
                    if (u < 0 || u == r.out || e->tensors[u].binding >= 0) continue;
                    size_t ulo, uhi;
                    trange(u, &ulo, &uhi);
                    if (ulo < ohi && olo < uhi) f.war_upto = q;
                }
            }
            producer[r.out] = l;
            flops += ls[i + l].flops, bytes += ls[i + l].bytes;
        }
        for (int l = 0; l < n; ++l)
            if (layers[l].info.tiles_m > 32767) return fail(B2_EINVAL, "layer too large for the persistent kernel (M tiles > 32767)");
        auto run = std::make_shared<NetRun>();
        const size_t off_layers = 0;
        const size_t off_deps = align_up(off_layers + size_t(n) * sizeof(b2k::NetLayer), 256);
        const size_t off_mt = align_up(off_deps + deps.size() * sizeof(short2), 256);
        const size_t off_ld = off_mt + size_t(flag_cursor) * sizeof(int);
        const size_t off_ctrl = off_ld + size_t(n) * sizeof(int);
        const size_t total = off_ctrl + 2 * sizeof(int);
        if (cudaMalloc(&run->d_blob, total) != cudaSuccess) {
            cudaGetLastError();
            return fail(B2_ENOMEM, "cudaMalloc(%zu) for the persistent-kernel tables failed", total);
        }
        uint8_t* d = static_cast<uint8_t*>(run->d_blob);
        {   // on a private non-blocking stream: other threads may be capturing graphs, which forbids legacy-stream work
            cudaStream_t up = nullptr;
            B2_CUDA(cudaStreamCreateWithFlags(&up, cudaStreamNonBlocking));
            cudaError_t ue = cudaMemsetAsync(d, 0, total, up);
            if (ue == cudaSuccess) ue = cudaMemcpyAsync(d + off_layers, layers.data(), size_t(n) * sizeof(b2k::NetLayer), cudaMemcpyHostToDevice, up);
            if (ue == cudaSuccess) ue = cudaMemcpyAsync(d + off_deps, deps.data(), deps.size() * sizeof(short2), cudaMemcpyHostToDevice, up);
            if (ue == cudaSuccess) ue = cudaStreamSynchronize(up);
            cudaStreamDestroy(up);
            if (ue != cudaSuccess) return fail(B2_ECUDA, "upload of the persistent-kernel tables failed: %s", cudaGetErrorString(ue));
        }
        run->args.layers = reinterpret_cast<const b2k::NetLayer*>(d + off_layers);
        run->args.deps = reinterpret_cast<const short2*>(d + off_deps);
        run->args.mt_done = reinterpret_cast<int*>(d + off_mt);
        run->args.layer_done = reinterpret_cast<int*>(d + off_ld);
        run->args.ctrl = reinterpret_cast<int*>(d + off_ctrl);
        run->args.n_layers = n, run->args.total_tiles = tile_cursor, run->args.n_flags = flag_cursor;
        // ring depth: the deepest that still lets two CTAs share an SM (227 KiB less 1 KiB of system use per CTA)
        int stages = c->net_stages > 0 ? c->net_stages : 4;
        while (c->net_stages <= 0 && stages > 2 && 2 * (b2k::net_smem_bytes(n, stages) + 1024) > 227 * 1024) --stages;
        run->args.stages = std::max(2, std::min(stages, 4));
        const int per_sm = 2 * (b2k::net_smem_bytes(n, run->args.stages) + 1024) <= 227 * 1024 ? 2 : 1;
        run->ctas = c->net_ctas > 0 ? c->net_ctas : 148 * per_sm;
        run->ctas = std::max(1, std::min(run->ctas, std::min(148 * per_sm, tile_cursor)));
        run->first_op = int(i), run->last_op = int(j);
        Launch L;
        L.kind = L_NET;
        L.name = ls[i].name + ".." + ls[j].name;
        L.flops = flops, L.bytes = bytes;
        L.N = batch;
        L.net = run;
        fused.push_back(std::move(L));
        i = j + 1;
    }
    for (Launch& L : fused) L.side_join = -1;  // launch indices no longer equal op indices: no forked side branches
    ls = std::move(fused);
    plan->has_net = true;
    return B2_OK;
}

// global average pool -> FC -> softmax (the classifier tail) as one launch; the pooled tensor and the logits vector of
// the plan serve as its scratch, so tapping them as outputs still works.
void fuse_tail(b2_context* c, Plan* plan, int batch) {
    if (!c->fuse_tail || !c->e->half()) return;
    std::vector<Launch>& ls = plan->launches;
    for (size_t i = 0; i + 2 < ls.size(); ++i) {
        const Launch &P = ls[i], &F = ls[i + 1], &S = ls[i + 2];
        if (P.kind != L_AVGPOOL || F.kind != L_FC || S.kind != L_SOFTMAX) continue;
        if (F.in != P.out || S.in != F.out || F.out_binding >= 0 || S.in_binding >= 0 || S.out_binding < 0 || P.C_phys % 8) continue;
        if (F.K != P.C_phys || S.C != F.Cout || !b2k::tail_f16_applies(batch, P.H * P.W, P.C_phys, F.Cout)) continue;
        Launch T;
        T.kind = L_TAIL;
        T.name = P.name + "+" + F.name + "+" + S.name;
        T.N = batch;
        T.flops = F.flops, T.bytes = P.bytes + F.bytes + S.bytes;
        T.out_binding = S.out_binding;
        T.tail.in = static_cast<const __half*>(P.in);
        T.tail.w = static_cast<const __half*>(F.w);
        T.tail.bias = F.bias;
        T.tail.pooled = static_cast<__half*>(P.out);
        T.tail.logits = static_cast<float*>(F.out);
        T.tail.ctrl = c->d_tail_ctrl;
        T.tail.N = batch, T.tail.HW = P.H * P.W, T.tail.C = P.C_phys, T.tail.Cout = F.Cout;
        ls[i] = std::move(T);
        ls.erase(ls.begin() + long(i) + 1, ls.begin() + long(i) + 3);  // (launches before i keep their indices: side joins stay valid)
        return;
    }
}

// ---- per-batch launch plan ---------------------------------------------------------------------
int build_plan(b2_context* c, int batch, Plan** out) {
    b2_engine* e = c->e;
    if (!c->scratch || !c->cur) return fail(B2_ESTATE, "b2_context_set_device_memory has not been called");
    auto it = c->cur->plans.find(batch);
    if (it != c->cur->plans.end()) {
        *out = it->second.get();
        return B2_OK;
    }
    if (load_driver_entry_points() != 0) return fail(B2_ECUDA, "cuTensorMapEncode* driver entry points unavailable");
    auto plan = std::make_unique<Plan>();
    plan->batch = batch;
    const bool half = e->half();
    const size_t elt = half ? 2 : 4;
    auto tptr = [&](int ti) -> uint8_t* {
        const Tensor& t = e->tensors[ti];
        return t.binding >= 0 ? nullptr : c->scratch + t.offset;
    };
    for (const Op& op : e->ops) {
        const b2plan::OpRec& r = op.r;
        Launch L;
        L.name = op.name;
        L.N = batch;
        L.side_join = op.side_join;
        switch (r.type) {
            case b2plan::OP_INPUT_CAST: {
                const Tensor& t = e->tensors[r.out];
                L.kind = L_INPUT_CAST;
                L.in_binding = r.binding;
                const Binding& b = e->bindings[r.binding];
                L.src_dtype = b.dtype;
                L.out = tptr(r.out);
                L.C = t.c, L.H = t.h, L.W = t.w, L.C_phys = t.c_phys;
                L.k = int(r.k);  // 2: horizontal space-to-depth (tensor is [H, W/2, 8]; binding is [C, H, W] or [src_h, src_w, C])
                L.max_blocks = c->input_ctas;
                if (b.dtype == B2_DT_UINT8) {  // {src_h, src_w, C} cropped to the tensor's H x W (validated at load)
                    L.norm = b.norm;
                    L.C = b.norm.C;
                    if (!half || t.c_phys != 8 || (r.k != 2 && int(t.c) != L.C))
                        return fail(B2_EINVAL, "input cast %s: a uint8 binding needs the fp16 8-channel input layout", op.name.c_str());
                }
                if (r.k == 2) {  // pad_ / stride = zero pixels written left / right of every packed row
                    const bool u8 = b.dtype == B2_DT_UINT8;
                    const int C = u8 ? b.dims[2] : b.dims[0], H = u8 ? int(t.h) : b.dims[1];
                    const int W = u8 ? 2 * (int(t.w) - int(r.pad_) - int(r.stride)) : b.dims[2];
                    if (!half || b.nd != 3 || C > 4 || t.c_phys != 8 || int(t.h) != H || W < 2 ||
                        int(t.w) != W / 2 + int(r.pad_) + int(r.stride) || W % 2)
                        return fail(B2_EINVAL, "input cast %s: inconsistent space-to-depth geometry", op.name.c_str());
                    L.C = C, L.W = W;
                    L.pad = int(r.pad_), L.stride = int(r.stride);
                }
                if (b.dtype == B2_DT_UINT8)  // the crop's bytes in, the padded fp16 tensor out
                    L.bytes = double(batch) * (double(L.H) * L.W * L.C + double(t.h) * t.w * t.c_phys * elt);
                else
                    L.bytes = double(batch) * t.h * t.w * (t.c * 4.0 + t.c_phys * elt);
                break;
            }
            case b2plan::OP_QUANTIZE: {
                const Tensor& ti = e->tensors[r.in];
                const Tensor& to = e->tensors[r.out];
                L.kind = L_QUANTIZE;
                L.in = tptr(r.in), L.out = tptr(r.out);
                L.C = ti.c, L.H = ti.h, L.W = ti.w, L.C_in_phys = ti.c_phys, L.C_phys = to.c_phys;
                L.qscale = float(1.0 / double(to.scale));
                L.bytes = double(batch) * (ti.item_bytes + to.item_bytes);
                break;
            }
            case b2plan::OP_OUTPUT_CAST: {
                const Tensor& t = e->tensors[r.in];
                L.kind = t.scale > 0.f ? L_OUTPUT_CAST_I8 : L_OUTPUT_CAST;
                L.qscale = t.scale;
                L.in = tptr(r.in);
                L.out_binding = r.binding;
                L.C = t.c, L.H = t.h, L.W = t.w, L.C_phys = t.c_phys;
                L.bytes = double(batch) * t.h * t.w * (t.c * 4.0 + t.c_phys * elt);
                break;
            }
            case b2plan::OP_CONV: {
                const Tensor& ti = e->tensors[r.in];
                const Tensor& to = e->tensors[r.out];
                const uint8_t* w = e->d_payload + r.w_off;
                const float* bias = reinterpret_cast<const float*>(e->d_payload + r.b_off);
                const int M = batch * int(to.h) * int(to.w);
                L.flops = 2.0 * M * r.cout * op.algo_k();
                L.bytes = double(batch) * (ti.item_bytes + to.item_bytes * (r.res >= 0 ? 2 : 1)) + double(r.w_bytes);
                const bool kb64 = r.cin_phys % 64 == 0;
                const bool kb8 = r.cin_phys == 8;
                const bool tc_ok = half && !c->force_simt && (kb64 || kb8) && r.cout_phys % 32 == 0 &&
                                   (kb64 || r.taps_phys % 2 == 0);
                if (r.relu & 4) {  // INT8 tensor path
                    L.kind = L_CONV_I8;
                    // one tactic, by rule: the 128-wide N tile with a ring no deeper than the K loop, shallow enough (2-3
                    // stages) that two CTAs share an SM (measured: profiles/probe_r2_int8_*.log); "i8_bn" / "i8_stages" override
                    // tactic = (N tile, ring depth): timed at load (b2_engine_tune) or carried by the plan; untuned engines use
                    // a rule -- many CTAs want shallow rings (more CTAs per SM), few CTAs a 2-deep one (profiles/probe_r2_int8*)
                    const int m_tiles = (batch * int(e->tensors[r.out].h * e->tensors[r.out].w) + 127) / 128;
                    int bn = 128, st = m_tiles * (int(r.cout_phys) / 128) >= 2 * 148 ? 1 : 2;
                    if (c->autotune) {
                        std::lock_guard<std::mutex> lock(e->tune_mutex);
                        tune_cache_load(e);
                        const int op_index = int(&op - &e->ops[0]);
                        auto it = e->tuned.find({op_index, batch});
                        if (it == e->tuned.end()) it = e->tuned.find({op_index, e->max_batch});
                        if (it != e->tuned.end()) bn = it->second.bn, st = it->second.stages;
                    }
                    if (c->i8_bn > 0) bn = c->i8_bn;
                    if (c->i8_stages > 0) st = c->i8_stages;
                    if (int(r.cout_phys) % bn) bn = 128;
                    if (!b2k::conv_i8_config_exists(bn, st)) bn = 128, st = 2;
                    int rc = make_i8_conv_launch(c, op, batch, bn, st, &L.i8);
                    if (rc) return rc;
                } else if (tc_ok) {
                    L.kind = L_CONV_TC;
                    const int kbsz = conv_kb(c, op);
                    const int nkb = conv_num_kblocks(c, op);
                    ConvConfig cfg = pick_conv_config(M, int(r.cout_phys), nkb, kbsz, r.res >= 0, c, true);
                    if (cfg.bn == 0)  // a forced tile that does not divide this layer: fall back to the model
                        cfg = pick_conv_config(M, int(r.cout_phys), nkb, kbsz, r.res >= 0, c, false);
                    if (cfg.bn == 0) return fail(B2_EINVAL, "conv %s: no kernel configuration", op.name.c_str());
                    if (c->force_sps == 2 && b2k::conv_config_exists(cfg.bn, kbsz, cfg.stages, 2) &&
                        b2k::conv_smem_bytes(cfg.bn, cfg.stages, r.res >= 0, 2) <= 227 * 1024)
                        cfg.sps = 2;
                    if (c->force_ws > 0 && kbsz == 64 && (r.relu & 2) && cfg.splits == 1 &&
                        b2k::conv_ws_config_exists(cfg.bn, cfg.stages, cfg.sps) &&
                        b2k::conv_ws_smem(cfg.bn, cfg.stages, cfg.sps, r.res >= 0) <= 227 * 1024)
                        cfg.ws = std::min(((M + 127) / 128) * (int(r.cout_phys) / cfg.bn), c->force_ws > 1 ? c->force_ws : 148);
                    if (c->force_halo > 0 && conv_halo_rows(c, op) && b2k::conv_halo_config_exists(cfg.bn) && cfg.splits == 1 &&
                        int(r.cin_phys) / 64 <= 8 && b2k::conv_halo_smem(cfg.bn, int(to.w), conv_halo_rows(c, op), int(r.cin_phys) / 64) <= 227 * 1024)
                        cfg.halo = 1, cfg.ws = 0, cfg.cn = 1;
                    if (c->force_cn > 1 && kbsz == 64 && cfg.ws == 0 && !cfg.halo && (int(r.cout_phys) / cfg.bn) % c->force_cn == 0) cfg.cn = c->force_cn;
                    const bool forced = c->force_bn || c->force_stages || c->force_splits || c->force_sps;
                    const int op_index = int(&op - &e->ops[0]);
                    // member of a persistent-kernel run: 64-channel K blocks, packed weights, 64 | Cout; no tactic to tune
                    const bool net_ok = c->net && !forced && kbsz == 64 && (r.relu & 2) && !c->no_pack && r.cout_phys % 64 == 0 &&
                                        c->force_ws <= 0 && c->force_cn <= 0 && c->force_halo <= 0 && !c->force_im2col;
                    if (net_ok) {
                        int bn = (r.cout_phys % 128 == 0) ? 128 : 64;
                        if (c->net_bn == 64) bn = 64;
                        cfg = ConvConfig{bn, 4, 1, 0.0, 1, 0, 1};
                        cfg.halo = 0;
                        L.net_member = true;
                    } else if (!forced && c->autotune) {
                        // Tactics are measured ahead of time (b2_engine_tune at model registration, or the table the plan
                        // blob carries) -- never here, on the request path.  A batch size that was not tuned itself uses
                        // the max-batch tactic (every tactic is valid for every batch; the split-K factor is shared by
                        // construction, so an image's result does not depend on its batch); no entry at all = cost model.
                        std::lock_guard<std::mutex> lock(e->tune_mutex);
                        tune_cache_load(e);
                        auto it = e->tuned.find({op_index, batch});
                        if (it == e->tuned.end()) it = e->tuned.find({op_index, e->max_batch});
                        if (it != e->tuned.end() && tactic_applies(c, op, batch, it->second)) cfg = it->second;
                    }
                    if (op.side_join >= 0 && cfg.splits > 1) cfg.splits = 1;  // forced / cached tactic on a side-branch op
                    int rc = make_conv_launch(c, op, batch, cfg, &L.conv);
                    if (rc) return rc;
                } else {
                    L.kind = L_CONV_SIMT;
                    b2k::SimtConvArgs& a = L.simt;
                    memset(&a, 0, sizeof a);
                    a.in = tptr(r.in), a.w = w, a.bias = bias;
                    a.residual = r.res >= 0 ? tptr(r.res) : nullptr;
                    a.out = tptr(r.out);
                    a.N = batch, a.H = int(ti.h), a.W = int(ti.w), a.Cin = int(r.cin), a.Cin_phys = int(r.cin_phys);
                    a.Ho = int(to.h), a.Wo = int(to.w), a.Cout = int(r.cout), a.Cout_phys = int(r.cout_phys);
                    a.kh = op.kh(), a.kw = op.kw(), a.taps_phys = int(r.taps_phys);
                    a.stride_h = op.sh(), a.stride_w = op.sw(), a.pad_h = op.ph(), a.pad_w = op.pw_lo();
                    a.relu = int(r.relu & 1);
                    a.w_packed = int((r.relu >> 1) & 1);
                }
                break;
            }
            case b2plan::OP_MAXPOOL: {
                const Tensor& ti = e->tensors[r.in];
                const Tensor& to = e->tensors[r.out];
                L.kind = L_MAXPOOL;
                L.in = tptr(r.in), L.out = tptr(r.out);
                L.H = ti.h, L.W = ti.w, L.C_phys = ti.c_phys, L.Ho = to.h, L.Wo = to.w;
                L.k = r.k, L.stride = r.stride, L.pad = r.pad_;
                L.bytes = double(batch) * (ti.item_bytes + to.item_bytes);
                break;
            }
            case b2plan::OP_AVGPOOL: {
                const Tensor& ti = e->tensors[r.in];
                L.kind = ti.scale > 0.f ? L_AVGPOOL_I8 : L_AVGPOOL;
                L.in = tptr(r.in), L.out = tptr(r.out);
                L.H = ti.h, L.W = ti.w, L.C_phys = ti.c_phys;
                if (ti.scale > 0.f) {  // int8 in, fp16 out
                    L.C = ti.c, L.C_in_phys = ti.c_phys, L.C_phys = e->tensors[r.out].c_phys;
                    L.qscale = float(double(ti.scale) / double(ti.h * ti.w));
                }
                L.bytes = double(batch) * ti.item_bytes;
                break;
            }
            case b2plan::OP_FC: {
                const Tensor& ti = e->tensors[r.in];
                const Tensor& to = e->tensors[r.out];
                L.kind = L_FC;
                L.in = tptr(r.in);
                L.out = tptr(r.out);
                L.out_binding = to.binding;
                L.w = e->d_payload + r.w_off;
                L.bias = reinterpret_cast<const float*>(e->d_payload + r.b_off);
                L.K = int(ti.h * ti.w * ti.c_phys);
                L.Cout = int(r.cout);
                L.flops = 2.0 * batch * ti.h * ti.w * ti.c * r.cout;
                L.bytes = double(r.w_bytes) + double(batch) * (ti.item_bytes + to.item_bytes);
                break;
            }
            case b2plan::OP_SOFTMAX: {
                const Tensor& ti = e->tensors[r.in];
                const Tensor& to = e->tensors[r.out];
                L.kind = L_SOFTMAX;
                L.in = tptr(r.in);
                L.in_binding = ti.binding;
                L.out = tptr(r.out);
                L.out_binding = to.binding;
                L.C = int(ti.c);
                L.bytes = double(batch) * ti.c * 8.0;
                break;
            }
            default:
                return fail(B2_EINVAL, "op %s: unknown type", op.name.c_str());
        }
        plan->launches.push_back(std::move(L));
    }
    int rc = fuse_net_runs(c, plan.get(), batch);
    if (rc) return rc;
    fuse_tail(c, plan.get(), batch);
    {   // split into binding-dependent launches and binding-independent (graphable) runs
        const std::vector<Launch>& ls = plan->launches;
        size_t i = 0;
        while (i < ls.size()) {
            const bool dep = ls[i].in_binding >= 0 || ls[i].out_binding >= 0;
            size_t j = i + 1;
            if (!dep)
                while (j < ls.size() && ls[j].in_binding < 0 && ls[j].out_binding < 0) ++j;
            Segment sg;
            sg.begin = int(i), sg.end = int(j);
            sg.graphable = !dep && (j - i) >= 3 && !plan->has_net;
            plan->segments.push_back(sg);
            i = j;
        }
    }
    *out = plan.get();
    c->cur->plans[batch] = std::move(plan);
    return B2_OK;
}

int run_launch(const b2_engine* e, const Launch& L, void* const* bindings, cudaStream_t s) {
    const bool half = e->half();
    const void* in = L.in_binding >= 0 ? bindings[L.in_binding] : L.in;
    void* out = L.out_binding >= 0 ? bindings[L.out_binding] : L.out;
    switch (L.kind) {
        case L_INPUT_CAST:
            if (L.src_dtype == B2_DT_UINT8) {
                if (L.k == 2) return b2k::launch_input_cast_u8_s2d(in, out, L.N, L.H, L.W, L.pad, L.stride, L.norm, L.max_blocks, s);
                return b2k::launch_input_cast_u8_c8(in, out, L.N, L.H, L.W, L.norm, L.max_blocks, s);
            }
            if (L.k == 2)
                return b2k::launch_input_cast_s2d(in, L.src_dtype == B2_DT_HALF, out, L.N, L.C, L.H, L.W, L.pad, L.stride, L.max_blocks, s);
            return b2k::launch_input_cast(in, L.src_dtype == B2_DT_HALF, out, L.N, L.C, L.H, L.W, L.C_phys, half, L.max_blocks, s);
        case L_OUTPUT_CAST:
            return b2k::launch_output_cast(in, static_cast<float*>(out), L.N, L.C, L.H, L.W, L.C_phys, half, s);
        case L_CONV_TC:
            return b2k::launch_conv_f16_tcgen05(L.conv, s);
        case L_CONV_SIMT:
            return b2k::launch_conv_simt(L.simt, half, s);
        case L_MAXPOOL:
            return b2k::launch_maxpool(in, out, L.N, L.H, L.W, L.C_phys, L.Ho, L.Wo, L.k, L.stride, L.pad, half, s);
        case L_AVGPOOL:
            return b2k::launch_avgpool(in, out, L.N, L.H * L.W, L.C_phys, half, s);
        case L_FC:
            return b2k::launch_fc(in, L.w, L.bias, static_cast<float*>(out), L.N, L.K, L.Cout, half, s);
        case L_SOFTMAX:
            return b2k::launch_softmax(static_cast<const float*>(in), static_cast<float*>(out), L.N, L.C, s);
        case L_NET:
            return b2k::launch_net_f16_tcgen05(L.net->args, L.net->ctas, s);
        case L_QUANTIZE:
            return b2k::launch_quantize_h_to_i8(in, out, static_cast<long long>(L.N) * L.H * L.W, L.C, L.C_in_phys, L.C_phys, L.qscale, s);
        case L_CONV_I8:
            return b2k::launch_conv_i8_tcgen05(L.i8, s);
        case L_AVGPOOL_I8:
            return b2k::launch_avgpool_i8(in, out, L.N, L.H * L.W, L.C, L.C_in_phys, L.C_phys, L.qscale, s);
        case L_OUTPUT_CAST_I8:
            return b2k::launch_output_cast_i8(in, static_cast<float*>(out), L.N, L.C, L.H, L.W, L.C_phys, L.qscale, s);
        case L_TAIL: {
            b2k::TailArgs t = L.tail;
            t.out = static_cast<float*>(out);
            return b2k::launch_tail_f16(t, s);
        }
    }
    return int(cudaErrorInvalidValue);
}

// Launches the plan on `s`.  Side branches go to the context's second stream between a fork and a join event: inside
// a stream capture that becomes a parallel branch of the graph, outside it is plain two-stream concurrency.
int run_range(b2_context* c, const Plan& plan, size_t first, size_t last, void* const* bindings, cudaStream_t s);
int run_all(b2_context* c, const Plan& plan, void* const* bindings, cudaStream_t s) {
    return run_range(c, plan, 0, plan.launches.size(), bindings, s);
}
int run_range(b2_context* c, const Plan& plan, size_t first, size_t last, void* const* bindings, cudaStream_t s) {
    const b2_engine* e = c->e;
    bool fork = c->fork != 0;
    if (fork && !c->side) {
        if (cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->fork_ev, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->join_ev, cudaEventDisableTiming) != cudaSuccess) {
            cudaGetLastError();
            fork = false;
        }
    }
    int pending_join = -1;
    for (size_t i = first; i < last; ++i) {
        const Launch& L = plan.launches[i];
        if (pending_join == int(i)) {
            B2_CUDA(cudaStreamWaitEvent(s, c->join_ev, 0));
            pending_join = -1;
        }
        int rc;
        if (fork && pending_join < 0 && L.side_join > int(i) && L.side_join < int(last)) {
            B2_CUDA(cudaEventRecord(c->fork_ev, s));
            B2_CUDA(cudaStreamWaitEvent(c->side, c->fork_ev, 0));
            rc = run_launch(e, L, bindings, c->side);
            if (rc == 0) {
                B2_CUDA(cudaEventRecord(c->join_ev, c->side));
                pending_join = L.side_join;
            }
        } else {
            rc = run_launch(e, L, bindings, s);
        }
        if (rc != 0)
            return fail(B2_ECUDA, "launch of %s failed: %s", L.name.c_str(), cudaGetErrorString(cudaError_t(rc)));
    }
    if (pending_join >= 0) B2_CUDA(cudaStreamWaitEvent(s, c->join_ev, 0));  // never leave the branch dangling
    return B2_OK;
}

// Captures launches [begin, end) of the plan -- none of which touches a binding -- on `stream` (which must be idle-able:
// capture only records) and instantiates the graph once for the life of the plan.
int instantiate_segment(b2_context* c, Plan* plan, Segment* sg, void* const* bindings, cudaStream_t stream) {
    cudaGraph_t graph = nullptr;
    B2_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    int rc = run_range(c, *plan, size_t(sg->begin), size_t(sg->end), bindings, stream);
    cudaError_t ce = cudaStreamEndCapture(stream, &graph);
    if (rc) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
    }
    if (ce != cudaSuccess) return fail(B2_ECUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
    ce = cudaGraphInstantiate(&sg->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) {
        sg->exec = nullptr;
        return fail(B2_ECUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce));
    }
    return B2_OK;
}

// Which argument of a binding-dependent launch carries the binding pointer (positions in the kernels' parameter lists,
// kernels.cu) and how many arguments the kernel has.
bool patch_layout(const b2_engine* e, const Launch& L, BindPatch* p) {
    const bool half = e->half();
    switch (L.kind) {
        case L_INPUT_CAST:
            if (L.src_dtype == B2_DT_UINT8 && L.k == 2) p->n_params = 8;    // input_cast_u8_s2d_kernel(src, dst, N, H, W, pad_l, pad_r, nrm)
            else if (L.src_dtype == B2_DT_UINT8) p->n_params = 6;           // input_cast_u8_c8_kernel(src, dst, N, H, W, nrm)
            else if (L.k == 2) p->n_params = 8;                             // input_cast_s2d_kernel(src, dst, N, C, H, W, pad_l, pad_r)
            else if (half && L.C_phys == 8 && L.C <= 8) p->n_params = 5;    // input_cast_c8_kernel(src, dst, N, C, HW)
            else p->n_params = 6;                                           // input_cast_kernel(src, dst, N, C, HW, C_phys)
            p->in_index = 0;
            return true;
        case L_OUTPUT_CAST:
            p->n_params = 6, p->out_index = 1;                              // output_cast_kernel(src, dst, N, C, HW, C_phys)
            return true;
        case L_OUTPUT_CAST_I8:
            p->n_params = 7, p->out_index = 1;                              // output_cast_i8_kernel(src, dst, N, C, HW, C_phys, s)
            return true;
        case L_FC:
            p->n_params = 7, p->out_index = 3;                              // fc kernels (in, w, bias, out, N, K, Cout)
            return L.in_binding < 0;
        case L_SOFTMAX:
            p->n_params = 3;                                                // softmax_kernel(in, out, C)
            if (L.in_binding >= 0) p->in_index = 0;
            if (L.out_binding >= 0) p->out_index = 1;
            return true;
        case L_TAIL:
            p->n_params = 1, p->is_tail = true, p->tail = L.tail;
            return true;
        default:
            return false;
    }
}

// Captures the WHOLE plan once (programmatic edges between all kernels survive) and remembers the kernel nodes that touch
// a binding.  Returns B2_OK with plan->exec == nullptr if the plan cannot be patched (then graph mode 3 takes over).
int instantiate_plan_graph(b2_context* c, Plan* plan, void* const* bindings, cudaStream_t stream) {
    std::vector<BindPatch> patches;
    cudaGraph_t graph = nullptr;
    bool patchable = true;
    B2_CUDA(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    int rc = B2_OK;
    for (size_t i = 0; i < plan->launches.size() && !rc; ++i) {
        const Launch& L = plan->launches[i];
        rc = run_range(c, *plan, i, i + 1, bindings, stream);
        if (rc || (L.in_binding < 0 && L.out_binding < 0)) continue;
        BindPatch p;
        p.launch = int(i);
        if (!patch_layout(c->e, L, &p)) {
            patchable = false;
            continue;
        }
        cudaStreamCaptureStatus st;
        const cudaGraphNode_t* deps = nullptr;
        size_t ndeps = 0;
        if (cudaStreamGetCaptureInfo_v2(stream, &st, nullptr, nullptr, &deps, &ndeps) != cudaSuccess || ndeps != 1) {
            cudaGetLastError();
            patchable = false;
            continue;
        }
        p.node = deps[0];
        patches.push_back(p);
    }
    cudaError_t ce = cudaStreamEndCapture(stream, &graph);
    if (rc) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
    }
    if (ce != cudaSuccess) return fail(B2_ECUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
    for (BindPatch& p : patches) {
        cudaGraphNodeType ty;
        if (!patchable || cudaGraphNodeGetType(p.node, &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel ||
            cudaGraphKernelNodeGetParams(p.node, &p.np) != cudaSuccess || p.np.kernelParams == nullptr) {
            cudaGetLastError();
            patchable = false;
            break;
        }
        p.params.assign(p.np.kernelParams, p.np.kernelParams + p.n_params);
    }
    if (!patchable) {
        cudaGraphDestroy(graph);
        return B2_OK;
    }
    cudaGraphExec_t exec = nullptr;
    ce = cudaGraphInstantiate(&exec, graph, 0);
    if (ce != cudaSuccess) {
        cudaGraphDestroy(graph);
        return fail(B2_ECUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce));
    }
    plan->graph = graph, plan->exec = exec, plan->patches = std::move(patches);
    // the values captured are the ones the graph holds now
    for (BindPatch& p : plan->patches) {
        const Launch& L = plan->launches[size_t(p.launch)];
        p.in_value = L.in_binding >= 0 ? bindings[L.in_binding] : nullptr;
        p.out_value = L.out_binding >= 0 ? bindings[L.out_binding] : nullptr;
    }
    return B2_OK;
}

// Points the binding-dependent nodes at this request's buffers (no-op for pointers the graph already holds).
int patch_plan_graph(Plan* plan, void* const* bindings) {
    for (BindPatch& p : plan->patches) {
        const Launch& L = plan->launches[size_t(p.launch)];
        void* in = L.in_binding >= 0 ? bindings[L.in_binding] : nullptr;
        void* out = L.out_binding >= 0 ? bindings[L.out_binding] : nullptr;
        if (in == p.in_value && out == p.out_value) continue;
        p.in_value = in, p.out_value = out;
        if (p.is_tail) {
            p.tail.out = static_cast<float*>(out);
            p.params[0] = &p.tail;
        } else {
            if (p.in_index >= 0) p.params[size_t(p.in_index)] = &p.in_value;
            if (p.out_index >= 0) p.params[size_t(p.out_index)] = &p.out_value;
        }
        cudaKernelNodeParams np = p.np;
        np.kernelParams = p.params.data();
        np.extra = nullptr;
        B2_CUDA(cudaGraphExecKernelNodeSetParams(plan->exec, p.node, &np));
    }
    return B2_OK;
}

int check_args(b2_context* c, int batch, void* const* bindings) {
    if (!c || !bindings) return fail(B2_EINVAL, "null context or bindings");
    if (batch < 1 || batch > c->e->max_batch) return fail(B2_EINVAL, "batch %d outside [1, %d]", batch, c->e->max_batch);
    for (size_t i = 0; i < c->e->bindings.size(); ++i)
        if (!bindings[i]) return fail(B2_EINVAL, "binding %zu (%s) is null", i, c->e->bindings[i].name.c_str());
    return B2_OK;
}

}  // namespace

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int b2_abi_version(void) { return B2_ABI_VERSION; }
const char* b2_last_error(void) { return g_err.c_str(); }

int b2_runtime_create(b2_runtime** out) {
    if (!out) return fail(B2_EINVAL, "null out");
    *out = new b2_runtime();
    return B2_OK;
}
void b2_runtime_destroy(b2_runtime* rt) { delete rt; }

int b2_runtime_set_allocator(b2_runtime* rt, b2_alloc_fn alloc, b2_free_fn free_, void* user) {
    if (!rt) return fail(B2_EINVAL, "null runtime");
    if ((alloc == nullptr) != (free_ == nullptr)) return fail(B2_EINVAL, "alloc and free must be set together");
    rt->alloc = alloc, rt->free_ = free_, rt->user = user;
    return B2_OK;
}

static int deserialize_impl(b2_runtime* rt, const void* blob, size_t nbytes, bool inspect_only, b2_engine** out) {
    if (!out) return fail(B2_EINVAL, "null out");
    *out = nullptr;
    std::unique_ptr<b2_engine> e(new b2_engine());
    e->rt = rt;
    e->inspect_only = inspect_only;
    const uint8_t* payload = nullptr;
    int rc = parse_blob(blob, nbytes, e.get(), &payload);
    if (rc) return rc;
    for (size_t i = 0; i < e->ops.size(); ++i) {  // the fused-residual rescale factor is a kernel ARGUMENT: keep a host copy
        const b2plan::OpRec& r = e->ops[i].r;
        if (r.type == b2plan::OP_CONV && (r.relu & 4)) {
            float rr = 0.f;
            memcpy(&rr, payload + r.b_off + size_t(r.cout_phys) * 8, sizeof rr);
            e->requant_r[int(i)] = rr;
        }
    }
    plan_arena(e.get());
    if (!inspect_only) {
        int dev = -1;
        if (cudaGetDevice(&dev) != cudaSuccess) {
            cudaGetLastError();
            return fail(B2_ENODEVICE, "no CUDA device available (this engine has no CPU fallback)");
        }
        cudaDeviceProp prop;
        B2_CUDA(cudaGetDeviceProperties(&prop, dev));
        if (prop.major != 10)
            return fail(B2_ENODEVICE, "device %d is sm_%d%d; this library only carries sm_100a code", dev, prop.major, prop.minor);
        e->device = dev;
        rc = b2k::init_conv_kernels();
        if (!rc) rc = b2k::init_net_kernel();
        if (!rc) rc = b2k::init_conv_i8_kernels();
        if (rc) return fail(B2_ECUDA, "kernel attribute setup failed: %s", cudaGetErrorString(cudaError_t(rc)));
        const size_t bytes = std::max<size_t>(e->payload_bytes, 256);
        if (rt && rt->alloc) {
            e->alloc = rt->alloc, e->free_ = rt->free_, e->alloc_user = rt->user;
            e->d_payload = static_cast<uint8_t*>(rt->alloc(rt->user, bytes, 256, 0));
            if (!e->d_payload) return fail(B2_ENOMEM, "user allocator returned null for %zu weight bytes", bytes);
        } else {
            void* p = nullptr;
            if (cudaMalloc(&p, bytes) != cudaSuccess) {
                cudaGetLastError();
                return fail(B2_ENOMEM, "cudaMalloc(%zu) for weights failed", bytes);
            }
            e->d_payload = static_cast<uint8_t*>(p);
        }
        if (e->payload_bytes) B2_CUDA(cudaMemcpy(e->d_payload, payload, e->payload_bytes, cudaMemcpyHostToDevice));
    }
    *out = e.release();
    return B2_OK;
}

int b2_engine_deserialize(b2_runtime* rt, const void* blob, size_t nbytes, b2_engine** out) {
    return deserialize_impl(rt, blob, nbytes, false, out);
}

// metadata-only load (no device, no weights); contexts cannot be created from it
int b2_engine_inspect(const void* blob, size_t nbytes, b2_engine** out) {
    return deserialize_impl(nullptr, blob, nbytes, true, out);
}

void b2_engine_destroy(b2_engine* e) {
    if (!e) return;
    if (e->d_payload) {
        if (e->free_)
            e->free_(e->alloc_user, e->d_payload);
        else
            cudaFree(e->d_payload);
    }
    delete e;
}

int b2_engine_nb_bindings(const b2_engine* e) { return e ? int(e->bindings.size()) : 0; }
const char* b2_engine_binding_name(const b2_engine* e, int i) {
    return (e && i >= 0 && i < int(e->bindings.size())) ? e->bindings[i].name.c_str() : nullptr;
}
int b2_engine_binding_index(const b2_engine* e, const char* name) {
    if (!e || !name) return -1;
    for (size_t i = 0; i < e->bindings.size(); ++i)
        if (e->bindings[i].name == name) return int(i);
    return -1;
}
int b2_engine_binding_is_input(const b2_engine* e, int i) {
    return (e && i >= 0 && i < int(e->bindings.size())) ? int(e->bindings[i].is_input) : 0;
}
int b2_engine_binding_dtype(const b2_engine* e, int i) {
    return (e && i >= 0 && i < int(e->bindings.size())) ? e->bindings[i].dtype : -1;
}
int b2_engine_binding_dims(const b2_engine* e, int i, int32_t* dims, int* nd) {
    if (!e || i < 0 || i >= int(e->bindings.size()) || !dims || !nd) return fail(B2_EINVAL, "bad binding query");
    *nd = e->bindings[i].nd;
    for (int d = 0; d < 8; ++d) dims[d] = e->bindings[i].dims[d];
    return B2_OK;
}
int b2_engine_max_batch(const b2_engine* e) { return e ? e->max_batch : 0; }
int b2_engine_precision(const b2_engine* e) { return e ? e->precision : -1; }
const char* b2_engine_name(const b2_engine* e) { return e ? e->name.c_str() : nullptr; }
size_t b2_engine_device_memory_size(const b2_engine* e) { return e ? e->arena_bytes : 0; }
size_t b2_engine_weights_size(const b2_engine* e) { return e ? e->payload_bytes : 0; }
double b2_engine_flops(const b2_engine* e, int batch) { return e ? e->flops_per_item * batch : 0.0; }
int b2_engine_nb_layers(const b2_engine* e) { return e ? int(e->ops.size()) : 0; }

int b2_context_create(b2_engine* e, b2_context** out) {
    if (!e || !out) return fail(B2_EINVAL, "null engine or out");
    if (e->inspect_only) return fail(B2_ESTATE, "engine was loaded with b2_engine_inspect (no device resources)");
    b2_context* c = new b2_context();
    c->e = e;
    c->use_graph = env_int("B2_GRAPH", 1);
    c->force_simt = env_int("B2_FORCE_SIMT", 0);
    c->force_im2col = env_int("B2_FORCE_IM2COL", 0);
    c->force_bn = env_int("B2_FORCE_BN", 0);
    c->force_stages = env_int("B2_FORCE_STAGES", 0);
    c->force_splits = env_int("B2_FORCE_SPLITS", 0);
    c->force_sps = env_int("B2_FORCE_SPS", 0);
    c->force_ws = env_int("B2_FORCE_WS", 0);
    c->force_cn = env_int("B2_FORCE_CN", 0);
    c->force_halo = env_int("B2_FORCE_HALO", 0);
    c->pdl_trigger = env_int("B2_PDL_TRIGGER", 1);
    c->autotune = env_int("B2_AUTOTUNE", 4);
    c->fork = env_int("B2_FORK", 0);
    c->net = env_int("B2_NET", 0);
    c->net_ctas = env_int("B2_NET_CTAS", 0);
    c->net_bn = env_int("B2_NET_BN", 0);
    c->net_stages = env_int("B2_NET_STAGES", 0);
    c->fuse_tail = env_int("B2_FUSE_TAIL", 1);
    c->input_ctas = env_int("B2_INPUT_CTAS", 0);
    c->i8_bn = env_int("B2_I8_BN", 0);
    c->i8_stages = env_int("B2_I8_STAGES", 0);
    if (getenv("B2_PDL")) b2k::set_pdl(env_int("B2_PDL", 1) != 0);
    void* p = nullptr;
    if (cudaMalloc(&p, (kMaxSplitTiles + 16) * sizeof(int)) != cudaSuccess || cudaMemset(p, 0, (kMaxSplitTiles + 16) * sizeof(int)) != cudaSuccess) {
        cudaGetLastError();
        delete c;
        return fail(B2_ENOMEM, "cudaMalloc for split-K counters failed");
    }
    c->d_counters = static_cast<int*>(p);
    c->d_tail_ctrl = c->d_counters + kMaxSplitTiles;
    *out = c;
    return B2_OK;
}

static void drop_cached(b2_context* c) {
    c->states.clear();
    c->cur = c->scratch ? &c->states[c->scratch] : nullptr;
}

void b2_context_destroy(b2_context* c) {
    if (!c) return;
    drop_cached(c);
    if (c->d_counters) cudaFree(c->d_counters);
    if (c->side) cudaStreamDestroy(c->side);
    if (c->fork_ev) cudaEventDestroy(c->fork_ev);
    if (c->join_ev) cudaEventDestroy(c->join_ev);
    delete c;
}

int b2_context_set_device_memory(b2_context* c, void* scratch) {
    if (!c || !scratch) return fail(B2_EINVAL, "null context or scratch");
    if (reinterpret_cast<uintptr_t>(scratch) % 256 != 0) return fail(B2_EINVAL, "scratch must be 256-byte aligned (cudaMalloc alignment)");
    if (c->states.size() >= 32 && c->states.find(static_cast<uint8_t*>(scratch)) == c->states.end()) drop_cached(c);
    c->scratch = static_cast<uint8_t*>(scratch);
    c->cur = &c->states[c->scratch];
    return B2_OK;
}

int b2_context_set_option(b2_context* c, const char* key, int value) {
    if (!c || !key) return fail(B2_EINVAL, "null context or key");
    const std::string k(key);
    if (k == "graph") {
        c->use_graph = value;
        return B2_OK;
    }
    if (k == "pdl") {
        b2k::set_pdl(value != 0);  // process-wide
        value = 0;
    } else if (k == "simt") c->force_simt = value;
    else if (k == "im2col") c->force_im2col = value;
    else if (k == "bn") c->force_bn = value;
    else if (k == "stages") c->force_stages = value;
    else if (k == "splits") c->force_splits = value;
    else if (k == "sps") c->force_sps = value;
    else if (k == "ws") c->force_ws = value;
    else if (k == "cn") c->force_cn = value;
    else if (k == "halo") c->force_halo = value;
    else if (k == "fork") c->fork = value;
    else if (k == "net") c->net = value;
    else if (k == "net_ctas") c->net_ctas = value;
    else if (k == "net_bn") c->net_bn = value;
    else if (k == "net_stages") c->net_stages = value;
    else if (k == "fuse_tail") c->fuse_tail = value;
    else if (k == "i8_bn") c->i8_bn = value;
    else if (k == "i8_stages") c->i8_stages = value;
    else if (k == "input_ctas") c->input_ctas = value;
    else if (k == "pdl_trigger") c->pdl_trigger = value;
    else if (k == "autotune") c->autotune = value;
    else if (k == "no_fold") c->no_fold = value;
    else return fail(B2_EINVAL, "unknown option '%s'", key);
    drop_cached(c);
    return B2_OK;
}

int b2_context_nb_launches(b2_context* c, int batch) {
    if (!c) return -1;
    Plan* plan = nullptr;
    if (build_plan(c, batch, &plan)) return -1;
    return int(plan->launches.size());
}

// ---- ahead-of-time work: tactics and graphs never get built on the request path ------------------------------
int b2_engine_tune(b2_engine* e, int streams, int all_batches) {
    if (!e) return fail(B2_EINVAL, "null engine");
    if (e->inspect_only) return fail(B2_ESTATE, "engine was loaded with b2_engine_inspect (no device resources)");
    if (!e->half() || e->tactics_from_plan) return B2_OK;  // fp32 engines have no tactics; the plan brought its own
    std::lock_guard<std::mutex> run_lock(e->tune_run_mutex);
    b2_context* c = nullptr;
    int rc = b2_context_create(e, &c);
    if (rc) return rc;
    c->autotune = streams > 0 ? streams : c->autotune;
    void* scratch = nullptr;
    if (c->autotune <= 0) {
        b2_context_destroy(c);
        return B2_OK;
    }
    if (cudaMalloc(&scratch, std::max<size_t>(e->arena_bytes, 1024)) != cudaSuccess) {
        cudaGetLastError();
        b2_context_destroy(c);
        return fail(B2_ENOMEM, "cudaMalloc(%zu) for the tuning arena failed", e->arena_bytes);
    }
    rc = b2_context_set_device_memory(c, scratch);
    if (!rc && load_driver_entry_points() != 0) rc = fail(B2_ECUDA, "cuTensorMapEncode* driver entry points unavailable");
    {
        std::lock_guard<std::mutex> lock(e->tune_mutex);
        tune_cache_load(e);
    }
    if (!rc) rc = tune_engine_batch(c, e->max_batch);
    for (int b = 1; !rc && all_batches && b < e->max_batch; ++b) rc = tune_engine_batch(c, b);
    cudaDeviceSynchronize();
    b2_context_destroy(c);
    cudaFree(scratch);
    if (!rc) e->tuned_at_load = true;
    return rc;
}

// ---- network-level refinement of the tactic table ---------------------------------------------------------------
// The per-layer tuner times a layer against copies of ITSELF on N streams.  In service the N contexts are at DIFFERENT
// layers and each forward pass is a chain of dependent launches, so what a tactic costs the others (shared memory it
// holds while it waits) and what it gains (a shorter chain) only shows in the whole-network rate.  This pass walks the
// convolutions and keeps a tactic change when it raises the measured throughput of `streams` contexts running whole
// forward passes concurrently.  Every tactic computes the same bits, so this is purely a performance choice.
namespace {
struct RefineCtx {
    b2_context* c = nullptr;
    void* scratch = nullptr;
    std::vector<void*> bind;
    cudaStream_t s = nullptr;
};
}  // namespace

int b2_engine_refine_tactics(b2_engine* e, int streams, int passes, double* gain_out) {
    if (gain_out) *gain_out = 1.0;
    if (!e) return fail(B2_EINVAL, "null engine");
    if (e->inspect_only) return fail(B2_ESTATE, "engine was loaded with b2_engine_inspect (no device resources)");
    if (!e->half() || e->tactics_from_plan) return B2_OK;
    streams = std::max(1, std::min(streams > 0 ? streams : 4, 8));
    int rc = b2_engine_tune(e, streams, 0);  // start from the per-layer table
    if (rc) return rc;
    std::lock_guard<std::mutex> run_lock(e->tune_run_mutex);
    const int batch = e->max_batch;
    std::vector<RefineCtx> ctx(static_cast<size_t>(streams));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    auto cleanup = [&] {
        cudaDeviceSynchronize();
        for (auto& x : ctx) {
            if (x.c) b2_context_destroy(x.c);
            if (x.scratch) cudaFree(x.scratch);
            for (void* p : x.bind)
                if (p) cudaFree(p);
            if (x.s) cudaStreamDestroy(x.s);
        }
        if (e0) cudaEventDestroy(e0);
        if (e1) cudaEventDestroy(e1);
    };
    bool ok = cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess;
    for (auto& x : ctx) {
        if (!ok) break;
        ok = b2_context_create(e, &x.c) == B2_OK && cudaMalloc(&x.scratch, std::max<size_t>(e->arena_bytes, 1024)) == cudaSuccess &&
             b2_context_set_device_memory(x.c, x.scratch) == B2_OK && cudaStreamCreateWithFlags(&x.s, cudaStreamNonBlocking) == cudaSuccess;
        x.bind.assign(e->bindings.size(), nullptr);
        for (size_t i = 0; i < e->bindings.size() && ok; ++i) {
            const size_t bytes = e->bindings[i].item_bytes * size_t(e->max_batch);
            ok = cudaMalloc(&x.bind[i], bytes) == cudaSuccess && cudaMemset(x.bind[i], 0, bytes) == cudaSuccess;
        }
    }
    if (!ok) {
        cudaGetLastError();
        cleanup();
        return fail(B2_ENOMEM, "refine: cannot set up %d contexts", streams);
    }
    const int iters = std::max(8, env_int("B2_REFINE_ITERS", 24));  // forward passes per context and measurement
    int status = B2_OK;
    auto measure = [&]() -> double {  // ms per forward pass of the whole job (all contexts), best of 2
        for (auto& x : ctx) {
            drop_cached(x.c);
            if ((status = b2_context_prepare(x.c, batch, x.s))) return 1e30;
        }
        double best = 1e30;
        for (int rep = 0; rep < 3 && !status; ++rep) {  // rep 0 = warm-up
            for (auto& x : ctx) cudaStreamSynchronize(x.s);
            cudaEventRecord(e0, ctx[0].s);
            for (size_t k = 1; k < ctx.size(); ++k) cudaStreamWaitEvent(ctx[k].s, e0, 0);
            const int n = rep == 0 ? 4 : iters;
            for (int i = 0; i < n && !status; ++i)
                for (auto& x : ctx)
                    if ((status = b2_context_enqueue(x.c, batch, x.bind.data(), x.s, nullptr))) break;
            for (size_t k = 1; k < ctx.size(); ++k) {
                cudaEvent_t d = nullptr;
                cudaEventCreateWithFlags(&d, cudaEventDisableTiming);
                cudaEventRecord(d, ctx[k].s);
                cudaStreamWaitEvent(ctx[0].s, d, 0);
                cudaEventDestroy(d);
            }
            cudaEventRecord(e1, ctx[0].s);
            if (cudaStreamSynchronize(ctx[0].s) != cudaSuccess) {
                status = fail(B2_ECUDA, "refine: forward pass failed: %s", cudaGetErrorString(cudaGetLastError()));
                break;
            }
            float ms = 0.f;
            cudaEventElapsedTime(&ms, e0, e1);
            if (rep > 0) best = std::min(best, double(ms) / (double(n) * double(ctx.size())));
        }
        return best;
    };
    double base = measure();
    const double first = base;
    const double keep = 1.0 - std::max(0.0, double(env_int("B2_REFINE_MIN_GAIN_PERMILLE", 7))) / 1000.0;  // accept only clear wins
    for (int pass = 0; pass < std::max(1, passes) && !status; ++pass) {
        int changed = 0;
        for (size_t i = 0; i < e->ops.size() && !status; ++i) {
            const Op& op = e->ops[i];
            const b2plan::OpRec& r = op.r;
            if (r.type != b2plan::OP_CONV || (r.relu & 4)) continue;
            ConvConfig cur;
            {
                std::lock_guard<std::mutex> lock(e->tune_mutex);
                auto it = e->tuned.find({int(i), batch});
                if (it == e->tuned.end()) continue;
                cur = it->second;
            }
            const int kbsz = conv_kb(ctx[0].c, op);
            if (kbsz != 64 || cur.ws || cur.cn > 1) continue;
            const int nkb = conv_num_kblocks(ctx[0].c, op);
            std::vector<ConvConfig> cands;
            // split-K: a deep-K layer with few tiles (res4 / res5 3x3) is a LONG link of the dependency chain on a handful
            // of SMs; splitting K shortens the link and puts more SMs on it.  The per-layer tuner rejects it (more total
            // work), the chain-bound whole-network rate is where it can pay.  (The split factor fixes the fp32 summation
            // order; it is chosen here, at max batch, and shared by every batch size.)
            if (env_int("B2_TUNE_SPLITK", 0) != 0 && !(op.side_join >= 0) && cur.splits == 1 && !cur.halo) {  // opt-in: changes bits
                const int m_tiles = (batch * int(e->tensors[r.out].h * e->tensors[r.out].w) + 127) / 128;
                for (int sp : {2, 4}) {
                    const int tiles = m_tiles * (int(r.cout_phys) / cur.bn);
                    const int kpc = (nkb + sp - 1) / sp;
                    if (nkb < 16 || tiles >= 100 || tiles * sp > 160 || kpc < 4 || (sp - 1) * kpc >= nkb || tiles > kMaxSplitTiles / 8 ||
                        size_t(tiles) * sp * 128 * cur.bn * 4 > kSplitWorkspaceBytes)
                        continue;
                    for (int st : {2, 4}) {
                        if (!b2k::conv_config_exists(cur.bn, kbsz, st, 1) || b2k::conv_smem_bytes(cur.bn, st, r.res >= 0, 1) > 227 * 1024) continue;
                        cands.push_back(ConvConfig{cur.bn, st, sp, 0.0, 1, 0, 1});
                    }
                }
            }
            if (cur.splits > 1) continue;  // already split: leave it
            for (int bn : {64, 128, 256}) {
                if (int(r.cout_phys) % bn) continue;
                for (int sps = 1; sps <= 2; ++sps)
                    for (int st : {1, 2, 4, 8}) {
                        if (!b2k::conv_config_exists(bn, kbsz, st, sps) || b2k::conv_smem_bytes(bn, st, r.res >= 0, sps) > 227 * 1024) continue;
                        if (st * sps > nkb + 1 && st > 1) continue;  // a ring deeper than the K loop only costs shared memory
                        if (sps == 2 && nkb < 4) continue;
                        if (bn == cur.bn && st == cur.stages && sps == cur.sps && !cur.halo) continue;
                        cands.push_back(ConvConfig{bn, st, 1, 0.0, sps, 0, 1});
                    }
                if (conv_halo_rows(ctx[0].c, op) && b2k::conv_halo_config_exists(bn) && int(r.cin_phys) / 64 <= 8 && !(cur.halo && cur.bn == bn) &&
                    b2k::conv_halo_smem(bn, int(e->tensors[r.out].w), conv_halo_rows(ctx[0].c, op), int(r.cin_phys) / 64) <= 227 * 1024) {
                    ConvConfig hc{bn, kHaloStagesTag, 1, 0.0, 1, 0, 1};
                    hc.halo = 1;
                    cands.push_back(hc);
                }
            }
            ConvConfig best = cur;
            for (const ConvConfig& cand : cands) {
                {
                    std::lock_guard<std::mutex> lock(e->tune_mutex);
                    e->tuned[{int(i), batch}] = cand;
                }
                const double t = measure();
                if (status) break;
                if (t < base * keep) base = t, best = cand, ++changed;
            }
            std::lock_guard<std::mutex> lock(e->tune_mutex);
            e->tuned[{int(i), batch}] = best;
        }
        if (!changed) break;
    }
    if (!status) {
        const double last = measure();  // (re-measured with the final table)
        if (gain_out && last > 0 && last < 1e29) *gain_out = first / last;
    }
    cleanup();
    return status;
}

int b2_engine_nb_tactics(const b2_engine* e) {
    if (!e) return 0;
    std::lock_guard<std::mutex> lock(const_cast<b2_engine*>(e)->tune_mutex);
    return int(e->tuned.size());
}
// 10 x uint32 per tactic, the TacticRec layout of plan_format.h; returns the number written
int b2_engine_get_tactics(const b2_engine* e, uint32_t* out, int cap) {
    if (!e || !out) return 0;
    std::lock_guard<std::mutex> lock(const_cast<b2_engine*>(e)->tune_mutex);
    int n = 0;
    for (const auto& kv : e->tuned) {
        if (n >= cap) break;
        const ConvConfig& g = kv.second;
        const uint32_t rec[10] = {uint32_t(kv.first.first), uint32_t(kv.first.second), uint32_t(g.bn), uint32_t(g.stages), uint32_t(g.splits),
                                  uint32_t(g.sps), uint32_t(g.ws), uint32_t(g.cn), uint32_t(g.halo), 0u};
        memcpy(out + size_t(n) * 10, rec, sizeof rec);
        ++n;
    }
    return n;
}

// Builds the launch plan of `batch` for the context's current arena and instantiates its graph segments, so that the
// first request at this batch size pays neither.  `stream` is only used to record the capture.
int b2_context_prepare(b2_context* c, int batch, b2_stream_t stream_) {
    if (!c) return fail(B2_EINVAL, "null context");
    if (batch < 1 || batch > c->e->max_batch) return fail(B2_EINVAL, "batch %d outside [1, %d]", batch, c->e->max_batch);
    Plan* plan = nullptr;
    int rc = build_plan(c, batch, &plan);
    if (rc) return rc;
    if (!c->use_graph || plan->has_net) return B2_OK;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    cudaStream_t own = nullptr;
    if (!stream) {
        B2_CUDA(cudaStreamCreateWithFlags(&own, cudaStreamNonBlocking));
        stream = own;
    }
    // placeholder binding pointers: a capture only RECORDS launches, and every request re-points the nodes that use them
    std::vector<void*> dummy(c->e->bindings.size(), reinterpret_cast<void*>(uintptr_t(256)));
    if (c->use_graph != 3 && !plan->exec && !plan->graph_failed) {
        rc = instantiate_plan_graph(c, plan, dummy.data(), stream);
        plan->graph_failed = !rc && plan->exec == nullptr;
    }
    if (!rc && !plan->exec)
        for (Segment& sg : plan->segments)
            if (sg.graphable && !sg.exec && (rc = instantiate_segment(c, plan, &sg, dummy.data(), stream))) break;
    if (own) cudaStreamDestroy(own);
    return rc;
}

int b2_context_enqueue(b2_context* c, int batch, void* const* bindings, b2_stream_t stream_, b2_event_t consumed) {
    int rc = check_args(c, batch, bindings);
    if (rc) return rc;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    Plan* plan = nullptr;
    if ((rc = build_plan(c, batch, &plan))) return rc;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    B2_CUDA(cudaStreamIsCapturing(stream, &cap));
    // Inside a caller's capture (the reference graphs enqueueV2 itself, workspace.cc:51-56), with graphs off, or for a plan
    // that is a handful of launches anyway (persistent network kernel): plain launches.
    if (cap != cudaStreamCaptureStatusNone || !c->use_graph || plan->has_net) {
        if ((rc = run_all(c, *plan, bindings, stream))) return rc;
    } else {
        if (c->use_graph != 3 && !plan->exec && !plan->graph_failed) {
            if ((rc = instantiate_plan_graph(c, plan, bindings, stream))) return rc;
            plan->graph_failed = plan->exec == nullptr;
        }
        if (plan->exec) {  // one graph for the whole forward pass, re-pointed at this request's bindings
            if ((rc = patch_plan_graph(plan, bindings))) return rc;
            B2_CUDA(cudaGraphLaunch(plan->exec, stream));
        } else {
            for (Segment& sg : plan->segments) {
                if (!sg.graphable) {
                    if ((rc = run_range(c, *plan, size_t(sg.begin), size_t(sg.end), bindings, stream))) return rc;
                    continue;
                }
                if (!sg.exec && (rc = instantiate_segment(c, plan, &sg, bindings, stream))) return rc;
                B2_CUDA(cudaGraphLaunch(sg.exec, stream));
            }
        }
    }
    if (consumed) B2_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(consumed), stream));
    return B2_OK;
}

int b2_context_profile(b2_context* c, int batch, void* const* bindings, b2_stream_t stream_, float* ms, int cap) {
    if (check_args(c, batch, bindings)) return -1;
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    Plan* plan = nullptr;
    if (build_plan(c, batch, &plan)) return -1;
    const int n = int(plan->launches.size());
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) cudaEventCreate(&e);
    int rc = 0;
    cudaEventRecord(ev[0], stream);
    for (int i = 0; i < n && !rc; ++i) {
        rc = run_launch(c->e, plan->launches[i], bindings, stream);
        cudaEventRecord(ev[i + 1], stream);
    }
    cudaError_t se = cudaStreamSynchronize(stream);
    if (rc || se != cudaSuccess) {
        fail(B2_ECUDA, "profile run failed: %s", cudaGetErrorString(rc ? cudaError_t(rc) : se));
        n > 0 ? (void)0 : (void)0;
    } else {
        for (int i = 0; i < n && i < cap; ++i) cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return (rc || se != cudaSuccess) ? -1 : n;
}

static const Launch* get_launch(b2_context* c, int batch, int i) {
    if (!c) return nullptr;
    Plan* plan = nullptr;
    if (build_plan(c, batch, &plan)) return nullptr;
    if (i < 0 || i >= int(plan->launches.size())) return nullptr;
    return &plan->launches[i];
}
// Debug aid (not part of the drop-in surface): run launch `i` of the plan `reps` times back to back on `stream`
// with per-CTA phase timestamps enabled; `stamps` receives 16 int64 per CTA of the LAST repetition.
int b2_context_debug_conv_timing(b2_context* c, int batch, int i, int reps, b2_stream_t stream_, long long* stamps,
                                 int cap_ctas, int* n_ctas) {
    const int dbg_mode = env_int("B2_DBG_MODE", 0);
    Plan* plan = nullptr;
    if (!c || build_plan(c, batch, &plan)) return fail(B2_EINVAL, "no plan");
    if (i < 0 || i >= int(plan->launches.size()) || plan->launches[i].kind != L_CONV_TC) return fail(B2_EINVAL, "not a tcgen05 conv launch");
    b2k::ConvLaunch cl = plan->launches[i].conv;
    const int ctas = cl.ws_ctas > 0 ? cl.ws_ctas : cl.grid_m * cl.grid_n * cl.args.splits;
    if (n_ctas) *n_ctas = ctas;
    if (ctas > cap_ctas) return fail(B2_EINVAL, "stamp buffer too small (%d CTAs)", ctas);
    long long* d = nullptr;
    B2_CUDA(cudaMalloc(&d, size_t(ctas) * 16 * sizeof(long long)));
    cudaMemset(d, 0, size_t(ctas) * 16 * sizeof(long long));
    cl.args.dbg = d;
    cl.args.dbg_mode = dbg_mode;
    cudaStream_t s = static_cast<cudaStream_t>(stream_);
    int rc = 0;
    for (int r = 0; r < reps && !rc; ++r) rc = b2k::launch_conv_f16_tcgen05(cl, s);
    cudaError_t se = cudaStreamSynchronize(s);
    if (!rc && se == cudaSuccess) cudaMemcpy(stamps, d, size_t(ctas) * 16 * sizeof(long long), cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (rc || se != cudaSuccess) return fail(B2_ECUDA, "debug launch failed: %s", cudaGetErrorString(rc ? cudaError_t(rc) : se));
    return B2_OK;
}

// Debug aid (not part of the drop-in surface): one forward pass with the instrumented instantiation of the persistent
// network kernel; `out` receives 8 roles x 8 int64 counters per CTA (see net_kernel.cu), `n_ctas` the CTA count.
int b2_context_debug_net_timing(b2_context* c, int batch, void* const* bindings, b2_stream_t stream_, long long* out, int cap_ctas,
                                int* n_ctas) {
    Plan* plan = nullptr;
    if (!c || build_plan(c, batch, &plan)) return fail(B2_EINVAL, "no plan");
    NetRun* run = nullptr;
    for (Launch& L : plan->launches)
        if (L.kind == L_NET) run = L.net.get();
    if (!run) return fail(B2_EINVAL, "the plan has no persistent network kernel");
    if (n_ctas) *n_ctas = run->ctas;
    if (run->ctas > cap_ctas) return fail(B2_EINVAL, "counter buffer too small (%d CTAs)", run->ctas);
    long long* d = nullptr;
    const size_t bytes = size_t(run->ctas) * 64 * sizeof(long long);
    B2_CUDA(cudaMalloc(&d, bytes));
    cudaMemset(d, 0, bytes);
    cudaStream_t s = static_cast<cudaStream_t>(stream_);
    run->args.dbg = d;
    int rc = run_all(c, *plan, bindings, s);
    cudaError_t se = cudaStreamSynchronize(s);
    run->args.dbg = nullptr;
    if (!rc && se == cudaSuccess) cudaMemcpy(out, d, bytes, cudaMemcpyDeviceToHost);
    cudaFree(d);
    if (rc) return rc;
    if (se != cudaSuccess) return fail(B2_ECUDA, "debug launch failed: %s", cudaGetErrorString(se));
    return B2_OK;
}

const char* b2_context_launch_name(b2_context* c, int batch, int i) {
    static thread_local std::string s;
    const Launch* L = get_launch(c, batch, i);
    if (!L) return nullptr;
    static const char* kinds[] = {"input_cast", "conv_tcgen05", "conv_simt", "maxpool", "avgpool", "fc", "softmax", "output_cast", "net_tcgen05", "tail_pool_fc_softmax",
                                  "quantize", "conv_i8_tcgen05", "avgpool_i8", "output_cast_i8"};
    s = std::string(kinds[L->kind]) + ":" + L->name;
    if (L->kind == L_CONV_TC)
        s += " bn=" + std::to_string(L->conv.bn) + " kb=" + std::to_string(L->conv.kb) +
             " st=" + std::to_string(L->conv.stages) + "x" + std::to_string(L->conv.sps) +
             (L->conv.ws_ctas ? " ws=" + std::to_string(L->conv.ws_ctas) : std::string()) +
             (L->conv.cn > 1 ? " cn=" + std::to_string(L->conv.cn) : std::string()) + (L->conv.halo ? " halo" : "") +
             (L->conv.args.a_mode == b2k::A_TILED ? " tiled" : " im2col") +
             " grid=" + std::to_string(L->conv.grid_n) + "x" + std::to_string(L->conv.grid_m) + "x" +
             std::to_string(L->conv.args.splits) + " kblk=" + std::to_string(L->conv.args.num_kblocks);
    if (L->kind == L_CONV_I8)
        s += " bn=" + std::to_string(L->i8.bn) + " st=" + std::to_string(L->i8.stages) + (L->i8.args.a_mode == b2k::A_TILED ? " tiled" : " im2col") + " grid=" +
             std::to_string(L->i8.grid_n) + "x" + std::to_string(L->i8.grid_m) + " kblk=" + std::to_string(L->i8.args.num_kblocks);
    if (L->kind == L_NET)
        s += " layers=" + std::to_string(L->net->args.n_layers) + " tiles=" + std::to_string(L->net->args.total_tiles) +
             " ctas=" + std::to_string(L->net->ctas) + " stages=" + std::to_string(L->net->args.stages);
    if (L->side_join >= 0) s += " side";
    return s.c_str();
}
double b2_context_launch_flops(b2_context* c, int batch, int i) {
    const Launch* L = get_launch(c, batch, i);
    return L ? L->flops : 0.0;
}
double b2_context_launch_bytes(b2_context* c, int batch, int i) {
    const Launch* L = get_launch(c, batch, i);
    return L ? L->bytes : 0.0;
}

}  // extern "C"
