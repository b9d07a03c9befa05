/*
 * b200infer.h -- C ABI of the B200-native inference engine that replaces TensorRT underneath
 * trtlab/tensorrt (NVIDIA/tensorrt-laboratory).  Plain C, plain pointers and sizes; no C++/torch types.
 *
 * Every entry point mirrors 1:1 one nvinfer1:: call the reference makes on its per-request hot path.
 * The "replaces" notes cite the reference call site (file:line under /root/reference).
 *
 * Conventions: functions returning int return 0 on success, non-zero B2_E* on failure and set a
 * thread-local message readable with b2_last_error().  An engine is immutable and may be shared by
 * any number of contexts/threads; a context is single-flight (one enqueue in flight at a time), the
 * same contract as nvinfer1::IExecutionContext.  All work is asynchronous on the caller's stream.
 *
 * There is NO CPU fallback: b2_engine_deserialize fails with B2_ENODEVICE if the current device is not
 * an sm_100 part or no CUDA device is present.
 */
#ifndef B200INFER_H_
#define B200INFER_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_ABI_VERSION 1

enum {
    B2_OK = 0,
    B2_EINVAL = 1,    /* bad argument / malformed blob            */
    B2_ENODEVICE = 2, /* no CUDA device, or not sm_100            */
    B2_ECUDA = 3,     /* a CUDA runtime / driver call failed      */
    B2_ENOMEM = 4,    /* allocation failed                        */
    B2_ESTATE = 5     /* call sequence error (e.g. no device memory set) */
};

/* binding data types; same order as the reference's dtype switch (trtlab/tensorrt/src/utils.cc:40-46).
 * B2_DT_UINT8 (= nvinfer1::DataType::kUINT8; 4 = kBOOL stays unused): image input bindings of fp16 / INT8 engines, per item
 * {src_h, src_w, C} HWC bytes; the input cast crops, reorders channels and normalises them (builder.preprocess_u8). */
enum { B2_DT_FLOAT = 0, B2_DT_HALF = 1, B2_DT_INT8 = 2, B2_DT_INT32 = 3, B2_DT_UINT8 = 5 };

/* engine arithmetic ("precision" of the plan, cf. trtexec --fp16) */
enum { B2_PREC_FP32 = 0, B2_PREC_FP16 = 1, B2_PREC_INT8 = 2 /* INT8 bottleneck convolutions, fp16 stem / classifier */ };

typedef struct b2_runtime b2_runtime;
typedef struct b2_engine b2_engine;
typedef struct b2_context b2_context;

/* CUDA handles cross the ABI as opaque pointers (cudaStream_t / cudaEvent_t are pointers). */
typedef void* b2_stream_t;
typedef void* b2_event_t;

/* device allocator callbacks; mirrors nvinfer1::IGpuAllocator::allocate/free
 * (reference trtlab/tensorrt/src/allocator.cc:38-58) */
typedef void* (*b2_alloc_fn)(void* user, uint64_t size, uint64_t alignment, uint32_t flags);
typedef void (*b2_free_fn)(void* user, void* ptr);

int b2_abi_version(void);
const char* b2_last_error(void); /* thread-local, never NULL */

/* replaces nvinfer1::createInferRuntime (trtlab/tensorrt/src/runtime.cc:47) */
int b2_runtime_create(b2_runtime** out);
void b2_runtime_destroy(b2_runtime* rt);
/* replaces IRuntime::setGpuAllocator (runtime.cc:126); NULL fns restore cudaMalloc/cudaFree */
int b2_runtime_set_allocator(b2_runtime* rt, b2_alloc_fn alloc, b2_free_fn free_, void* user);

/* replaces IRuntime::deserializeCudaEngine (runtime.cc:139).  `blob` is a B2ENGINE plan
 * (tensorrt_laboratory_b200/builder.py).  Weights are uploaded to the CURRENT device. */
int b2_engine_deserialize(b2_runtime* rt, const void* blob, size_t nbytes, b2_engine** out);
/* metadata-only load: parses the plan without touching a device (no weights uploaded).  Binding and
 * size queries work; b2_context_create on such an engine fails with B2_ESTATE.  For tooling/tests. */
int b2_engine_inspect(const void* blob, size_t nbytes, b2_engine** out);
void b2_engine_destroy(b2_engine* e);

/* replace ICudaEngine::getNbBindings / getBindingName / bindingIsInput / getBindingDataType /
 * getBindingDimensions / getMaxBatchSize (trtlab/tensorrt/src/model.cc:76-116,
 * execution_context.cc:24-25).  Dims are PER BATCH ITEM (implicit batch), e.g. {3,224,224}. */
int b2_engine_nb_bindings(const b2_engine* e);
const char* b2_engine_binding_name(const b2_engine* e, int i);
int b2_engine_binding_index(const b2_engine* e, const char* name); /* -1 if absent */
int b2_engine_binding_is_input(const b2_engine* e, int i);
int b2_engine_binding_dtype(const b2_engine* e, int i);
int b2_engine_binding_dims(const b2_engine* e, int i, int32_t* dims, int* nd); /* dims[8] */
int b2_engine_max_batch(const b2_engine* e);
int b2_engine_precision(const b2_engine* e);
const char* b2_engine_name(const b2_engine* e);
/* replaces ICudaEngine::getDeviceMemorySize (workspace.cc:40): activation arena at max batch */
size_t b2_engine_device_memory_size(const b2_engine* e);
/* bytes of weights resident on the device (reference Model::GetWeightsMemorySize) */
size_t b2_engine_weights_size(const b2_engine* e);
/* algorithmic work of one forward pass at `batch` (2*MAC of conv+fc); for roofline reporting */
double b2_engine_flops(const b2_engine* e, int batch);
int b2_engine_nb_layers(const b2_engine* e);

/* replaces ICudaEngine::createExecutionContextWithoutDeviceMemory (execution_context.cc:10) */
int b2_context_create(b2_engine* e, b2_context** out);
void b2_context_destroy(b2_context* c);
/* replaces IExecutionContext::setDeviceMemory (workspace.cc:41); `scratch` must hold
 * b2_engine_device_memory_size() bytes, 256-byte aligned, and outlive every enqueue */
int b2_context_set_device_memory(b2_context* c, void* scratch);
/* replaces IExecutionContext::enqueue / enqueueV2 (workspace.cc:47,52).  `bindings[i]` are DEVICE
 * pointers in binding order.  Asynchronous on `stream`; legal inside cudaStreamBeginCapture
 * (the reference captures it into a graph, workspace.cc:51-56).  If `input_consumed` is non-NULL the
 * event is recorded on `stream` once the input bindings may be overwritten. */
int b2_context_enqueue(b2_context* c, int batch, void* const* bindings, b2_stream_t stream,
                       b2_event_t input_consumed);
/* number of kernels one enqueue at `batch` launches (for reporting) */
int b2_context_nb_launches(b2_context* c, int batch);

/* ---- ahead-of-time work (the role of TensorRT's builder / trtexec, reference models/setup.py:53-55): tactic selection
 * and graph instantiation happen at model-registration time, never inside b2_context_enqueue. ---- */
/* Times the kernel tactics of every convolution on THIS device, on a private arena, at max batch (and at every batch
 * size 1..max when `all_batches` != 0) with `streams` concurrent streams (0 = default 4); results are kept on the engine.
 * No-op for fp32 engines and for plans that carry a tactic table.  Untuned engines run on a closed-form cost model. */
int b2_engine_tune(b2_engine* e, int streams, int all_batches);
/* Network-level refinement of the tactic table (build-time work, tens of seconds): starting from b2_engine_tune's
 * per-layer choices, keep a tactic change when it raises the throughput of `streams` contexts running whole forward passes
 * concurrently (the serving regime), up to `passes` sweeps over the convolutions.  *gain (optional) = rate after / before.
 * Export the result with b2_engine_get_tactics and ship it in the plan (builder.attach_tactics). */
int b2_engine_refine_tactics(b2_engine* e, int streams, int passes, double* gain);
int b2_engine_nb_tactics(const b2_engine* e);
/* exports the tactic table, 10 x uint32 per record {op, batch, bn, stages, splits, sps, ws, cn, halo, 0} (the TacticRec
 * layout of the plan format); builder.attach_tactics() appends it to a plan blob.  Returns the records written. */
int b2_engine_get_tactics(const b2_engine* e, uint32_t* out, int cap_records);
/* Builds the launch plan of `batch` for the context's current device memory and instantiates its CUDA-graph segments
 * (one graph per context and batch, independent of the binding pointers).  `stream` may be NULL. */
int b2_context_prepare(b2_context* c, int batch, b2_stream_t stream);
/* knobs: "graph"=0/1 replay the forward as a cached CUDA graph (default 1); "simt"=0/1 force the
 * SIMT reference kernels instead of the tcgen05 path (debug); "bn"/"stages"/"splits" force the conv tile,
 * pipeline depth and split-K factor (0 = cost model); "pdl"=0/1 programmatic dependent launch (process-wide);
 * "pdl_trigger"=0/1 release point of the dependent kernel; "autotune"=0 (cost model) / 1 (latency) / N>=2 (N-stream
 * throughput, default 4) on-device tactic selection; "sps"=2 double-width pipeline stages; tactic switches
 * "halo"=1/-1 (3x3 halo kernel everywhere it applies / never; 0 = tuner decides), "ws"=1/N/-1 (persistent
 * warp-specialised kernel), "cn"=2/4/-1 (cluster multicast of the activation tile), "fork"=0/1 (shortcut convolutions
 * on a parallel graph branch); returns B2_EINVAL for unknown keys.  Every tactic computes bit-identical results.
 * Environment: B2_TUNE_CACHE=<file> persists tuned tactics across processes (timing cache). */
int b2_context_set_option(b2_context* c, const char* key, int value);

/* per-layer device timing of one forward (serialised launches, CUDA events): fills up to `cap`
 * entries of ms[] in launch order and returns the number of launches, or <0 on error */
int b2_context_profile(b2_context* c, int batch, void* const* bindings, b2_stream_t stream,
                       float* ms, int cap);
const char* b2_context_launch_name(b2_context* c, int batch, int i);
double b2_context_launch_flops(b2_context* c, int batch, int i);
double b2_context_launch_bytes(b2_context* c, int batch, int i);

#ifdef __cplusplus
}
#endif
#endif /* B200INFER_H_ */
