/*
 * trtlab_host.h -- extern "C" handles onto the C++ host layer (trtlab::TensorRT::InferenceManager,
 * InferRunner, InferBench, TimedBenchmarkWorkspace) so that Python (ctypes) tests and bench.py drive the
 * SAME pipeline a C++ trtlab application uses.  Not needed by C++ callers, who include
 * the trtlab/tensorrt headers directly.  Return codes / b2_last_error() as in b200infer.h.
 */
#ifndef TRTLAB_HOST_H_
#define TRTLAB_HOST_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct trt_manager trt_manager;

/* InferenceManager(max_exec, max_buffers /0 -> 2x/) + "pre"/"cuda"/"post" pools + StandardRuntime;
 * mirrors the setup in reference examples/00_TensorRT/infer.cc:88-114 */
int trt_manager_create(int max_exec, int max_buffers, int pre_threads, int cuda_threads, int post_threads,
                       trt_manager** out);
void trt_manager_destroy(trt_manager* m);
/* Runtime::DeserializeEngine + InferenceManager::RegisterModel (max_concurrency <= 0: manager default) */
int trt_manager_register_model(trt_manager* m, const char* name, const void* blob, size_t nbytes, int max_concurrency);
int trt_manager_allocate(trt_manager* m); /* InferenceManager::AllocateResources */
/* one request through InferRunner::Infer(pre, post): pinned H2D -> forward -> D2H, blocking */
int trt_manager_infer(trt_manager* m, const char* model, int batch, const void* input, size_t input_bytes,
                      float* output, size_t output_bytes, double* compute_seconds);
/* `n` single-image requests through BatchedInferRunner (Dispatcher<StandardBatcher>, window_us): inputs/outputs are
 * contiguous [n][item]; *batches_executed = number of merged forward passes it took */
int trt_manager_infer_batched(trt_manager* m, const char* model, int n, const void* inputs, void* outputs, int window_us,
                              int* batches_executed);
/* the same path as one flood of `n` single-image requests cycling through `ring` (ring_items images); *window_seconds spans
 * the completions of requests [warm, n - cool) -- steady state, free of the pipeline's fill and drain; outputs: n items */
int trt_manager_bench_batched(trt_manager* m, const char* model, int n, const void* ring, int ring_items, void* outputs,
                              int window_us, int warm, int cool, double* window_seconds, double* total_seconds,
                              int* batches_executed);
/* Prometheus text exposition of the manager's metrics (request/compute summaries per model, load-ratio histogram,
 * GPU power gauge sampled now through NVML); returns the text length (excluding the NUL) or a negative B2_E* code;
 * at most cap-1 bytes are written */
int trt_manager_metrics_text(trt_manager* m, char* buf, size_t cap);
/* serve that text over HTTP (GET /metrics) from a background thread, the role of prometheus::Exposer in the reference
 * service (metrics.cc:34-60); port 0 = kernel-chosen, reported through *bound_port; stops with the manager */
int trt_manager_serve_metrics(trt_manager* m, int port, int* bound_port);
/* write a distinct batch from `ring` into the pinned input region of every pooled Buffers */
int trt_manager_prefill_inputs(trt_manager* m, const char* model, const void* ring, size_t ring_batches);
/* InferBench::Run closed loop; results16[InferBenchKey]; optional per-request latencies (seconds) */
int trt_manager_bench(trt_manager* m, const char* model, int batch, double seconds, size_t max_batches,
                      double* results16, double* latencies, size_t lat_cap, size_t* lat_count);
/* one continuous closed loop of warm + steps + cool requests; *window_seconds spans the `steps` completions in the middle
 * (pipeline full on both sides), latencies[] = those requests' latencies */
int trt_manager_bench_window(trt_manager* m, const char* model, int batch, size_t warm, size_t steps, size_t cool,
                             double* window_seconds, double* latencies, size_t lat_cap, size_t* lat_count);
/* ... `windows` back-to-back windows of `steps` completions each inside the same loop (window_seconds[windows]): a single
 * scheduling hiccup then costs one window, not the measurement; latencies[] covers all windows */
int trt_manager_bench_windows(trt_manager* m, const char* model, int batch, size_t warm, size_t steps, size_t windows, size_t cool,
                              double* window_seconds, double* latencies, size_t lat_cap, size_t* lat_count);
/* TimedBenchmarkWorkspace::enqueue_pipeline averaged over iters */
int trt_timed_pipeline(const void* blob, size_t nbytes, int iters, float* h2d_ms, float* compute_ms, float* d2h_ms);
/* v2 surface: BenchmarkWorkspace (caller-captured graph of the forward pass, reference workspace.cc:21-124) at max batch:
 * pinned input -> async_h2d -> enqueue() -> async_d2h, `iters` times; returns the output of the last pass.
 * managed_runtime != 0: weights through ManagedRuntime (cudaMallocManaged + ReadMostly, allocator.cc:72-77) */
int trt_workspace_infer(const void* blob, size_t nbytes, const void* input, size_t input_bytes, void* output,
                        size_t output_bytes, int managed_runtime, int iters);
/* the v1 hot path by hand over CyclicBuffers<CudaPinnedHostMemory, CudaDeviceMemory> (buffers.h:122-154): `rounds`
 * requests cut from a 3-segment ring (which therefore wraps); output and device time of the last request */
int trt_cyclic_infer(const void* blob, size_t nbytes, int batch, const void* input, size_t input_bytes, void* output,
                     size_t output_bytes, int managed_runtime, int rounds, double* compute_seconds);
/* device-resident throughput of `contexts` concurrent execution contexts (inputs cycled through a device ring).
 * Timed step i runs on context i % contexts with input ring[i % ring_batches].  last_outputs (may be NULL): after the
 * timed region, the `batch` rows of every output binding computed by the last timed step, back to back in binding
 * order; last_outputs_bytes must equal their total size */
int trt_device_throughput(const void* blob, size_t nbytes, int contexts, int batch, int steps, int warmup,
                          const void* host_ring, int ring_batches, double* elapsed_ms, int* launches_per_step,
                          void* last_outputs, size_t last_outputs_bytes);

#ifdef __cplusplus
}
#endif
#endif /* TRTLAB_HOST_H_ */
