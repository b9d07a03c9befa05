// extern "C" access to the C++ host layer (InferenceManager / InferRunner / InferBench / workspaces) for
// the Python tests and bench.py.  Exceptions become B2_E* codes + b2_last_error().
#define B2_WITH_CUDA_RUNTIME 1
#include <cuda_runtime.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <thread>
#include <vector>
#include <exception>

#include "../b2_internal.h"
#include "trtlab/tensorrt/tensorrt.h"
#include "trtlab_host.h"

using namespace trtlab;
using namespace trtlab::TensorRT;
using b2i::fail;

struct trt_manager {
    std::shared_ptr<InferenceManager> mgr;
    std::shared_ptr<Runtime> runtime;
    std::unique_ptr<trtlab::MetricsExposer> exposer;  // declared last: stops serving before the manager goes away
};

#define TRT_TRY try {
#define TRT_CATCH                                                                  \
    }                                                                              \
    catch (const std::bad_alloc&) { return fail(B2_ENOMEM, "out of memory"); }     \
    catch (const std::exception& ex) { return fail(B2_EINVAL, "%s", ex.what()); }

extern "C" {

int trt_manager_create(int max_exec, int max_buffers, int pre_threads, int cuda_threads, int post_threads,
                       trt_manager** out) {
    if (!out || max_exec < 1) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    auto* m = new trt_manager();
    m->mgr = std::make_shared<InferenceManager>(max_exec, max_buffers);
    m->runtime = std::make_shared<StandardRuntime>();
    // same pool names/sizes the reference's infer.x registers (examples/00_TensorRT/infer.cc:91-93)
    m->mgr->RegisterThreadPool("pre", std::make_unique<ThreadPool>(size_t(std::max(pre_threads, 1))));
    m->mgr->RegisterThreadPool("cuda", std::make_unique<ThreadPool>(size_t(std::max(cuda_threads, 1))));
    m->mgr->RegisterThreadPool("post", std::make_unique<ThreadPool>(size_t(std::max(post_threads, 1))));
    m->mgr->RegisterRuntime("default", m->runtime);
    m->mgr->SetActiveRuntime("default");
    *out = m;
    return B2_OK;
    TRT_CATCH
}

void trt_manager_destroy(trt_manager* m) {
    if (!m) return;
    m->mgr->JoinAllThreads();
    delete m;
}

int trt_manager_register_model(trt_manager* m, const char* name, const void* blob, size_t nbytes, int max_concurrency) {
    if (!m || !name || !blob) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    auto model = m->mgr->ActiveRuntime().DeserializeEngine(blob, nbytes);
    if (max_concurrency > 0)
        m->mgr->RegisterModel(name, model, uint32_t(max_concurrency));
    else
        m->mgr->RegisterModel(name, model);
    return B2_OK;
    TRT_CATCH
}

int trt_manager_allocate(trt_manager* m) {
    if (!m) return fail(B2_EINVAL, "null manager");
    TRT_TRY
    m->mgr->AllocateResources();
    return B2_OK;
    TRT_CATCH
}

int trt_manager_infer(trt_manager* m, const char* model_name, int batch, const void* input, size_t input_bytes,
                      float* output, size_t output_bytes, double* compute_seconds) {
    if (!m || !model_name || !input || !output) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    auto model = m->mgr->GetModel(model_name);
    if (model->GetInputBindingIds().size() != 1 || model->GetOutputBindingIds().size() != 1)
        return fail(B2_EINVAL, "trt_manager_infer handles single-input single-output models");
    const uint32_t in_id = model->GetInputBindingIds()[0], out_id = model->GetOutputBindingIds()[0];
    if (batch < 1 || batch > model->GetMaxBatchSize()) return fail(B2_EINVAL, "batch %d out of range", batch);
    if (input_bytes != model->GetBinding(in_id).bytesPerBatchItem * size_t(batch) ||
        output_bytes != model->GetBinding(out_id).bytesPerBatchItem * size_t(batch))
        return fail(B2_EINVAL, "binding size mismatch");
    InferRunner runner(model, m->mgr);
    auto fut = runner.Infer(
        [&](Bindings& b) {  // "pre" stage: fill the pinned input binding
            b.SetBatchSize(uint32_t(batch));
            memcpy(b.HostAddress(in_id), input, input_bytes);
        },
        [&](std::shared_ptr<Bindings>& b) {  // "post" stage: read the pinned output binding
            memcpy(output, b->HostAddress(out_id), output_bytes);
            return b->ComputeTime();  // device time of the forward pass (ExecutionContext::Synchronize, server.cc:169)
        });
    const double seconds = fut.get();
    if (compute_seconds) *compute_seconds = seconds;
    return B2_OK;
    TRT_CATCH
}

int trt_manager_infer_batched(trt_manager* m, const char* model_name, int n, const void* inputs, void* outputs, int window_us,
                              int* batches_executed) {
    if (!m || !model_name || n < 1 || !inputs || !outputs) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    auto model = m->mgr->GetModel(model_name);
    const size_t in_item = model->GetBinding(model->GetInputBindingIds()[0]).bytesPerBatchItem;
    const size_t out_item = model->GetBinding(model->GetOutputBindingIds()[0]).bytesPerBatchItem;
    BatchedInferRunner runner(model, m->mgr, std::chrono::microseconds(window_us > 0 ? window_us : 2000));
    std::vector<BatchedInferRunner::future_type> futures;
    for (int i = 0; i < n; ++i)
        futures.push_back(runner.Infer(static_cast<const char*>(inputs) + size_t(i) * in_item, static_cast<char*>(outputs) + size_t(i) * out_item));
    for (auto& f : futures) f.get();
    runner.Shutdown();
    if (batches_executed) *batches_executed = int(runner.BatchesExecuted());
    return B2_OK;
    TRT_CATCH
}

// The same path as one continuous flood of `n` single-image requests whose inputs cycle through `ring` (ring_items
// images); *window_seconds spans the completions of requests [warm, n - cool): the batcher, every lane and every Buffers
// are busy on both sides of the window, so the rate is free of the pipeline's fill and drain.
int trt_manager_bench_batched(trt_manager* m, const char* model_name, int n, const void* ring, int ring_items, void* outputs,
                              int window_us, int warm, int cool, double* window_seconds, double* total_seconds, int* batches_executed) {
    if (!m || !model_name || n < 1 || !ring || ring_items < 1 || !outputs || warm < 0 || cool < 0 || warm + cool >= n || !window_seconds)
        return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    auto model = m->mgr->GetModel(model_name);
    const size_t in_item = model->GetBinding(model->GetInputBindingIds()[0]).bytesPerBatchItem;
    const size_t out_item = model->GetBinding(model->GetOutputBindingIds()[0]).bytesPerBatchItem;
    BatchedInferRunner runner(model, m->mgr, std::chrono::microseconds(window_us > 0 ? window_us : 2000));
    std::vector<BatchedInferRunner::future_type> futures;
    futures.reserve(size_t(n));
    const auto t0 = std::chrono::steady_clock::now();
    for (int i = 0; i < n; ++i)
        futures.push_back(runner.Infer(static_cast<const char*>(ring) + size_t(i % ring_items) * in_item,
                                       static_cast<char*>(outputs) + size_t(i) * out_item));
    std::chrono::steady_clock::time_point t_lo = t0, t_hi = t0;
    for (int i = 0; i < n; ++i) {
        futures[size_t(i)].get();
        if (i == warm - 1) t_lo = std::chrono::steady_clock::now();  // request `warm` starts counting after its predecessor is out
        if (i == n - cool - 1) t_hi = std::chrono::steady_clock::now();
    }
    const auto t1 = std::chrono::steady_clock::now();
    runner.Shutdown();
    *window_seconds = std::chrono::duration<double>(t_hi - t_lo).count();
    if (total_seconds) *total_seconds = std::chrono::duration<double>(t1 - t0).count();
    if (batches_executed) *batches_executed = int(runner.BatchesExecuted());
    return B2_OK;
    TRT_CATCH
}

int trt_manager_metrics_text(trt_manager* m, char* buf, size_t cap) {
    if (!m || !buf || cap == 0) return -fail(B2_EINVAL, "bad arguments");
    try {
        m->mgr->GetMetrics().SamplePower(m->mgr->Device());
        const std::string text = m->mgr->GetMetrics().Expose();
        const size_t n = std::min(text.size(), cap - 1);
        memcpy(buf, text.data(), n);
        buf[n] = 0;
        return int(text.size());
    } catch (const std::exception& e) {
        return -fail(B2_ESTATE, "%s", e.what());
    }
}

// Give every pooled Buffers a distinct input batch in its pinned host stack.  Bindings are bump-allocated
// from a stack that is Reset() on return, so the addresses (and contents) persist across requests.
// HTTP endpoint for the Prometheus scraper (reference examples/02_TensorRT_GRPC/src/metrics.cc:34-60: Exposer on a port)
int trt_manager_serve_metrics(trt_manager* m, int port, int* bound_port) {
    if (!m) return fail(B2_EINVAL, "null manager");
    TRT_TRY
    auto mgr = m->mgr;
    m->exposer = std::make_unique<trtlab::MetricsExposer>(port, [mgr] {
        mgr->GetMetrics().SamplePower(mgr->Device());
        return mgr->GetMetrics().Expose();
    });
    if (bound_port) *bound_port = m->exposer->Port();
    return B2_OK;
    TRT_CATCH
}

int trt_manager_prefill_inputs(trt_manager* m, const char* model_name, const void* ring, size_t ring_batches) {
    if (!m || !model_name || !ring || ring_batches == 0) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    auto model = m->mgr->GetModel(model_name);
    const uint32_t in_id = model->GetInputBindingIds()[0];
    const size_t bytes = model->GetBinding(in_id).bytesPerBatchItem * size_t(model->GetMaxBatchSize());
    std::vector<std::shared_ptr<Buffers>> held;
    for (int i = 0; i < m->mgr->MaxCopyConcurrency(); ++i) {
        auto buffers = m->mgr->GetBuffers();
        auto bindings = buffers->CreateBindings(model);
        memcpy(bindings->HostAddress(in_id), reinterpret_cast<const char*>(ring) + (size_t(i) % ring_batches) * bytes, bytes);
        held.push_back(buffers);  // hold all of them so each pop yields a different Buffers
    }
    return B2_OK;
    TRT_CATCH
}

int trt_manager_bench(trt_manager* m, const char* model_name, int batch, double seconds, size_t max_batches,
                      double* results16, double* latencies, size_t lat_cap, size_t* lat_count) {
    if (!m || !model_name || !results16) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    auto model = m->mgr->GetModel(model_name);
    InferBench bench(m->mgr);
    std::vector<double> lat;
    InferBench::ModelsList models = {model};
    auto res = bench.Run(models, uint32_t(batch), seconds, max_batches, latencies ? &lat : nullptr);
    for (int i = 0; i < 16; ++i) results16[i] = 0.0;
    for (const auto& kv : *res)
        if (int(kv.first) < 16) results16[int(kv.first)] = kv.second;
    if (latencies && lat_count) {
        *lat_count = std::min(lat.size(), lat_cap);
        memcpy(latencies, lat.data(), *lat_count * sizeof(double));
    }
    return B2_OK;
    TRT_CATCH
}

// One CONTINUOUS closed loop of warm + steps + cool requests (InferBench::Run); rates the `steps` completions in the
// middle: *window_seconds = time from the warm-th completion to the (warm + steps)-th, latencies[] = those requests'
// latencies.  The pipeline (8 Buffers, 4 lanes) is full on both sides of the window, so a short window measures the
// steady state instead of the fill / drain transients a bracketed run of the same length is dominated by.
int trt_manager_bench_windows(trt_manager* m, const char* model_name, int batch, size_t warm, size_t steps, size_t windows, size_t cool,
                              double* window_seconds, double* latencies, size_t lat_cap, size_t* lat_count) {
    if (!m || !model_name || !window_seconds || steps < 1 || windows < 1) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    auto model = m->mgr->GetModel(model_name);
    InferBench bench(m->mgr);
    std::vector<double> lat, done;
    InferBench::ModelsList models = {model};
    const size_t total = warm + steps * windows + cool;
    bench.Run(models, uint32_t(batch), 3600.0, total, &lat, &done);
    if (done.size() != total) return fail(B2_EINVAL, "bench loop ended early (%zu of %zu requests)", done.size(), total);
    std::vector<size_t> order(done.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return done[a] < done[b]; });
    for (size_t w = 0; w < windows; ++w) {  // window w = completions warm + w*steps + 1 .. warm + (w+1)*steps
        const size_t first = warm + w * steps;
        const double t_begin = first ? done[order[first - 1]] : 0.0;
        window_seconds[w] = done[order[first + steps - 1]] - t_begin;
    }
    size_t n = 0;
    for (size_t k = warm; k < warm + steps * windows && latencies && n < lat_cap; ++k) latencies[n++] = lat[order[k]];
    if (lat_count) *lat_count = n;
    return B2_OK;
    TRT_CATCH
}
int trt_manager_bench_window(trt_manager* m, const char* model_name, int batch, size_t warm, size_t steps, size_t cool,
                             double* window_seconds, double* latencies, size_t lat_cap, size_t* lat_count) {
    return trt_manager_bench_windows(m, model_name, batch, warm, steps, 1, cool, window_seconds, latencies, lat_cap, lat_count);
}

// H2D / compute / D2H breakdown of the v2 single-stream pipeline (TimedBenchmarkWorkspace)
int trt_timed_pipeline(const void* blob, size_t nbytes, int iters, float* h2d_ms, float* compute_ms, float* d2h_ms) {
    if (!blob || iters < 1) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    auto runtime = std::make_shared<StandardRuntime>();
    auto model = runtime->deserialize_engine(blob, nbytes);
    TimedBenchmarkWorkspace ws(model);
    double a = 0, b = 0, c = 0;
    for (int i = 0; i < iters + 2; ++i) {
        ws.enqueue_pipeline();
        if (cudaStreamSynchronize(ws.stream()) != cudaSuccess) return fail(B2_ECUDA, "pipeline failed");
        if (i >= 2) {
            a += ws.get_h2d_time_ms();
            b += ws.get_compute_time_ms();
            c += ws.get_d2h_time_ms();
        }
    }
    if (h2d_ms) *h2d_ms = float(a / iters);
    if (compute_ms) *compute_ms = float(b / iters);
    if (d2h_ms) *d2h_ms = float(c / iters);
    return B2_OK;
    TRT_CATCH
}

// Device-resident throughput: `contexts` execution contexts on independent streams, inputs cycled through
// a device ring (sized by the caller to exceed L2), `steps` forward passes issued round-robin, timed with
// CUDA events from the first launch to the completion of the last stream.
// v2 surface: BenchmarkWorkspace (StaticSingleModelGraphWorkspace underneath: the CALLER captures b2_context_enqueue into
// its own CUDA graph, reference workspace.cc:51-56,75) -- pinned input -> async_h2d -> enqueue() -> async_d2h, `iters`
// times; the output of the last pass is returned.  `managed_runtime`: weights through ManagedRuntime (allocator.cc:72-77).
int trt_workspace_infer(const void* blob, size_t nbytes, const void* input, size_t input_bytes, void* output, size_t output_bytes,
                        int managed_runtime, int iters) {
    if (!blob || !input || !output || iters < 1) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    std::shared_ptr<Runtime> rt;
    if (managed_runtime) rt = std::make_shared<ManagedRuntime>();
    else rt = std::make_shared<StandardRuntime>();
    auto model = rt->DeserializeEngine(blob, nbytes);
    if (model->GetInputBindingIds().size() != 1 || model->GetOutputBindingIds().size() != 1)
        return fail(B2_EINVAL, "trt_workspace_infer handles single-input single-output models");
    const uint32_t in_id = model->GetInputBindingIds()[0], out_id = model->GetOutputBindingIds()[0];
    BenchmarkWorkspace ws(model);
    if (input_bytes != ws.binding_bytes(in_id) || output_bytes != ws.binding_bytes(out_id))
        return fail(B2_EINVAL, "binding size mismatch (the workspace runs at max batch): %zu/%zu vs %zu/%zu", input_bytes,
                    ws.binding_bytes(in_id), output_bytes, ws.binding_bytes(out_id));
    memcpy(ws.host_binding(in_id), input, input_bytes);
    for (int i = 0; i < iters; ++i) {
        ws.async_h2d();
        ws.enqueue();
        ws.async_d2h();
    }
    if (cudaStreamSynchronize(ws.stream()) != cudaSuccess) return fail(B2_ECUDA, "workspace stream failed: %s", cudaGetErrorString(cudaGetLastError()));
    memcpy(output, ws.host_binding(out_id), output_bytes);
    return B2_OK;
    TRT_CATCH
}

namespace {
struct RewindableCyclicBuffers : CyclicBuffers<CudaPinnedHostMemory, CudaDeviceMemory> {
    using CyclicBuffers<CudaPinnedHostMemory, CudaDeviceMemory>::CyclicBuffers;
    void Rewind() { Reset(); }  // what InferenceManager::GetBuffers()'s return hook does for pooled Buffers
};
}  // namespace

// The hot path by hand (SURVEY.md 8a rows a2-a9) over CyclicBuffers<CudaPinnedHostMemory, CudaDeviceMemory> (buffers.h:122-154):
// `rounds` requests, each cutting its bindings from the segment ring (so the ring wraps and recycles segments), through
// CreateBindings / CopyToDevice / ExecutionContext::Infer / CopyFromDevice / Synchronize.  Output of the last request.
int trt_cyclic_infer(const void* blob, size_t nbytes, int batch, const void* input, size_t input_bytes, void* output,
                     size_t output_bytes, int managed_runtime, int rounds, double* compute_seconds) {
    if (!blob || !input || !output || rounds < 1 || batch < 1) return fail(B2_EINVAL, "bad arguments");
    TRT_TRY
    std::shared_ptr<Runtime> rt;
    if (managed_runtime) rt = std::make_shared<ManagedRuntime>();
    else rt = std::make_shared<StandardRuntime>();
    auto model = rt->DeserializeEngine(blob, nbytes);
    if (model->GetInputBindingIds().size() != 1 || model->GetOutputBindingIds().size() != 1)
        return fail(B2_EINVAL, "trt_cyclic_infer handles single-input single-output models");
    if (batch > model->GetMaxBatchSize()) return fail(B2_EINVAL, "batch %d out of range", batch);
    const uint32_t in_id = model->GetInputBindingIds()[0], out_id = model->GetOutputBindingIds()[0];
    if (input_bytes != model->GetBinding(in_id).bytesPerBatchItem * size_t(batch) ||
        output_bytes != model->GetBinding(out_id).bytesPerBatchItem * size_t(batch))
        return fail(B2_EINVAL, "binding size mismatch");
    // every segment holds ONE request's bindings (+ alignment), so each request moves the ring on by one segment
    const size_t per_request = model->GetBindingMemorySize() + model->GetBindingsCount() * 256;
    auto buffers = std::make_shared<RewindableCyclicBuffers>(
        std::make_unique<CyclicAllocator<CudaPinnedHostMemory>>(3, per_request), std::make_unique<CyclicAllocator<CudaDeviceMemory>>(3, per_request));
    ExecutionContext ctx(std::max<size_t>(model->GetActivationsMemorySize(), 1024));
    double seconds = 0.0;
    for (int r = 0; r < rounds; ++r) {
        auto bindings = buffers->CreateBindings(model);
        bindings->SetBatchSize(uint32_t(batch));
        memcpy(bindings->HostAddress(in_id), input, input_bytes);
        bindings->CopyToDevice(bindings->InputBindings());
        ctx.SetContext(model->CreateExecutionContext());
        ctx.Infer(bindings);
        bindings->CopyFromDevice(bindings->OutputBindings());
        seconds = ctx.Synchronize();
        bindings->Synchronize();
        if (r == rounds - 1) memcpy(output, bindings->HostAddress(out_id), output_bytes);
        ctx.Reset();
        bindings.reset();
        buffers->Rewind();  // releases the request's descriptors: the segment may be recycled
    }
    if (compute_seconds) *compute_seconds = seconds;
    return B2_OK;
    TRT_CATCH
}

int trt_device_throughput(const void* blob, size_t nbytes, int contexts, int batch, int steps, int warmup,
                          const void* host_ring, int ring_batches, double* elapsed_ms, int* launches_per_step,
                          void* last_outputs, size_t last_outputs_bytes) {
    if (!blob || contexts < 1 || steps < 1 || !host_ring || ring_batches < 1 || !elapsed_ms) return fail(B2_EINVAL, "bad arguments");
    b2_runtime* rt = nullptr;
    b2_engine* eng = nullptr;
    int rc = b2_runtime_create(&rt);
    if (rc) return rc;
    rc = b2_engine_deserialize(rt, blob, nbytes, &eng);
    if (rc) {
        b2_runtime_destroy(rt);
        return rc;
    }
    {   // tactics are timed ahead of the requests, in the regime of the run (`contexts` concurrent streams)
        const char* at = getenv("B2_AUTOTUNE");
        if (!at || atoi(at) != 0) rc = b2_engine_tune(eng, at ? atoi(at) : std::max(1, std::min(contexts, 8)), 0);
        if (rc) {
            b2_engine_destroy(eng);
            b2_runtime_destroy(rt);
            return rc;
        }
    }
    const int nb = b2_engine_nb_bindings(eng);
    int in_id = -1;
    std::vector<size_t> bytes(nb);
    for (int i = 0; i < nb; ++i) {
        int32_t dims[8];
        int nd = 0;
        b2_engine_binding_dims(eng, i, dims, &nd);
        size_t n = dtype_size(b2_engine_binding_dtype(eng, i));
        for (int d = 0; d < nd; ++d) n *= size_t(dims[d]);
        bytes[i] = n * size_t(b2_engine_max_batch(eng));
        if (b2_engine_binding_is_input(eng, i)) in_id = i;
    }
    auto batch_bytes = [&](int i) { return bytes[size_t(i)] / size_t(b2_engine_max_batch(eng)) * size_t(batch); };
    if (last_outputs) {
        size_t want = 0;
        for (int i = 0; i < nb; ++i)
            if (i != in_id) want += batch_bytes(i);
        if (last_outputs_bytes != want) {
            b2_engine_destroy(eng);
            b2_runtime_destroy(rt);
            return fail(B2_EINVAL, "last_outputs_bytes %zu != %zu (the output bindings of one batch)", last_outputs_bytes, want);
        }
    }
    struct Ctx {
        b2_context* c = nullptr;
        void* scratch = nullptr;
        std::vector<void*> bind;
        cudaStream_t s = nullptr;
        cudaEvent_t done = nullptr;
    };
    std::vector<Ctx> ctx(contexts);
    std::vector<void*> ring(ring_batches, nullptr);
    cudaStream_t ctrl = nullptr;
    cudaEvent_t start = nullptr, stop = nullptr;
    int status = B2_OK;
    auto cuda_ok = [&](cudaError_t e, const char* what) {
        if (e != cudaSuccess && status == B2_OK) status = fail(B2_ECUDA, "%s: %s", what, cudaGetErrorString(e));
        return e == cudaSuccess;
    };
    const size_t in_bytes = bytes[in_id] / size_t(b2_engine_max_batch(eng)) * size_t(batch);
    for (int r = 0; r < ring_batches && status == B2_OK; ++r) {
        if (cuda_ok(cudaMalloc(&ring[r], bytes[in_id]), "cudaMalloc ring"))
            cuda_ok(cudaMemcpy(ring[r], reinterpret_cast<const char*>(host_ring) + size_t(r) * in_bytes, in_bytes, cudaMemcpyHostToDevice), "ring upload");
    }
    for (auto& x : ctx) {
        if (status != B2_OK) break;
        if ((status = b2_context_create(eng, &x.c))) break;
        // the contexts share the GPU: each persistent network kernel gets its share of the 2 x 148 CTA slots (B2_NET_CTAS overrides)
        if (!getenv("B2_NET_CTAS")) b2_context_set_option(x.c, "net_ctas", std::max(1, 296 / contexts));
        if (!cuda_ok(cudaMalloc(&x.scratch, std::max<size_t>(b2_engine_device_memory_size(eng), 1024)), "cudaMalloc scratch")) break;
        if ((status = b2_context_set_device_memory(x.c, x.scratch))) break;
        x.bind.assign(nb, nullptr);
        for (int i = 0; i < nb; ++i)
            if (i != in_id && !cuda_ok(cudaMalloc(&x.bind[i], bytes[i]), "cudaMalloc binding")) break;
        cuda_ok(cudaStreamCreate(&x.s), "cudaStreamCreate");
        cuda_ok(cudaEventCreateWithFlags(&x.done, cudaEventDisableTiming), "cudaEventCreate");
    }
    if (status == B2_OK) {
        cuda_ok(cudaStreamCreate(&ctrl), "cudaStreamCreate");
        cuda_ok(cudaEventCreate(&start), "cudaEventCreate");
        cuda_ok(cudaEventCreate(&stop), "cudaEventCreate");
    }
    // B2_PROBE_STAGGER=1: de-phase the streams (stream k first runs one forward pass of a smaller batch), the way
    // independently arriving requests meet each other; without it all contexts march through the layers in lockstep.
    const int tiny_h2d = getenv("B2_PROBE_TINY_H2D") ? atoi(getenv("B2_PROBE_TINY_H2D")) : 0;
    void *tiny_dev = nullptr, *tiny_host = nullptr;
    if (tiny_h2d > 0) {
        cuda_ok(cudaMalloc(&tiny_dev, size_t(tiny_h2d)), "cudaMalloc probe");
        cuda_ok(cudaMallocHost(&tiny_host, size_t(tiny_h2d)), "cudaMallocHost probe");
    }
    const bool stagger = getenv("B2_PROBE_STAGGER") && atoi(getenv("B2_PROBE_STAGGER")) > 0;
    auto issue = [&](int n_steps, int offset) {
        for (int k = 1; stagger && k < contexts && status == B2_OK; ++k) {
            Ctx& x = ctx[size_t(k)];
            x.bind[in_id] = ring[0];
            status = b2_context_enqueue(x.c, std::max(1, batch * k / contexts), x.bind.data(), x.s, nullptr);
        }
        for (int i = 0; i < n_steps && status == B2_OK; ++i) {
            Ctx& x = ctx[size_t(i % contexts)];
            x.bind[in_id] = ring[size_t((i + offset) % ring_batches)];
            // B2_PROBE_TINY_H2D=n: a n-byte pinned->device copy ahead of every forward pass (diagnostic: the cost of a
            // copy-engine -> compute dependency in front of the graph launch, without the PCIe traffic of a real input)
            if (tiny_h2d > 0) cudaMemcpyAsync(tiny_dev, tiny_host, size_t(tiny_h2d), cudaMemcpyHostToDevice, x.s);
            status = b2_context_enqueue(x.c, batch, x.bind.data(), x.s, nullptr);
        }
    };
    if (status == B2_OK) {
        issue(std::max(warmup, contexts * ring_batches <= 256 ? contexts * ring_batches : warmup), 0);  // also builds every cached graph
        cuda_ok(cudaDeviceSynchronize(), "warmup sync");
    }
    // B2_PROBE_BG_H2D=1: keep the copy engine busy with pinned 'input' uploads nobody consumes while the forward passes
    // run -- isolates how much PCIe traffic alone slows the kernels down (diagnostic, off by default)
    std::atomic<bool> bg_stop{false};
    std::thread bg;
    if (status == B2_OK && getenv("B2_PROBE_BG_H2D") && atoi(getenv("B2_PROBE_BG_H2D")) > 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        bg = std::thread([&, dev] {
            cudaSetDevice(dev);
            void *h = nullptr, *d = nullptr;
            cudaStream_t s = nullptr;
            if (cudaMallocHost(&h, in_bytes) == cudaSuccess && cudaMalloc(&d, in_bytes) == cudaSuccess &&
                cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess) {
                const int burst = atoi(getenv("B2_PROBE_BG_H2D"));  // copies queued per host synchronisation
                while (!bg_stop.load()) {
                    for (int k = 0; k < burst; ++k) cudaMemcpyAsync(d, h, in_bytes, cudaMemcpyHostToDevice, s);
                    cudaStreamSynchronize(s);
                }
            }
            if (s) cudaStreamDestroy(s);
            if (d) cudaFree(d);
            if (h) cudaFreeHost(h);
        });
    }
    if (status == B2_OK) {
        cuda_ok(cudaEventRecord(start, ctrl), "record start");
        for (auto& x : ctx) cuda_ok(cudaStreamWaitEvent(x.s, start, 0), "wait start");
        issue(steps, 0);
        for (auto& x : ctx) {
            cuda_ok(cudaEventRecord(x.done, x.s), "record done");
            cuda_ok(cudaStreamWaitEvent(ctrl, x.done, 0), "wait done");
        }
        cuda_ok(cudaEventRecord(stop, ctrl), "record stop");
        cuda_ok(cudaStreamSynchronize(ctrl), "sync");
        float ms = 0.f;
        if (status == B2_OK && cuda_ok(cudaEventElapsedTime(&ms, start, stop), "elapsed")) *elapsed_ms = ms;
        if (launches_per_step) *launches_per_step = b2_context_nb_launches(ctx[0].c, batch);
        if (status == B2_OK && last_outputs) {  // outside the timed region; no later step used this context
            const Ctx& x = ctx[size_t((steps - 1) % contexts)];
            char* dst = static_cast<char*>(last_outputs);
            for (int i = 0; i < nb; ++i) {
                if (i == in_id) continue;
                if (!cuda_ok(cudaMemcpy(dst, x.bind[size_t(i)], batch_bytes(i), cudaMemcpyDeviceToHost), "last outputs download")) break;
                dst += batch_bytes(i);
            }
        }
    }
    bg_stop = true;
    if (bg.joinable()) bg.join();
    cudaDeviceSynchronize();
    if (tiny_dev) cudaFree(tiny_dev);
    if (tiny_host) cudaFreeHost(tiny_host);
    for (auto& x : ctx) {
        if (x.c) b2_context_destroy(x.c);
        if (x.scratch) cudaFree(x.scratch);
        for (int i = 0; i < nb && i < int(x.bind.size()); ++i)
            if (i != in_id && x.bind[i]) cudaFree(x.bind[i]);
        if (x.s) cudaStreamDestroy(x.s);
        if (x.done) cudaEventDestroy(x.done);
    }
    for (void* p : ring)
        if (p) cudaFree(p);
    if (ctrl) cudaStreamDestroy(ctrl);
    if (start) cudaEventDestroy(start);
    if (stop) cudaEventDestroy(stop);
    b2_engine_destroy(eng);
    b2_runtime_destroy(rt);
    return status;
}

}  // extern "C"
