// trtlab::TensorRT -- the reference's C++ surface for the per-request inference hot path, re-hosted on
// the B200-native engine (include/b200infer.h) instead of nvinfer1.  No NvInfer.h is included anywhere.
//
// v1 ("legacy", the drop-in contract named by the north star; reference include root
// tensorrt/laboratory/*.h):  Runtime/StandardRuntime/ManagedRuntime, Model, Buffers/FixedBuffers,
// Bindings, ExecutionContext, InferenceManager, InferRunner, InferBench.
//   reference: trtlab/tensorrt/src/{inference_manager,buffers,bindings,infer_bench}.cc,
//              trtlab/tensorrt/include/trtlab/tensorrt/{infer_runner,infer_bench,bindings,buffers}.h
// v2 (what the reference tree links today): Runtime::deserialize_engine, Model::binding_*,
//   StaticSingleModelGraphWorkspace / BenchmarkWorkspace / TimedBenchmarkWorkspace.
//   reference: trtlab/tensorrt/src/{runtime,model,execution_context,workspace}.cc
#pragma once

#include <atomic>
#include <chrono>
#include <cstring>
#include <functional>
#include <future>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "b200cuda.h"
#include "b200infer.h"
#include "trtlab/core/batcher.h"
#include "trtlab/tensorrt/metrics.h"
#include "trtlab/core/hotpath_core.h"
#include "trtlab/cuda/sync.h"

// CUDA handle aliases: when the CUDA runtime header is present use its types, otherwise opaque pointers
#if defined(__CUDACC__) || defined(__CUDA_RUNTIME_H__) || defined(B2_WITH_CUDA_RUNTIME)
#include <cuda_runtime.h>
#else
typedef struct CUstream_st* cudaStream_t;
typedef struct CUevent_st* cudaEvent_t;
#endif

namespace trtlab {
namespace TensorRT {

class Model;
class Buffers;
class Bindings;
class Runtime;
class InferenceManager;

// bytes of one element of a B2_DT_* binding dtype (the one place binding sizes are derived from)
size_t dtype_size(int dtype);

// ------------------------------------------------------------------------------------------------
// memory tags used by FixedBuffers<Host, Device> (reference trtlab/cuda memory types:
// trtlab/cuda/include/trtlab/cuda/memory/device_memory.h:36-84)
// ------------------------------------------------------------------------------------------------
struct CudaPinnedHostMemory {
    static const char* TypeName() { return "CudaPinnedHostMemory"; }
    static constexpr size_t DefaultAlignment() { return 64; }
    static void* Allocate(size_t bytes);
    static void Free(void* ptr);
};
struct CudaDeviceMemory {
    static const char* TypeName() { return "CudaDeviceMemory"; }
    static constexpr size_t DefaultAlignment() { return 256; }
    static void* Allocate(size_t bytes);
    static void Free(void* ptr);
};

// bump allocator over one allocation; Reset() rewinds (legacy MemoryStack semantics, see
// examples/10_Internals/README.md:41-48)
template <typename MemoryType>
class MemoryStack {
  public:
    explicit MemoryStack(size_t size) : m_Size(size), m_Used(0) {
        m_Base = static_cast<char*>(MemoryType::Allocate(size));
        if (!m_Base) throw std::bad_alloc();
    }
    ~MemoryStack() { MemoryType::Free(m_Base); }
    DELETE_COPYABILITY(MemoryStack);
    void* Allocate(size_t size) {
        const size_t start = Align(m_Used, MemoryType::DefaultAlignment());
        if (start + size > m_Size) throw std::bad_alloc();
        m_Used = start + size;
        return m_Base + start;
    }
    void Reset() { m_Used = 0; }
    size_t Size() const { return m_Size; }
    size_t Allocated() const { return m_Used; }
    size_t Available() const { return m_Size - m_Used; }

  private:
    char* m_Base;
    size_t m_Size, m_Used;
};

// ------------------------------------------------------------------------------------------------
// Model  (v1 method names observed at the reference's call sites: inference_manager.cc:112-154,
// bindings.cc:58,167,173, pybind/trtlab/infer.cc:214-269; v2: model.h:17-47, model.cc:76-117)
// ------------------------------------------------------------------------------------------------
struct IExecutionContext {  // stands in for nvinfer1::IExecutionContext (created without device memory)
    explicit IExecutionContext(b2_context* c) : handle(c) {}
    ~IExecutionContext() { b2_context_destroy(handle); }
    DELETE_COPYABILITY(IExecutionContext);
    b2_context* handle;
};

class Model {
  public:
    struct TensorBindingInfo {
        std::string name;
        bool isInput;
        int dtype;  // B2_DT_*
        size_t dtypeSize;
        std::vector<int> dims;
        size_t elementsPerBatchItem;
        size_t bytesPerBatchItem;
    };

    Model(b2_engine* engine, std::shared_ptr<Runtime> runtime);
    virtual ~Model();
    DELETE_COPYABILITY(Model);

    const std::string& Name() const { return m_Name; }
    void SetName(const std::string& name) { m_Name = name; }

    virtual int GetMaxBatchSize() const;
    uint32_t GetBindingsCount() const { return uint32_t(m_Bindings.size()); }
    const TensorBindingInfo& GetBinding(uint32_t id) const;
    const TensorBindingInfo& GetBinding(const std::string& name) const;
    uint32_t BindingId(const std::string& name) const;
    const std::vector<uint32_t>& GetInputBindingIds() const { return m_Inputs; }
    const std::vector<uint32_t>& GetOutputBindingIds() const { return m_Outputs; }
    size_t GetBindingMemorySize() const;      // sum over bindings at max batch
    size_t GetActivationsMemorySize() const;  // replaces ICudaEngine::getDeviceMemorySize
    size_t GetWeightsMemorySize() const;
    std::shared_ptr<IExecutionContext> CreateExecutionContext() const;

    // v2 spellings
    std::size_t binding_element_count(std::uint32_t id) const { return GetBinding(id).elementsPerBatchItem * GetMaxBatchSize(); }
    std::size_t binding_size_in_bytes(std::uint32_t id) const { return GetBinding(id).bytesPerBatchItem * GetMaxBatchSize(); }
    std::string bindings_info() const;
    std::string binding_info(std::uint32_t id) const;
    b2_engine* engine() const { return m_Engine; }
    double flops(int batch) const { return b2_engine_flops(m_Engine, batch); }

  private:
    b2_engine* m_Engine;
    std::shared_ptr<Runtime> m_Runtime;  // an engine keeps its Runtime alive (runtime.cc:138-141)
    std::string m_Name;
    std::vector<TensorBindingInfo> m_Bindings;
    std::vector<uint32_t> m_Inputs, m_Outputs;
};

// ------------------------------------------------------------------------------------------------
// Runtime  (runtime.h:43-110, runtime.cc:47-143)
// ------------------------------------------------------------------------------------------------
class Runtime : public std::enable_shared_from_this<Runtime> {
  public:
    virtual ~Runtime();
    DELETE_COPYABILITY(Runtime);

    std::shared_ptr<Model> DeserializeEngine(const std::string& plan_file);
    std::shared_ptr<Model> DeserializeEngine(const void* data, size_t size);
    std::shared_ptr<Model> deserialize_engine(const std::string& plan_file) { return DeserializeEngine(plan_file); }
    std::shared_ptr<Model> deserialize_engine(const void* data, size_t size) { return DeserializeEngine(data, size); }

    // {address, size} of every weight allocation made while deserializing (NvAllocator::use_weights_allocator)
    struct Pointer {
        void* addr;
        size_t size;
    };
    const std::vector<Pointer>& weight_pointers() const { return m_Weights; }

  protected:
    Runtime();
    std::vector<char> ReadEngineFile(const std::string&) const;
    virtual void* AllocateDevice(uint64_t size, uint64_t alignment, uint32_t flags) = 0;
    virtual void FreeDevice(void* ptr) = 0;

  private:
    static void* AllocThunk(void* user, uint64_t size, uint64_t alignment, uint32_t flags);
    static void FreeThunk(void* user, void* ptr);
    b2_runtime* m_Runtime;
    std::vector<Pointer> m_Weights;
};

// cudaMalloc-backed weights (reference StandardAllocator, allocator.cc:61-70)
class StandardRuntime : public Runtime {
  public:
    StandardRuntime() = default;
  protected:
    void* AllocateDevice(uint64_t size, uint64_t alignment, uint32_t flags) override;
    void FreeDevice(void* ptr) override;
};
// cudaMallocManaged + ReadMostly advice (reference ManagedAllocator, allocator.cc:72-77)
class ManagedRuntime : public Runtime {
  public:
    ManagedRuntime() = default;
  protected:
    void* AllocateDevice(uint64_t size, uint64_t alignment, uint32_t flags) override;
    void FreeDevice(void* ptr) override;
};

// ------------------------------------------------------------------------------------------------
// Buffers / FixedBuffers / Bindings  (buffers.h:52-121, buffers.cc:42-78, bindings.h:60-120,
// bindings.cc:55-175)
// ------------------------------------------------------------------------------------------------
class Buffers : public std::enable_shared_from_this<Buffers> {
  public:
    Buffers();
    virtual ~Buffers();
    DELETE_COPYABILITY(Buffers);

    auto CreateBindings(const std::shared_ptr<Model>&) -> std::shared_ptr<Bindings>;
    inline cudaStream_t Stream() { return m_Stream; }
    void Synchronize();

  protected:
    virtual void Reset() = 0;
    void ConfigureBindings(const std::shared_ptr<Model>& model, std::shared_ptr<Bindings>);
    virtual void* AllocateHost(size_t size) = 0;
    virtual void* AllocateDevice(size_t size) = 0;

  private:
    cudaStream_t m_Stream;
    // The pool hands this object out through a SECOND shared_ptr (own control block, return-to-pool
    // deleter; core/pool.h:193-203), so shared_from_this() would not keep the lease alive.  GetBuffers()
    // records the lease here and CreateBindings() gives it to the Bindings, which is what makes
    // "a Bindings keeps its Buffers checked out" (bindings.h:107-108) actually hold.
    std::weak_ptr<Buffers> m_Lease;
    friend class InferenceManager;
};

template <typename HostMemoryType, typename DeviceMemoryType>
class FixedBuffers : public Buffers {
  public:
    FixedBuffers(size_t host_size, size_t device_size)
        : m_HostStack(new MemoryStack<HostMemoryType>(host_size)), m_DeviceStack(new MemoryStack<DeviceMemoryType>(device_size)) {}
    ~FixedBuffers() override {}

  protected:
    void* AllocateHost(size_t size) final override { return m_HostStack->Allocate(size); }
    void* AllocateDevice(size_t size) final override { return m_DeviceStack->Allocate(size); }
    void Reset() final override {
        m_HostStack->Reset();
        m_DeviceStack->Reset();
    }

  private:
    std::unique_ptr<MemoryStack<HostMemoryType>> m_HostStack;
    std::unique_ptr<MemoryStack<DeviceMemoryType>> m_DeviceStack;
};

// Buffers whose slices come from two rings of segments instead of two rewinding stacks (buffers.h:122-154):
// Reset() does not rewind anything -- the slices cut for a request are released when the Buffers comes back to
// the pool, and a segment is reused once everything cut from it has been released.
template <typename HostMemoryType, typename DeviceMemoryType>
class CyclicBuffers : public Buffers {
  public:
    using HostAllocatorType = std::unique_ptr<CyclicAllocator<HostMemoryType>>;
    using DeviceAllocatorType = std::unique_ptr<CyclicAllocator<DeviceMemoryType>>;
    using HostDescriptor = typename CyclicAllocator<HostMemoryType>::Descriptor;
    using DeviceDescriptor = typename CyclicAllocator<DeviceMemoryType>::Descriptor;

    CyclicBuffers(HostAllocatorType host, DeviceAllocatorType device)
        : m_HostAllocator(std::move(host)), m_DeviceAllocator(std::move(device)) {}
    ~CyclicBuffers() override {}

  protected:
    void* AllocateHost(size_t size) final override {
        m_Held.push_back(m_HostAllocator->Allocate(size));
        return m_Held.back().get();
    }
    void* AllocateDevice(size_t size) final override {
        m_Held.push_back(m_DeviceAllocator->Allocate(size));
        return m_Held.back().get();
    }
    void Reset() final override { m_Held.clear(); }

  private:
    HostAllocatorType m_HostAllocator;
    DeviceAllocatorType m_DeviceAllocator;
    std::vector<std::shared_ptr<void>> m_Held;  // descriptors of the request in flight
};

class Bindings {
  public:
    virtual ~Bindings();

    void* HostAddress(uint32_t binding_id);
    void* DeviceAddress(uint32_t binding_id);
    void** DeviceAddresses();
    void SetHostAddress(int binding_id, void* addr);
    void SetDeviceAddress(int binding_id, void* addr);

    void* ActivationsAddress() { return m_ActivationsAddress; }
    void SetActivationsAddress(void* addr) { m_ActivationsAddress = addr; }

    void CopyToDevice(uint32_t);
    void CopyToDevice(const std::vector<uint32_t>&);
    void CopyToDevice(uint32_t, void*, size_t);
    void CopyFromDevice(uint32_t);
    void CopyFromDevice(const std::vector<uint32_t>&);
    void CopyFromDevice(uint32_t, void*, size_t);

    const std::vector<uint32_t>& InputBindings() const { return m_Model->GetInputBindingIds(); }
    const std::vector<uint32_t>& OutputBindings() const { return m_Model->GetOutputBindingIds(); }

    auto GetModel() -> const std::shared_ptr<Model>& { return m_Model; }
    auto BatchSize() const { return m_BatchSize; }
    void SetBatchSize(uint32_t);

    inline cudaStream_t Stream() const { return m_Buffers->Stream(); }
    void Synchronize() const { m_Buffers->Synchronize(); }
    template <typename ThreadType>
    void Synchronize() const { cuda_sync<ThreadType>::stream_sync(reinterpret_cast<b2_stream_t>(Stream())); }
    // device time of this request's forward pass, filled in by InferRunner's post stage before the user's function runs
    // (what the reference's service reads from ctx->Synchronize(), server.cc:169)
    double ComputeTime() const { return m_ComputeSeconds; }
    void SetComputeTime(double seconds) { m_ComputeSeconds = seconds; }
    size_t BindingSize(uint32_t binding_id) const;

  private:
    Bindings(const std::shared_ptr<Model>, const std::shared_ptr<Buffers>);
    const std::shared_ptr<Model> m_Model;
    const std::shared_ptr<Buffers> m_Buffers;  // a Bindings keeps its Buffers alive (bindings.h:107-108)
    uint32_t m_BatchSize;
    std::vector<void*> m_HostAddresses;
    std::vector<void*> m_DeviceAddresses;
    std::map<uint32_t, void*> m_StagedDevice;  // zero-copy inputs: the device staging address the binding would have used
    void* m_ActivationsAddress;
    double m_ComputeSeconds = 0.0;
    friend class Buffers;
};

// ------------------------------------------------------------------------------------------------
// ExecutionContext  -- v1: the global concurrency token that owns the activation scratch
// (inference_manager.cc:200-204,254-273; contract examples/10_Internals/README.md:50-52)
// ------------------------------------------------------------------------------------------------
class ExecutionContext {
  public:
    // One activation arena and the completion event of the forward pass that used it last.  Several tokens may share
    // a lane: their forward passes are ordered ON THE DEVICE (cudaStreamWaitEvent), so the host can enqueue request
    // n+1 of a lane while request n still runs and the lane never waits for a host round trip between requests.
    struct Lane {
        explicit Lane(size_t workspace_bytes, int index = 0);
        ~Lane();
        void* workspace;
        size_t bytes;
        int index;              // position among the manager's lanes (engine-side contexts are pinned to a lane)
        std::mutex mutex;
        cudaEvent_t last_done;  // nullptr until the lane has been used
    };

    explicit ExecutionContext(size_t workspace_bytes);        // a lane of its own (the reference's token)
    explicit ExecutionContext(std::shared_ptr<Lane> lane);    // one of several tokens queued on `lane`
    virtual ~ExecutionContext();
    DELETE_COPYABILITY(ExecutionContext);

    void SetContext(std::shared_ptr<IExecutionContext> context);
    // async forward pass on bindings->Stream(); records the completion event
    void Infer(const std::shared_ptr<Bindings>&);
    // waits for the completion event, returns the GPU compute time in seconds
    double Synchronize();
    // the same wait under an explicit threading policy: Synchronize<userspace_threads>() polls and yields
    // (cuda_sync, trtlab/cuda/sync.h) instead of parking the OS thread in the driver
    template <typename ThreadType>
    double Synchronize() {
        cuda_sync<ThreadType>::event_sync(reinterpret_cast<b2_event_t>(m_Done));
        return ElapsedSeconds();
    }
    double ElapsedSeconds() const;  // start -> done of the last Infer(); valid once the completion event has fired
    // fiber-friendly variant: 0 when done, 1 while running (cuda_sync<userspace_threads>, sync.h:19-47)
    int Query();
    void Reset();
    int LaneIndex() const { return m_Lane->index; }
    void* Workspace() const { return m_Lane->workspace; }

  private:
    std::shared_ptr<IExecutionContext> m_Context;
    std::shared_ptr<Lane> m_Lane;
    cudaEvent_t m_Start, m_Done;
};

// ------------------------------------------------------------------------------------------------
// InferenceManager (inference_manager.cc:59-327)
// ------------------------------------------------------------------------------------------------
class InferenceManager : public ::trtlab::Resources {
  public:
    InferenceManager(int max_executions, int max_buffers);
    virtual ~InferenceManager();
    DELETE_COPYABILITY(InferenceManager);

    void RegisterModel(const std::string& name, std::shared_ptr<Model> model);
    void RegisterModel(const std::string& name, std::shared_ptr<Model> model, uint32_t max_concurrency);
    void AllocateResources();

    auto GetModel(std::string model_name) -> std::shared_ptr<Model>;
    auto GetBuffers() -> std::shared_ptr<Buffers>;
    auto GetExecutionContext(const Model* model) -> std::shared_ptr<ExecutionContext>;
    auto GetExecutionContext(const std::shared_ptr<Model>& model) -> std::shared_ptr<ExecutionContext>;

    auto AcquireThreadPool(const std::string&) -> ThreadPool&;
    void RegisterThreadPool(const std::string&, std::unique_ptr<ThreadPool> threads);
    bool HasThreadPool(const std::string&) const;
    void JoinAllThreads();

    void RegisterRuntime(const std::string&, std::shared_ptr<Runtime>);
    void SetActiveRuntime(const std::string&);
    Runtime& ActiveRuntime();

    void ForEachModel(std::function<void(const Model&)>);

    int MaxExecConcurrency() const;
    // how the post stage waits for the device: false = cuda_sync<standard_threads> (park in the driver, the default),
    // true = cuda_sync<userspace_threads> (poll + yield; TRTLAB_SYNC=yield), reference trtlab/cuda/sync.h:13-62
    static bool YieldingSync();
    // TRTLAB_ZERO_COPY_INPUT=1: Bindings::CopyToDevice(input) stages nothing -- the engine's input cast reads the mapped
    // pinned host buffer over PCIe itself (the transfer is fused into the first kernel of the forward pass)
    static bool ZeroCopyInput();
    static int EnqueueDepth();  // tokens queued per execution lane (TRTLAB_ENQUEUE_DEPTH, default 2)
    // request / compute summaries, load-ratio histogram, power gauge (metrics.h); fed by InferBench and by services
    Metrics& GetMetrics() { return m_Metrics; }
    // device time of finished forward passes (fed by InferRunner's post stage)
    void RecordComputeTime(double seconds);
    double MeanComputeTime(bool reset);
    int MaxCopyConcurrency() const;

    // CUDA's current device is per thread and defaults to 0: pipeline stages running on pool threads adopt the
    // device the manager was created on (one manager per GPU is the multi-GPU topology, SURVEY.md 8e)
    int Device() const { return m_Device; }
    void ActivateDevice() const;

  private:
    int m_Device;
    Metrics m_Metrics;
    std::atomic<uint64_t> m_ComputeNs{0};
    std::atomic<uint64_t> m_ComputeCount{0};
    int m_MaxExecutions;
    int m_MaxBuffers;
    size_t m_HostStackSize;
    size_t m_DeviceStackSize;
    size_t m_ActivationsSize;
    std::shared_ptr<Pool<Buffers>> m_Buffers;
    std::shared_ptr<Pool<ExecutionContext>> m_ExecutionContexts;
    std::map<std::string, std::shared_ptr<Runtime>> m_Runtimes;
    Runtime* m_ActiveRuntime;
    std::map<std::string, std::unique_ptr<ThreadPool>> m_ThreadPools;
    std::map<std::string, std::shared_ptr<Model>> m_Models;
    // Engine-side contexts per model.  When the model may use every lane (the default) there is ONE POOL PER LANE with
    // EnqueueDepth() contexts each: a context then only ever meets its lane's activation arena, so its launch plans and
    // CUDA graphs (one per batch size) can all be built in AllocateResources() -- nothing is captured, instantiated or
    // tuned on the request path.  A model with capped concurrency keeps the reference's single shared pool.
    std::map<const Model*, std::vector<std::shared_ptr<Pool<IExecutionContext>>>> m_ModelExecutionContexts;
    std::vector<std::shared_ptr<ExecutionContext::Lane>> m_Lanes;
    void PrepareModel(const Model* model);
};

// ------------------------------------------------------------------------------------------------
// InferRunner: pre -> cuda -> post pipeline over the manager's thread pools (infer_runner.h:37-157)
// ------------------------------------------------------------------------------------------------
struct InferRunner : public AsyncComputeWrapper<void(std::shared_ptr<Bindings>&)> {
    InferRunner(std::shared_ptr<Model> model, std::shared_ptr<InferenceManager> resources)
        : m_Model{model}, m_Resources{resources} {}
    InferRunner(InferRunner&&) = delete;
    InferRunner& operator=(InferRunner&&) = delete;
    InferRunner(const InferRunner&) = delete;
    InferRunner& operator=(const InferRunner&) = delete;
    virtual ~InferRunner() {}

    using BindingsHandle = std::shared_ptr<Bindings>;
    using PreFn = std::function<void(Bindings&)>;

    template <typename Post>
    auto Infer(PreFn pre, Post post) {
        auto compute = Wrap(post);
        auto future = compute->Future();
        Enqueue(pre, compute);
        return future.share();
    }

    template <typename Post>
    auto Infer(std::shared_ptr<Bindings> bindings, Post post) {
        auto compute = Wrap(post);
        auto future = compute->Future();
        Enqueue(bindings, compute);
        return future.share();
    }

  protected:
    template <typename T>
    void Enqueue(PreFn Pre, std::shared_ptr<AsyncCompute<T>> Post) {
        auto model = m_Model;
        auto resources = m_Resources;
        Workers("pre").enqueue([model, resources, Pre, Post]() mutable {
            resources->ActivateDevice();
            auto buffers = resources->GetBuffers();
            auto bindings = buffers->CreateBindings(model);
            Pre(*bindings);
            EnqueueStatic(resources, bindings, Post);
        });
    }

    template <typename T>
    void Enqueue(std::shared_ptr<Bindings> bindings, std::shared_ptr<AsyncCompute<T>> Post) {
        EnqueueStatic(m_Resources, bindings, Post);
    }

    // the pipeline stages only capture shared_ptrs, so the InferRunner may die before they run
    template <typename T>
    static void EnqueueStatic(std::shared_ptr<InferenceManager> resources, std::shared_ptr<Bindings> bindings,
                              std::shared_ptr<AsyncCompute<T>> Post) {
        resources->AcquireThreadPool("cuda").enqueue([resources, bindings, Post]() mutable {
            resources->ActivateDevice();
            bindings->CopyToDevice(bindings->InputBindings());                     // H2D
            auto trt_ctx = resources->GetExecutionContext(bindings->GetModel());   // may block on 2 pools
            trt_ctx->Infer(bindings);                                              // forward, async
            bindings->CopyFromDevice(bindings->OutputBindings());                  // D2H
            resources->AcquireThreadPool("post").enqueue([resources, bindings, trt_ctx, Post]() mutable {
                resources->ActivateDevice();
                const bool yielding = InferenceManager::YieldingSync();
                const double compute_seconds =
                    yielding ? trt_ctx->template Synchronize<userspace_threads>() : trt_ctx->Synchronize();
                resources->RecordComputeTime(compute_seconds);
                bindings->SetComputeTime(compute_seconds);
                trt_ctx.reset();  // returns both pool tokens
                if (yielding)
                    bindings->template Synchronize<userspace_threads>();
                else
                    bindings->Synchronize();
                (*Post)(bindings);
                bindings.reset();  // returns the Buffers
            });
        });
    }

    inline ThreadPool& Workers(std::string name) { return m_Resources->AcquireThreadPool(name); }

  public:
    int MaxBatchSize() const { return m_Model->GetMaxBatchSize(); }
    const Model& GetModel() const { return *m_Model; }
    const std::shared_ptr<Model> GetModelSmartPtr() const { return m_Model; }
    InferenceManager& Resources() { return *m_Resources; }

  private:
    std::shared_ptr<Model> m_Model;
    std::shared_ptr<InferenceManager> m_Resources;
};

// ------------------------------------------------------------------------------------------------
// InferBench (infer_bench.h:35-66, infer_bench.cc:39-110)
// ------------------------------------------------------------------------------------------------
enum InferBenchKey {
    kMaxExecConcurrency = 0,
    kMaxCopyConcurrency,
    kBatchSize,
    kWalltime,
    kBatchesComputed,
    kBatchesPerSecond,
    kInferencesPerSecond,
    kSecondsPerBatch,
    kExecutionTimePerBatch,
    // extensions (not in the reference): request latency percentiles, seconds
    kLatencyP50,
    kLatencyP90,
    kLatencyP99,
    kLatencyMax,
    kGpuComputeTimePerBatch  // mean device time of one forward pass (start/done events of its ExecutionContext)
};

// ------------------------------------------------------------------------------------------------
// BatchedInferRunner -- dynamic batching in front of the hot path (SURVEY.md 8f N3, host part): single requests of
// 1..k images are merged by a Dispatcher<StandardBatcher> until the model's max batch is reached or the batching
// window expires, then travel as ONE request through InferRunner (pinned H2D -> forward -> D2H) and are scattered back.
// Same roles as the reference's batching service (examples/03_Batching/inference-batcher.cc:298-366: window 2000 us,
// max batch from the model), with the engine instead of a TRTIS round trip behind it.  Single-input single-output models.
// ------------------------------------------------------------------------------------------------
class BatchedInferRunner {
  public:
    struct Request {
        const void* input;  // `items` batch items in the input binding's dtype/layout; valid until the future is ready
        void* output;       // room for `items` output items
        uint32_t items;
    };
    using future_type = std::shared_future<void>;

    BatchedInferRunner(std::shared_ptr<Model> model, std::shared_ptr<InferenceManager> resources,
                       std::chrono::nanoseconds window = std::chrono::microseconds(2000), size_t workers = 0)
        : m_Model(std::move(model)), m_Resources(std::move(resources)), m_Batches(std::make_shared<std::atomic<size_t>>(0)) {
        TRTLAB_CHECK(m_Model->GetInputBindingIds().size() == 1 && m_Model->GetOutputBindingIds().size() == 1)
            << "BatchedInferRunner handles single-input single-output models";
        auto model_ = m_Model;
        auto res = m_Resources;
        auto batches = m_Batches;
        auto execute = [model_, res, batches](const std::vector<Request>& reqs, std::function<void()> release) {
            res->ActivateDevice();
            const uint32_t in_id = model_->GetInputBindingIds()[0], out_id = model_->GetOutputBindingIds()[0];
            const size_t in_item = model_->GetBinding(in_id).bytesPerBatchItem, out_item = model_->GetBinding(out_id).bytesPerBatchItem;
            auto buffers = res->GetBuffers();
            auto bindings = buffers->CreateBindings(model_);
            buffers.reset();
            uint32_t total = 0;
            for (const auto& r : reqs) {
                memcpy(static_cast<char*>(bindings->HostAddress(in_id)) + size_t(total) * in_item, r.input, size_t(r.items) * in_item);
                total += r.items;
            }
            bindings->SetBatchSize(total);
            InferRunner runner(model_, res);
            auto done = runner.Infer(bindings, [&reqs, out_id, out_item](std::shared_ptr<Bindings>& b) {
                uint32_t at = 0;
                for (const auto& r : reqs) {
                    memcpy(r.output, static_cast<const char*>(b->HostAddress(out_id)) + size_t(at) * out_item, size_t(r.items) * out_item);
                    at += r.items;
                }
                b.reset();
            });
            // get(), not wait(): an exception thrown in the cuda / post stage must reach the batch promise (the dispatcher
            // turns it into set_exception) instead of being reported as success over unwritten outputs.
            // `reqs` lives in the batch, which the dispatcher keeps alive until this function returns.
            done.get();
            batches->fetch_add(1);
            release();
        };
        // every request carries one batch item, so "max requests per batch" == the model's max batch size
        // a worker stays with its merged batch until the results are scattered, and gathering 32 single-image requests
        // into the pinned batch is ~2 ms of memcpy on one core -- as long as a forward pass takes on a lane.  One worker
        // per pooled Buffers (never fewer than lanes + 1) lets every Buffers be in SOME stage: gather, H2D, forward, scatter.
        if (workers == 0)
            workers = std::max(size_t(m_Resources->MaxExecConcurrency()) + 1, size_t(m_Resources->MaxCopyConcurrency()));
        m_Dispatcher = std::make_unique<DispatcherType>(StandardBatcher<Request, standard_threads>(size_t(m_Model->GetMaxBatchSize())),
                                                        window, std::make_shared<ThreadPool>(workers),
                                                        std::make_shared<DeferredShortTaskPool>(), execute);
    }
    // one single-item request (the common case: one image per RPC)
    future_type Infer(const void* input, void* output) { return m_Dispatcher->enqueue(Request{input, output, 1}); }
    size_t BatchesExecuted() const { return m_Batches->load(); }
    void Shutdown() { m_Dispatcher->shutdown(); }

  private:
    using DispatcherType = Dispatcher<StandardBatcher<Request, standard_threads>>;
    std::shared_ptr<Model> m_Model;
    std::shared_ptr<InferenceManager> m_Resources;
    std::shared_ptr<std::atomic<size_t>> m_Batches;
    std::unique_ptr<DispatcherType> m_Dispatcher;
};

class InferBench {
  public:
    InferBench(std::shared_ptr<InferenceManager>);
    virtual ~InferBench();

    using ModelsList = std::vector<std::shared_ptr<Model>>;
    using Results = std::map<InferBenchKey, double>;

    std::unique_ptr<Results> Run(const std::shared_ptr<Model> model, uint32_t batch_size, double seconds = 5.0);
    std::unique_ptr<Results> Run(const ModelsList& models, uint32_t batch_size, double seconds = 5.0);
    // extension: stop after exactly `max_batches` requests (0 = time-bound only); per-request latencies
    // (Infer() call -> future ready) are appended to *latencies_s when non-null
    std::unique_ptr<Results> Run(const ModelsList& models, uint32_t batch_size, double seconds, size_t max_batches,
                                 std::vector<double>* latencies_s);
    // ... and the completion time of every request (seconds since the loop started, same order as the latencies): lets a
    // caller rate a window in the MIDDLE of one continuous closed loop, free of the pipeline's fill and drain
    std::unique_ptr<Results> Run(const ModelsList& models, uint32_t batch_size, double seconds, size_t max_batches,
                                 std::vector<double>* latencies_s, std::vector<double>* completions_s);

  protected:
    InferenceManager& InferResources() { return *m_Resources; }

  private:
    std::shared_ptr<InferenceManager> m_Resources;
};

// ------------------------------------------------------------------------------------------------
// v2 workspaces (workspace.h:29-106, workspace.cc:21-164)
// ------------------------------------------------------------------------------------------------
class StaticSingleModelGraphWorkspace {
  public:
    explicit StaticSingleModelGraphWorkspace(std::shared_ptr<Model>);
    virtual ~StaticSingleModelGraphWorkspace();
    DELETE_COPYABILITY(StaticSingleModelGraphWorkspace);
    DELETE_MOVEABILITY(StaticSingleModelGraphWorkspace);

    void enqueue();  // cudaGraphLaunch of the captured forward pass
    void* binding(std::uint32_t binding_id);
    std::size_t binding_bytes(std::uint32_t binding_id) const;
    cudaStream_t stream() { return m_Stream; }
    std::size_t batch_size();
    std::string name() const { return m_Name; }
    const Model& model() const { return *m_Model; }

  private:
    std::shared_ptr<Model> m_Model;
    std::shared_ptr<IExecutionContext> m_Context;
    std::vector<void*> m_Bindings;
    std::vector<size_t> m_BindingBytes;
    void* m_DeviceMemory;
    cudaStream_t m_Stream;
    void* m_Graph;          // cudaGraph_t
    void* m_GraphExecutor;  // cudaGraphExec_t
    std::string m_Name;
};

class BenchmarkWorkspace : public StaticSingleModelGraphWorkspace {
  public:
    explicit BenchmarkWorkspace(std::shared_ptr<Model>);
    ~BenchmarkWorkspace() override;
    void* host_binding(std::uint32_t binding_id);
    void async_h2d();
    void async_d2h();

  private:
    std::vector<void*> m_HostBindings;
};

class TimedBenchmarkWorkspace : private BenchmarkWorkspace {
  public:
    explicit TimedBenchmarkWorkspace(std::shared_ptr<Model>);
    ~TimedBenchmarkWorkspace() override;
    void enqueue_pipeline();
    float get_compute_time_ms();
    float get_h2d_time_ms();
    float get_d2h_time_ms();
    using BenchmarkWorkspace::binding;
    using BenchmarkWorkspace::host_binding;
    using BenchmarkWorkspace::stream;

  private:
    cudaEvent_t m_Start, m_CompleteAsyncH2D, m_CompleteCompute, m_CompleteAsyncD2H;
};

}  // namespace TensorRT
}  // namespace trtlab
