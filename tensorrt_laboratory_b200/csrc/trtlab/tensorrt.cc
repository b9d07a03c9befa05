// Implementation of the trtlab::TensorRT host surface on top of the b200infer C ABI.
// Each method cites the reference body it re-states (paths under /root/reference).
#define B2_WITH_CUDA_RUNTIME 1
#include "trtlab/tensorrt/tensorrt.h"

#include <cuda_runtime.h>
#include <sched.h>

#include <algorithm>
#include <fstream>
#include <sstream>

namespace trtlab {
namespace TensorRT {

#define TRT_CHECK_CUDA(expr)                                                                        \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) TRTLAB_LOG_FATAL << #expr << " failed: " << cudaGetErrorString(_e);  \
    } while (0)

#define TRT_CHECK_B2(expr)                                                          \
    do {                                                                            \
        int _rc = (expr);                                                           \
        if (_rc != 0) TRTLAB_LOG_FATAL << #expr << " failed: " << b2_last_error();  \
    } while (0)

// ---- memory tags ---------------------------------------------------------------------------------
// cuda_malloc_host / cuda_malloc raw allocators: std::bad_alloc on failure
// (trtlab/cuda/include/trtlab/cuda/memory/cuda_allocators.h:78-109)
void* CudaPinnedHostMemory::Allocate(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        throw std::bad_alloc();
    }
    return p;
}
void CudaPinnedHostMemory::Free(void* ptr) {
    if (ptr) cudaFreeHost(ptr);
}
void* CudaDeviceMemory::Allocate(size_t bytes) {
    void* p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) {
        cudaGetLastError();
        throw std::bad_alloc();
    }
    return p;
}
void CudaDeviceMemory::Free(void* ptr) {
    if (ptr) cudaFree(ptr);
}

// ---- Model ------------------------------------------------------------------------------------------
size_t dtype_size(int dtype) {  // utils.cc:36-50
    switch (dtype) {
        case B2_DT_FLOAT: return 4;
        case B2_DT_HALF: return 2;
        case B2_DT_INT8: return 1;
        case B2_DT_INT32: return 4;
        case B2_DT_UINT8: return 1;
    }
    TRTLAB_LOG_FATAL << "unknown binding dtype " << dtype;
    return 0;
}

Model::Model(b2_engine* engine, std::shared_ptr<Runtime> runtime) : m_Engine(engine), m_Runtime(std::move(runtime)) {
    if (!engine) throw std::runtime_error("Model: null engine");  // common.h:66-69 convention
    m_Name = b2_engine_name(engine);
    const int n = b2_engine_nb_bindings(engine);
    for (int i = 0; i < n; ++i) {  // model.cc:76-116
        TensorBindingInfo b;
        b.name = b2_engine_binding_name(engine, i);
        b.isInput = b2_engine_binding_is_input(engine, i) != 0;
        b.dtype = b2_engine_binding_dtype(engine, i);
        b.dtypeSize = dtype_size(b.dtype);
        int32_t dims[8];
        int nd = 0;
        TRT_CHECK_B2(b2_engine_binding_dims(engine, i, dims, &nd));
        b.elementsPerBatchItem = 1;
        for (int d = 0; d < nd; ++d) {
            b.dims.push_back(dims[d]);
            b.elementsPerBatchItem *= size_t(dims[d]);
        }
        b.bytesPerBatchItem = b.elementsPerBatchItem * b.dtypeSize;
        (b.isInput ? m_Inputs : m_Outputs).push_back(uint32_t(i));
        m_Bindings.push_back(std::move(b));
    }
}

Model::~Model() { b2_engine_destroy(m_Engine); }

int Model::GetMaxBatchSize() const { return b2_engine_max_batch(m_Engine); }

const Model::TensorBindingInfo& Model::GetBinding(uint32_t id) const {
    TRTLAB_CHECK_OP(id, <, m_Bindings.size()) << "invalid binding id";
    return m_Bindings[id];
}
uint32_t Model::BindingId(const std::string& name) const {
    for (size_t i = 0; i < m_Bindings.size(); ++i)
        if (m_Bindings[i].name == name) return uint32_t(i);
    TRTLAB_LOG_FATAL << "no binding named " << name << " in model " << m_Name;
    return 0;
}
const Model::TensorBindingInfo& Model::GetBinding(const std::string& name) const { return m_Bindings[BindingId(name)]; }

size_t Model::GetBindingMemorySize() const {
    size_t total = 0;
    for (const auto& b : m_Bindings) total += b.bytesPerBatchItem * size_t(GetMaxBatchSize());
    return total;
}
size_t Model::GetActivationsMemorySize() const { return b2_engine_device_memory_size(m_Engine); }
size_t Model::GetWeightsMemorySize() const { return b2_engine_weights_size(m_Engine); }

std::shared_ptr<IExecutionContext> Model::CreateExecutionContext() const {
    b2_context* c = nullptr;
    if (b2_context_create(m_Engine, &c) != 0) throw std::runtime_error(std::string("CreateExecutionContext: ") + b2_last_error());
    return std::make_shared<IExecutionContext>(c);
}

std::string Model::binding_info(std::uint32_t id) const {
    const auto& b = GetBinding(id);
    std::ostringstream os;
    os << "[" << id << "] " << b.name << (b.isInput ? " (input)" : " (output)") << " dtype=" << b.dtype << " dims=(";
    for (size_t d = 0; d < b.dims.size(); ++d) os << (d ? "," : "") << b.dims[d];
    os << ") bytes/item=" << b.bytesPerBatchItem;
    return os.str();
}
std::string Model::bindings_info() const {
    std::ostringstream os;
    for (uint32_t i = 0; i < GetBindingsCount(); ++i) os << binding_info(i) << "\n";
    return os.str();
}

// ---- Runtime -----------------------------------------------------------------------------------------
Runtime::Runtime() : m_Runtime(nullptr) {  // runtime.cc:47-50,124-127
    TRT_CHECK_B2(b2_runtime_create(&m_Runtime));
    TRT_CHECK_B2(b2_runtime_set_allocator(m_Runtime, &Runtime::AllocThunk, &Runtime::FreeThunk, this));
}
Runtime::~Runtime() { b2_runtime_destroy(m_Runtime); }

void* Runtime::AllocThunk(void* user, uint64_t size, uint64_t alignment, uint32_t flags) {
    auto* self = static_cast<Runtime*>(user);
    void* p = self->AllocateDevice(size, alignment, flags);
    if (p) self->m_Weights.push_back({p, size_t(size)});  // allocator.cc:38-53 records weight pointers
    return p;
}
void Runtime::FreeThunk(void* user, void* ptr) { static_cast<Runtime*>(user)->FreeDevice(ptr); }

std::vector<char> Runtime::ReadEngineFile(const std::string& path) const {  // runtime.cc:81-95
    std::ifstream file(path, std::ios::binary | std::ios::ate);
    if (!file.good()) throw std::runtime_error("Unable to open engine file: " + path);
    const std::streamsize size = file.tellg();
    file.seekg(0, std::ios::beg);
    std::vector<char> buffer(static_cast<size_t>(size));
    if (size > 0 && !file.read(buffer.data(), size)) throw std::runtime_error("Unable to read engine file: " + path);
    return buffer;
}

std::shared_ptr<Model> Runtime::DeserializeEngine(const std::string& plan_file) {  // runtime.cc:62-67
    auto buffer = ReadEngineFile(plan_file);
    return DeserializeEngine(buffer.data(), buffer.size());
}

std::shared_ptr<Model> Runtime::DeserializeEngine(const void* data, size_t size) {  // runtime.cc:134-143
    b2_engine* engine = nullptr;
    if (b2_engine_deserialize(m_Runtime, data, size, &engine) != 0)
        throw std::runtime_error(std::string("DeserializeEngine failed: ") + b2_last_error());
    return std::make_shared<Model>(engine, shared_from_this());
}

void* StandardRuntime::AllocateDevice(uint64_t size, uint64_t, uint32_t) {  // allocator.cc:61-70
    void* p = nullptr;
    if (cudaMalloc(&p, size) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void StandardRuntime::FreeDevice(void* ptr) { cudaFree(ptr); }

void* ManagedRuntime::AllocateDevice(uint64_t size, uint64_t, uint32_t) {  // allocator.cc:72-77
    void* p = nullptr;
    if (cudaMallocManaged(&p, size) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    int dev = 0;
    cudaGetDevice(&dev);
    cudaMemAdvise(p, size, cudaMemAdviseSetReadMostly, dev);
    cudaGetLastError();
    return p;
}
void ManagedRuntime::FreeDevice(void* ptr) { cudaFree(ptr); }

// ---- Buffers / Bindings --------------------------------------------------------------------------------
Buffers::Buffers() {  // buffers.cc:42-46 (blocking stream; the reference notes NonBlocking "breaks")
    TRT_CHECK_CUDA(cudaStreamCreate(&m_Stream));
}
Buffers::~Buffers() {  // buffers.cc:48-53
    cudaStreamSynchronize(m_Stream);
    cudaStreamDestroy(m_Stream);
}

auto Buffers::CreateBindings(const std::shared_ptr<Model>& model) -> std::shared_ptr<Bindings> {  // buffers.cc:55-60
    auto self = m_Lease.lock();  // the pooled lease when we came from InferenceManager::GetBuffers()
    if (!self) self = shared_from_this();
    auto bindings = std::shared_ptr<Bindings>(new Bindings(model, self));
    ConfigureBindings(model, bindings);
    return bindings;
}

void Buffers::ConfigureBindings(const std::shared_ptr<Model>& model, std::shared_ptr<Bindings> bindings) {  // buffers.cc:62-73
    for (uint32_t i = 0; i < model->GetBindingsCount(); i++) {
        const size_t binding_size = model->GetBinding(i).bytesPerBatchItem * size_t(model->GetMaxBatchSize());
        bindings->SetHostAddress(int(i), AllocateHost(binding_size));
        bindings->SetDeviceAddress(int(i), AllocateDevice(binding_size));
    }
}

void Buffers::Synchronize() { TRT_CHECK_CUDA(cudaStreamSynchronize(m_Stream)); }  // buffers.cc:75-78

Bindings::Bindings(const std::shared_ptr<Model> model, const std::shared_ptr<Buffers> buffers)
    : m_Model(model), m_Buffers(buffers), m_BatchSize(0), m_ActivationsAddress(nullptr) {  // bindings.cc:55-66
    const auto count = model->GetBindingsCount();
    m_HostAddresses.assign(count, nullptr);
    m_DeviceAddresses.assign(count, nullptr);
}
Bindings::~Bindings() {}

void Bindings::SetHostAddress(int binding_id, void* addr) {
    TRTLAB_CHECK_OP(size_t(binding_id), <, m_HostAddresses.size());
    m_HostAddresses[binding_id] = addr;
}
void Bindings::SetDeviceAddress(int binding_id, void* addr) {
    TRTLAB_CHECK_OP(size_t(binding_id), <, m_DeviceAddresses.size());
    m_DeviceAddresses[binding_id] = addr;
}
void* Bindings::HostAddress(uint32_t binding_id) {
    TRTLAB_CHECK_OP(binding_id, <, m_HostAddresses.size());
    return m_HostAddresses[binding_id];
}
void* Bindings::DeviceAddress(uint32_t binding_id) {
    TRTLAB_CHECK_OP(binding_id, <, m_DeviceAddresses.size());
    return m_DeviceAddresses[binding_id];
}
void** Bindings::DeviceAddresses() { return (void**)m_DeviceAddresses.data(); }

void Bindings::CopyToDevice(uint32_t id) {  // bindings.cc:121-126
    if (InferenceManager::ZeroCopyInput() && m_Model->GetBinding(id).isInput) {
        // the pinned host buffer is mapped into the device's address space: the forward pass's first kernel (the input
        // cast) reads it over PCIe itself -- the host->device transfer still happens inside the request, without the
        // copy engine and without the HBM round trip of a staged copy
        if (!m_StagedDevice.count(id)) m_StagedDevice[id] = m_DeviceAddresses[id];
        m_DeviceAddresses[id] = HostAddress(id);
        return;
    }
    CopyToDevice(id, HostAddress(id), BindingSize(id));
}
void Bindings::CopyToDevice(const std::vector<uint32_t>& ids) {
    for (auto id : ids) CopyToDevice(id);
}
void Bindings::CopyToDevice(uint32_t id, void* src, size_t bytes) {  // bindings.cc:136-141
    TRT_CHECK_CUDA(cudaMemcpyAsync(DeviceAddress(id), src, bytes, cudaMemcpyHostToDevice, Stream()));
}
void Bindings::CopyFromDevice(uint32_t id) { CopyFromDevice(id, HostAddress(id), BindingSize(id)); }  // bindings.cc:143-148
void Bindings::CopyFromDevice(const std::vector<uint32_t>& ids) {
    for (auto id : ids) CopyFromDevice(id);
}
void Bindings::CopyFromDevice(uint32_t id, void* dst, size_t bytes) {  // bindings.cc:158-163
    TRT_CHECK_CUDA(cudaMemcpyAsync(dst, DeviceAddress(id), bytes, cudaMemcpyDeviceToHost, Stream()));
}
void Bindings::SetBatchSize(uint32_t batch_size) {  // bindings.cc:165-169
    TRTLAB_CHECK_OP(batch_size, <=, uint32_t(m_Model->GetMaxBatchSize()));
    m_BatchSize = batch_size;
}
size_t Bindings::BindingSize(uint32_t binding_id) const {  // bindings.cc:171-175
    return m_Model->GetBinding(binding_id).bytesPerBatchItem * size_t(m_BatchSize ? m_BatchSize : m_Model->GetMaxBatchSize());
}

// ---- ExecutionContext ----------------------------------------------------------------------------------
ExecutionContext::Lane::Lane(size_t workspace_bytes, int index_)
    : workspace(CudaDeviceMemory::Allocate(std::max<size_t>(workspace_bytes, 1024))), bytes(std::max<size_t>(workspace_bytes, 1024)),
      index(index_), last_done(nullptr) {}
ExecutionContext::Lane::~Lane() { CudaDeviceMemory::Free(workspace); }

ExecutionContext::ExecutionContext(size_t workspace_bytes) : ExecutionContext(std::make_shared<Lane>(workspace_bytes)) {}
ExecutionContext::ExecutionContext(std::shared_ptr<Lane> lane) : m_Lane(std::move(lane)) {
    TRT_CHECK_CUDA(cudaEventCreate(&m_Start));
    TRT_CHECK_CUDA(cudaEventCreate(&m_Done));
}
ExecutionContext::~ExecutionContext() {
    {
        std::lock_guard<std::mutex> lock(m_Lane->mutex);
        if (m_Lane->last_done == m_Done) {  // nobody may wait on an event that is about to disappear
            cudaEventSynchronize(m_Done);
            m_Lane->last_done = nullptr;
        }
    }
    cudaEventDestroy(m_Start);
    cudaEventDestroy(m_Done);
}
void ExecutionContext::SetContext(std::shared_ptr<IExecutionContext> context) {
    m_Context = std::move(context);
    if (m_Context) TRT_CHECK_B2(b2_context_set_device_memory(m_Context->handle, m_Lane->workspace));
}
void ExecutionContext::Infer(const std::shared_ptr<Bindings>& bindings) {
    TRTLAB_CHECK(m_Context) << "ExecutionContext::Infer without a model context (SetContext)";
    TRTLAB_CHECK_OP(bindings->GetModel()->GetActivationsMemorySize(), <=, m_Lane->bytes);
    cudaStream_t s = bindings->Stream();
    const int batch = int(bindings->BatchSize() ? bindings->BatchSize() : bindings->GetModel()->GetMaxBatchSize());
    std::lock_guard<std::mutex> lock(m_Lane->mutex);  // enqueue order on the lane == execution order on the device
    if (m_Lane->last_done && m_Lane->last_done != m_Done) TRT_CHECK_CUDA(cudaStreamWaitEvent(s, m_Lane->last_done, 0));
    TRT_CHECK_CUDA(cudaEventRecord(m_Start, s));
    TRT_CHECK_B2(b2_context_enqueue(m_Context->handle, batch, bindings->DeviceAddresses(), s, nullptr));
    TRT_CHECK_CUDA(cudaEventRecord(m_Done, s));
    m_Lane->last_done = m_Done;
}
double ExecutionContext::Synchronize() {
    TRT_CHECK_CUDA(cudaEventSynchronize(m_Done));
    return ElapsedSeconds();
}
double ExecutionContext::ElapsedSeconds() const {
    float ms = 0.f;
    TRT_CHECK_CUDA(cudaEventElapsedTime(&ms, m_Start, m_Done));
    return double(ms) * 1e-3;
}
int ExecutionContext::Query() {
    cudaError_t e = cudaEventQuery(m_Done);
    if (e == cudaSuccess) return 0;
    if (e == cudaErrorNotReady) return 1;
    TRTLAB_LOG_FATAL << "cudaEventQuery failed: " << cudaGetErrorString(e);
    return -1;
}
void ExecutionContext::Reset() { m_Context.reset(); }  // inference_manager.cc:262-265

// ---- InferenceManager ----------------------------------------------------------------------------------
InferenceManager::InferenceManager(int max_executions, int max_buffers)  // inference_manager.cc:59-69
    : m_Device(0), m_MaxExecutions(max_executions), m_MaxBuffers(max_buffers ? max_buffers : max_executions * 2), m_HostStackSize(0),
      m_DeviceStackSize(0), m_ActivationsSize(0), m_Buffers{nullptr}, m_ExecutionContexts{nullptr}, m_ActiveRuntime{nullptr} {
    if (cudaGetDevice(&m_Device) != cudaSuccess) {
        cudaGetLastError();
        m_Device = 0;
    }
    TRTLAB_LOG_INFO << "-- Initialzing TensorRT Resource Manager --";
    TRTLAB_LOG_INFO << "Maximum Execution Concurrency: " << m_MaxExecutions;
    TRTLAB_LOG_INFO << "Maximum Copy Concurrency: " << m_MaxBuffers;
}

InferenceManager::~InferenceManager() { JoinAllThreads(); }

// Pool threads adopt the manager's device -- and, once per thread, the CPUs closest to it (reference
// trtlab/cuda/src/device_info.cc:66-85 DeviceInfo::Affinity; TRTLAB_AFFINITY=0 disables): with one replica per GPU the
// pre / cuda / post stages of replica i then run next to GPU i's PCIe root and its NUMA-local pinned Buffers.
void InferenceManager::ActivateDevice() const {
    TRT_CHECK_CUDA(cudaSetDevice(m_Device));
    static thread_local int bound_to = -1;
    if (bound_to != m_Device) {
        bound_to = m_Device;
        const char* v = getenv("TRTLAB_AFFINITY");
        if (!v || atoi(v) != 0) b2_bind_thread_to_device(m_Device, nullptr);
    }
}

bool InferenceManager::ZeroCopyInput() {
    static const bool v = [] {
        const char* e = getenv("TRTLAB_ZERO_COPY_INPUT");
        return e && atoi(e) != 0;
    }();
    return v;
}
bool InferenceManager::YieldingSync() {
    static const bool v = [] {
        const char* e = getenv("TRTLAB_SYNC");
        return e && (!strcmp(e, "yield") || !strcmp(e, "userspace") || !strcmp(e, "poll"));
    }();
    return v;
}
void InferenceManager::RecordComputeTime(double seconds) {
    m_ComputeNs.fetch_add(uint64_t(seconds * 1e9), std::memory_order_relaxed);
    m_ComputeCount.fetch_add(1, std::memory_order_relaxed);
}
double InferenceManager::MeanComputeTime(bool reset) {
    const uint64_t n = reset ? m_ComputeCount.exchange(0) : m_ComputeCount.load();
    const uint64_t ns = reset ? m_ComputeNs.exchange(0) : m_ComputeNs.load();
    return n ? double(ns) * 1e-9 / double(n) : 0.0;
}
int InferenceManager::MaxExecConcurrency() const { return m_MaxExecutions; }
int InferenceManager::MaxCopyConcurrency() const { return m_MaxBuffers; }

void InferenceManager::RegisterModel(const std::string& name, std::shared_ptr<Model> model) {
    RegisterModel(name, model, uint32_t(m_MaxExecutions));
}

void InferenceManager::RegisterModel(const std::string& name, std::shared_ptr<Model> model, uint32_t max_concurrency) {
    // inference_manager.cc:92-156
    if (m_Models.find(name) != m_Models.end()) {
        TRTLAB_LOG_ERROR << "Model naming collsion; Model with name=" << name << " is already registered.";
        return;
    }
    if (max_concurrency > uint32_t(m_MaxExecutions)) {
        TRTLAB_LOG_WARNING << "Requested concurrency (" << max_concurrency << ") exceeds max concurrency. "
                           << "Concurrency will be capped to " << m_MaxExecutions;
        max_concurrency = uint32_t(m_MaxExecutions);
    }
    // size according to the largest padding: one device alignment per binding
    const size_t bindings = model->GetBindingMemorySize() + model->GetBindingsCount() * CudaDeviceMemory::DefaultAlignment();
    const size_t activations = Align(model->GetActivationsMemorySize(), 128 * 1024);
    const size_t host = Align(bindings, 32 * 1024);
    const size_t device = Align(bindings, 128 * 1024);

    if (m_Buffers && (host > m_HostStackSize || device > m_DeviceStackSize))
        throw std::runtime_error("Required binding resources are greater than allocated capacity");
    if (m_ExecutionContexts && activations > m_ActivationsSize)
        throw std::runtime_error("Required activation workspace is greater than allocated capacity");

    m_HostStackSize = std::max(m_HostStackSize, host);
    m_DeviceStackSize = std::max(m_DeviceStackSize, device);
    m_ActivationsSize = std::max(m_ActivationsSize, activations);

    TRTLAB_LOG_INFO << "-- Registering Model: " << name << " --";
    TRTLAB_LOG_INFO << "Input/Output Tensors require " << BytesToString(model->GetBindingMemorySize());
    TRTLAB_LOG_INFO << "Execution Activations require " << BytesToString(model->GetActivationsMemorySize());
    if (auto weights = model->GetWeightsMemorySize()) TRTLAB_LOG_INFO << "Weights require " << BytesToString(weights);

    model->SetName(name);
    m_Models[name] = model;
    // Tactic selection is build-time work (the reference's engines come out of trtexec already tuned, models/setup.py:53-55):
    // time the kernels now, on a private arena, in the regime they will run in (m_MaxExecutions concurrent streams).
    // Plans that carry a tactic table skip this; B2_AUTOTUNE=0 leaves the closed-form cost model in charge.
    {
        const char* at = getenv("B2_AUTOTUNE");
        const char* all = getenv("TRTLAB_TUNE_ALL_BATCHES");
        if (!at || atoi(at) != 0) TRT_CHECK_B2(b2_engine_tune(model->engine(), at ? atoi(at) : std::max(1, std::min(m_MaxExecutions, 8)), all && atoi(all) != 0));
    }
    const uint32_t depth = uint32_t(EnqueueDepth());
    const bool per_lane = max_concurrency == uint32_t(m_MaxExecutions);
    std::vector<std::shared_ptr<Pool<IExecutionContext>>> pools;
    for (uint32_t p = 0; p < (per_lane ? max_concurrency : 1u); p++) {
        auto pool = Pool<IExecutionContext>::Create();
        for (uint32_t i = 0; i < (per_lane ? depth : max_concurrency * depth); i++) pool->Push(model->CreateExecutionContext());
        pools.push_back(pool);
    }
    m_ModelExecutionContexts[model.get()] = pools;
    if (m_ExecutionContexts) PrepareModel(model.get());  // registered after AllocateResources(): prepare right away
}

// Builds every launch plan and CUDA graph the request path will need (lane-pinned contexts x batch sizes 1..max).
void InferenceManager::PrepareModel(const Model* model) {
    auto item = m_ModelExecutionContexts.find(model);
    if (item == m_ModelExecutionContexts.end() || item->second.size() != m_Lanes.size()) return;  // shared pool: lazily, as the reference does
    const char* env = getenv("TRTLAB_PREPARE_BATCHES");  // "max" = only the max batch, "0" = none, default all (up to 64)
    const std::string mode = env ? env : "all";
    if (mode == "0") return;
    const int max_batch = model->GetMaxBatchSize();
    for (size_t lane = 0; lane < m_Lanes.size(); lane++) {
        auto& pool = item->second[lane];
        std::vector<std::shared_ptr<IExecutionContext>> held;
        const size_t n = pool->Size();
        for (size_t k = 0; k < n; k++) held.push_back(pool->PopWithoutReturn());
        for (auto& ctx : held) {
            TRT_CHECK_B2(b2_context_set_device_memory(ctx->handle, m_Lanes[lane]->workspace));
            if (!getenv("B2_NET_CTAS")) b2_context_set_option(ctx->handle, "net_ctas", std::max(1, 296 / std::max(1, m_MaxExecutions)));
            if (ZeroCopyInput() && !getenv("B2_INPUT_CTAS")) {  // a PCIe-paced cast must not hold every thread slot of the GPU
                const char* v = getenv("TRTLAB_ZERO_COPY_CTAS");
                b2_context_set_option(ctx->handle, "input_ctas", v ? atoi(v) : 74);
            }
            for (int b = (mode == "max" || max_batch > 64) ? max_batch : 1; b <= max_batch; b++)
                TRT_CHECK_B2(b2_context_prepare(ctx->handle, b, nullptr));
        }
        for (auto& ctx : held) pool->Push(std::move(ctx));
    }
}

Runtime& InferenceManager::ActiveRuntime() {
    TRTLAB_CHECK(m_ActiveRuntime) << "no active runtime";
    return *m_ActiveRuntime;
}
void InferenceManager::RegisterRuntime(const std::string& name, std::shared_ptr<Runtime> runtime) {
    TRTLAB_CHECK(m_Runtimes.find(name) == m_Runtimes.end()) << "runtime " << name << " already registered";
    m_Runtimes[name] = std::move(runtime);
}
void InferenceManager::SetActiveRuntime(const std::string& name) {
    auto search = m_Runtimes.find(name);
    TRTLAB_CHECK(search != m_Runtimes.end()) << "unknown runtime " << name;
    m_ActiveRuntime = search->second.get();
}

void InferenceManager::AllocateResources() {  // inference_manager.cc:181-205
    TRTLAB_LOG_INFO << "-- Allocating TensorRT Resources --";
    TRTLAB_LOG_INFO << "Creating " << m_MaxExecutions << " TensorRT execution tokens.";
    TRTLAB_LOG_INFO << "Creating a Pool of " << m_MaxBuffers << " Host/Device Memory Stacks";
    TRTLAB_LOG_INFO << "Each Host Stack contains " << BytesToString(m_HostStackSize);
    TRTLAB_LOG_INFO << "Each Device Stack contains " << BytesToString(m_DeviceStackSize);
    TRTLAB_LOG_INFO << "Total GPU Memory: " << BytesToString(m_MaxBuffers * m_DeviceStackSize + m_MaxExecutions * m_ActivationsSize);

    m_Buffers = Pool<Buffers>::Create();
    {
        // pinned host stacks on the GPU's NUMA node: the allocating thread sits on the GPU's CPUs while the pages are
        // first touched (cudaHostAlloc follows the thread's local policy), then gets its own mask back
        cpu_set_t before;
        const bool have = sched_getaffinity(0, sizeof before, &before) == 0;
        const char* v = getenv("TRTLAB_AFFINITY");
        int bound = 0;
        if (!v || atoi(v) != 0) b2_bind_thread_to_device(m_Device, &bound);
        for (int i = 0; i < m_MaxBuffers; i++)
            m_Buffers->Push(std::make_shared<FixedBuffers<CudaPinnedHostMemory, CudaDeviceMemory>>(m_HostStackSize, m_DeviceStackSize));
        if (have && bound > 0) sched_setaffinity(0, sizeof before, &before);
    }

    // m_MaxExecutions lanes (activation arenas == forward passes that can run at once), EnqueueDepth() tokens queued on each
    m_ExecutionContexts = Pool<ExecutionContext>::Create();
    m_Lanes.clear();
    for (int i = 0; i < m_MaxExecutions; i++) m_Lanes.push_back(std::make_shared<ExecutionContext::Lane>(m_ActivationsSize, i));
    for (int d = 0; d < EnqueueDepth(); d++)
        for (int i = 0; i < m_MaxExecutions; i++) m_ExecutionContexts->EmplacePush(new ExecutionContext(m_Lanes[size_t(i)]));
    for (const auto& item : m_Models) PrepareModel(item.second.get());
}

// Tokens per lane.  1 = the reference's behaviour (a lane is idle from the end of a forward pass until the host has
// noticed, released the token and enqueued the next request); 2 (default) keeps the next request queued on the device.
int InferenceManager::EnqueueDepth() {
    const char* v = getenv("TRTLAB_ENQUEUE_DEPTH");
    const int d = v ? atoi(v) : 2;
    return d < 1 ? 1 : (d > 4 ? 4 : d);
}

auto InferenceManager::GetModel(std::string model_name) -> std::shared_ptr<Model> {
    auto item = m_Models.find(model_name);
    TRTLAB_CHECK(item != m_Models.end()) << "Unable to find entry for model: " << model_name;
    return item->second;
}

auto InferenceManager::GetBuffers() -> std::shared_ptr<Buffers> {  // inference_manager.cc:232-239
    TRTLAB_CHECK(m_Buffers) << "Call AllocateResources() before trying to acquire a Buffers object.";
    auto lease = m_Buffers->Pop([](Buffers* ptr) {
        ptr->m_Lease.reset();
        ptr->Reset();
    });
    lease->m_Lease = lease;
    return lease;
}

auto InferenceManager::GetExecutionContext(const Model* model) -> std::shared_ptr<ExecutionContext> {
    // inference_manager.cc:254-273
    TRTLAB_CHECK(m_ExecutionContexts) << "Call AllocateResources() before trying to acquire an ExeuctionContext.";
    auto item = m_ModelExecutionContexts.find(model);
    TRTLAB_CHECK(item != m_ModelExecutionContexts.end()) << "No ExectionContext for model " << model->Name();
    // global concurrency limiter -- owns the activation scratch
    auto ctx = m_ExecutionContexts->Pop([](ExecutionContext* ptr) { ptr->Reset(); });
    // model concurrency limiter -- owns the engine-side context; it is pointed at the limiter's scratch.  Lane-pinned
    // pools: the context comes from the pool of the token's lane (never blocks: as many contexts as tokens per lane).
    auto& pools = item->second;
    auto& pool = pools.size() > 1 ? pools[size_t(ctx->LaneIndex()) % pools.size()] : pools[0];
    ctx->SetContext(pool->Pop([](IExecutionContext*) {}));
    return ctx;
}
auto InferenceManager::GetExecutionContext(const std::shared_ptr<Model>& model) -> std::shared_ptr<ExecutionContext> {
    return GetExecutionContext(model.get());
}

auto InferenceManager::AcquireThreadPool(const std::string& name) -> ThreadPool& {
    auto search = m_ThreadPools.find(name);
    TRTLAB_CHECK(search != m_ThreadPools.end()) << "no thread pool named " << name;
    return *(search->second);
}
void InferenceManager::RegisterThreadPool(const std::string& name, std::unique_ptr<ThreadPool> threads) {
    m_ThreadPools[name].swap(threads);
}
bool InferenceManager::HasThreadPool(const std::string& name) const { return m_ThreadPools.find(name) != m_ThreadPools.end(); }
void InferenceManager::JoinAllThreads() {
    // the "post" stage is fed by "cuda" which is fed by "pre": drain in that order so no stage
    // enqueues onto a pool that is already gone
    for (const char* name : {"pre", "cuda", "post"}) {
        auto it = m_ThreadPools.find(name);
        if (it != m_ThreadPools.end()) m_ThreadPools.erase(it);
    }
    m_ThreadPools.clear();
}
void InferenceManager::ForEachModel(std::function<void(const Model&)> callback) {
    for (const auto& item : m_Models) callback(*(item.second));
}

// ---- InferBench ------------------------------------------------------------------------------------------
InferBench::InferBench(std::shared_ptr<InferenceManager> resources) : m_Resources(resources) {}
InferBench::~InferBench() {}

std::unique_ptr<InferBench::Results> InferBench::Run(std::shared_ptr<Model> model, uint32_t batch_size, double seconds) {
    ModelsList models = {model};
    return Run(models, batch_size, seconds);
}
std::unique_ptr<InferBench::Results> InferBench::Run(const ModelsList& models, uint32_t batch_size, double seconds) {
    return Run(models, batch_size, seconds, 0, nullptr);
}

std::unique_ptr<InferBench::Results> InferBench::Run(const ModelsList& models, uint32_t batch_size, double seconds,
                                                     size_t max_batches, std::vector<double>* latencies_s) {
    return Run(models, batch_size, seconds, max_batches, latencies_s, nullptr);
}

std::unique_ptr<InferBench::Results> InferBench::Run(const ModelsList& models, uint32_t batch_size, double seconds,
                                                     size_t max_batches, std::vector<double>* latencies_s,
                                                     std::vector<double>* completions_s) {
    // infer_bench.cc:46-110: closed loop -- GetBuffers() blocks when all Buffers are in flight
    using clock = std::chrono::high_resolution_clock;
    size_t batch_count = 0;
    std::vector<std::shared_future<void>> futures;
    futures.reserve(max_batches ? max_batches : 1024 * 1024);
    for (const auto& model : models) TRTLAB_CHECK_OP(batch_size, <=, uint32_t(model->GetMaxBatchSize()));

    auto lat = std::make_shared<std::vector<double>>();
    auto done_at = std::make_shared<std::vector<double>>();  // completion time of every request, seconds since the loop started
    auto lat_mutex = std::make_shared<std::mutex>();
    if (latencies_s) lat->reserve(max_batches ? max_batches : 1 << 16);

    m_Resources->MeanComputeTime(true);
    auto start = clock::now();
    auto last = start + std::chrono::microseconds(static_cast<long long>(seconds * 1e6));
    while ((max_batches ? batch_count < max_batches : true) && clock::now() < last) {
        ++batch_count;
        const auto& model = models[batch_count % models.size()];
        auto buffers = InferResources().GetBuffers();  // <=== limited resource; may block
        auto bindings = buffers->CreateBindings(model);
        buffers.reset();
        bindings->SetBatchSize(batch_size);
        const auto t0 = clock::now();
        InferRunner runner(model, m_Resources);
        const bool want_lat = latencies_s != nullptr;
        const bool want_done = completions_s != nullptr;
        auto resources = m_Resources;
        futures.push_back(runner.Infer(bindings, [t0, start, lat, done_at, lat_mutex, want_lat, want_done, resources](std::shared_ptr<Bindings>& b) mutable {
            const auto now = clock::now();
            const double dt = std::chrono::duration<double>(now - t0).count();
            resources->GetMetrics().ObserveRequest(b->GetModel()->Name(), b->ComputeTime(), dt);
            if (want_lat || want_done) {
                std::lock_guard<std::mutex> l(*lat_mutex);
                if (want_lat) lat->push_back(dt);
                if (want_done) done_at->push_back(std::chrono::duration<double>(now - start).count());  // same order as `lat`
            }
            b.reset();
        }));
    }
    for (const auto& f : futures) f.wait();

    const double total_time = std::chrono::duration<double>(clock::now() - start).count();
    const double inferences = double(batch_count) * batch_size;
    auto results_ptr = std::make_unique<Results>();
    Results& results = *results_ptr;
    results[kBatchSize] = batch_size;
    results[kMaxExecConcurrency] = m_Resources->MaxExecConcurrency();
    results[kMaxCopyConcurrency] = m_Resources->MaxCopyConcurrency();
    results[kBatchesComputed] = double(batch_count);
    results[kWalltime] = total_time;
    results[kBatchesPerSecond] = batch_count / total_time;
    results[kInferencesPerSecond] = inferences / total_time;
    results[kSecondsPerBatch] = batch_count ? total_time / batch_count : 0.0;
    results[kGpuComputeTimePerBatch] = m_Resources->MeanComputeTime(true);
    results[kExecutionTimePerBatch] = batch_count ? total_time / (double(batch_count) / m_Resources->MaxExecConcurrency()) : 0.0;
    if (latencies_s && !lat->empty()) {
        std::vector<double> sorted(*lat);
        std::sort(sorted.begin(), sorted.end());
        auto pct = [&](double p) { return sorted[std::min(sorted.size() - 1, size_t(p * (sorted.size() - 1) + 0.5))]; };
        results[kLatencyP50] = pct(0.50);
        results[kLatencyP90] = pct(0.90);
        results[kLatencyP99] = pct(0.99);
        results[kLatencyMax] = sorted.back();
        latencies_s->insert(latencies_s->end(), lat->begin(), lat->end());
    }
    if (completions_s) completions_s->insert(completions_s->end(), done_at->begin(), done_at->end());
    return results_ptr;
}

// ---- v2 workspaces -----------------------------------------------------------------------------------------
StaticSingleModelGraphWorkspace::StaticSingleModelGraphWorkspace(std::shared_ptr<Model> model)
    : m_Model(std::move(model)), m_DeviceMemory(nullptr), m_Graph(nullptr), m_GraphExecutor(nullptr) {
    // workspace.cc:21-57
    std::stringstream ss;
    ss << this;
    m_Name = ss.str();
    m_Context = m_Model->CreateExecutionContext();
    for (uint32_t i = 0; i < m_Model->GetBindingsCount(); i++) {
        const size_t bytes = m_Model->binding_size_in_bytes(i);
        m_Bindings.push_back(CudaDeviceMemory::Allocate(bytes));
        m_BindingBytes.push_back(bytes);
        TRT_CHECK_CUDA(cudaMemset(m_Bindings.back(), 0, bytes));
    }
    m_DeviceMemory = CudaDeviceMemory::Allocate(std::max<size_t>(m_Model->GetActivationsMemorySize(), 1024));
    TRT_CHECK_B2(b2_context_set_device_memory(m_Context->handle, m_DeviceMemory));
    TRT_CHECK_CUDA(cudaStreamCreate(&m_Stream));
    const int batch = m_Model->GetMaxBatchSize();
    // the engine replays its own cached graph by default; here the CALLER captures, as the reference does
    TRT_CHECK_B2(b2_context_set_option(m_Context->handle, "graph", 0));
    TRT_CHECK_B2(b2_context_enqueue(m_Context->handle, batch, m_Bindings.data(), m_Stream, nullptr));  // warm up
    TRT_CHECK_CUDA(cudaStreamSynchronize(m_Stream));
    cudaGraph_t graph = nullptr;
    TRT_CHECK_CUDA(cudaStreamBeginCapture(m_Stream, cudaStreamCaptureModeRelaxed));
    TRT_CHECK_B2(b2_context_enqueue(m_Context->handle, batch, m_Bindings.data(), m_Stream, nullptr));
    TRT_CHECK_CUDA(cudaStreamEndCapture(m_Stream, &graph));
    cudaGraphExec_t exec = nullptr;
    TRT_CHECK_CUDA(cudaGraphInstantiate(&exec, graph, 0));
    m_Graph = graph;
    m_GraphExecutor = exec;
}

StaticSingleModelGraphWorkspace::~StaticSingleModelGraphWorkspace() {  // workspace.cc:59-71
    cudaStreamSynchronize(m_Stream);
    if (m_GraphExecutor) cudaGraphExecDestroy(static_cast<cudaGraphExec_t>(m_GraphExecutor));
    if (m_Graph) cudaGraphDestroy(static_cast<cudaGraph_t>(m_Graph));
    cudaStreamDestroy(m_Stream);
    m_Context.reset();
    for (void* p : m_Bindings) CudaDeviceMemory::Free(p);
    CudaDeviceMemory::Free(m_DeviceMemory);
}

void StaticSingleModelGraphWorkspace::enqueue() {  // workspace.cc:73-76
    TRT_CHECK_CUDA(cudaGraphLaunch(static_cast<cudaGraphExec_t>(m_GraphExecutor), m_Stream));
}
void* StaticSingleModelGraphWorkspace::binding(std::uint32_t binding_id) {
    TRTLAB_CHECK_OP(binding_id, <, m_Bindings.size());
    return m_Bindings[binding_id];
}
std::size_t StaticSingleModelGraphWorkspace::binding_bytes(std::uint32_t binding_id) const { return m_BindingBytes.at(binding_id); }
std::size_t StaticSingleModelGraphWorkspace::batch_size() { return size_t(m_Model->GetMaxBatchSize()); }

BenchmarkWorkspace::BenchmarkWorkspace(std::shared_ptr<Model> model) : StaticSingleModelGraphWorkspace(model) {  // workspace.cc:90-100
    for (uint32_t i = 0; i < this->model().GetBindingsCount(); i++) {
        m_HostBindings.push_back(CudaPinnedHostMemory::Allocate(binding_bytes(i)));
        memset(m_HostBindings.back(), 0, binding_bytes(i));
    }
}
BenchmarkWorkspace::~BenchmarkWorkspace() {
    cudaStreamSynchronize(stream());
    for (void* p : m_HostBindings) CudaPinnedHostMemory::Free(p);
}
void* BenchmarkWorkspace::host_binding(std::uint32_t binding_id) { return m_HostBindings.at(binding_id); }
void BenchmarkWorkspace::async_h2d() {  // workspace.cc:102-112
    for (uint32_t i = 0; i < m_HostBindings.size(); i++)
        if (model().GetBinding(i).isInput)
            TRT_CHECK_CUDA(cudaMemcpyAsync(binding(i), m_HostBindings[i], binding_bytes(i), cudaMemcpyHostToDevice, stream()));
}
void BenchmarkWorkspace::async_d2h() {  // workspace.cc:114-124
    for (uint32_t i = 0; i < m_HostBindings.size(); i++)
        if (!model().GetBinding(i).isInput)
            TRT_CHECK_CUDA(cudaMemcpyAsync(m_HostBindings[i], binding(i), binding_bytes(i), cudaMemcpyDeviceToHost, stream()));
}

TimedBenchmarkWorkspace::TimedBenchmarkWorkspace(std::shared_ptr<Model> model) : BenchmarkWorkspace(model) {  // workspace.cc:126-132
    TRT_CHECK_CUDA(cudaEventCreate(&m_Start));
    TRT_CHECK_CUDA(cudaEventCreate(&m_CompleteAsyncH2D));
    TRT_CHECK_CUDA(cudaEventCreate(&m_CompleteCompute));
    TRT_CHECK_CUDA(cudaEventCreate(&m_CompleteAsyncD2H));
}
TimedBenchmarkWorkspace::~TimedBenchmarkWorkspace() {
    cudaStreamSynchronize(stream());
    cudaEventDestroy(m_Start);
    cudaEventDestroy(m_CompleteAsyncH2D);
    cudaEventDestroy(m_CompleteCompute);
    cudaEventDestroy(m_CompleteAsyncD2H);
}
void TimedBenchmarkWorkspace::enqueue_pipeline() {  // workspace.cc:134-143
    TRT_CHECK_CUDA(cudaEventRecord(m_Start, stream()));
    async_h2d();
    TRT_CHECK_CUDA(cudaEventRecord(m_CompleteAsyncH2D, stream()));
    enqueue();
    TRT_CHECK_CUDA(cudaEventRecord(m_CompleteCompute, stream()));
    async_d2h();
    TRT_CHECK_CUDA(cudaEventRecord(m_CompleteAsyncD2H, stream()));
}
float TimedBenchmarkWorkspace::get_compute_time_ms() {
    float ms = 0.0;
    TRT_CHECK_CUDA(cudaEventElapsedTime(&ms, m_CompleteAsyncH2D, m_CompleteCompute));
    return ms;
}
float TimedBenchmarkWorkspace::get_h2d_time_ms() {
    float ms = 0.0;
    TRT_CHECK_CUDA(cudaEventElapsedTime(&ms, m_Start, m_CompleteAsyncH2D));
    return ms;
}
float TimedBenchmarkWorkspace::get_d2h_time_ms() {
    float ms = 0.0;
    TRT_CHECK_CUDA(cudaEventElapsedTime(&ms, m_CompleteCompute, m_CompleteAsyncD2H));
    return ms;
}

}  // namespace TensorRT
}  // namespace trtlab
