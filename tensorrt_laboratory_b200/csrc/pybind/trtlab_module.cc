// Python module `trtlab` -- the reference's pybind surface over the hot path (SURVEY.md 8f N2;
// trtlab/pybind/trtlab/infer.cc:83-122 PyInferenceManager, :406-545 PyInferRunner, :683-720 module definition).
// Same class / method / keyword names, so the reference's results-pinning script runs against this runtime as written:
//     models = trtlab.InferenceManager(max_exec_concurrency=2)
//     mnist  = models.register_tensorrt_engine("mnist", "mnist.plan")      # a B2ENGINE plan instead of a TensorRT one
//     models.update_resources()
//     results = [mnist.infer(Input3=x) for x in inputs];  results = [r.get() for r in results]
// (examples/30_PyTensorRT/server.py:19-31).  serve() and RemoteInferenceManager speak the TRTIS gRPC protocol, which is
// C++ over nvrpc / gRPC C++ in the reference (infer.cc:124-260, 430-642); gRPC C++ is not in this image, so both delegate to
// the grpcio restatement of that protocol in tensorrt_laboratory_b200/trtis.py (same wire format, same Python-visible API).
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cstring>
#include <future>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>

#include "trtlab/tensorrt/tensorrt.h"

namespace py = pybind11;
using namespace trtlab;
using namespace trtlab::TensorRT;

namespace {

py::dtype numpy_dtype(int b2_dtype) {  // same order as the reference's DataTypeToNumpy (infer.cc:62-81)
    switch (b2_dtype) {
        case B2_DT_FLOAT: return py::dtype::of<float>();
        case B2_DT_HALF: return py::dtype("float16");
        case B2_DT_INT8: return py::dtype::of<std::int8_t>();
        case B2_DT_INT32: return py::dtype::of<std::int32_t>();
        case B2_DT_UINT8: return py::dtype::of<std::uint8_t>();
    }
    throw std::runtime_error("unknown binding dtype");
}

py::dict binding_info(const Model& model, uint32_t id) {
    const auto& b = model.GetBinding(id);
    py::dict value;
    value["shape"] = b.dims;
    value["dtype"] = numpy_dtype(int(b.dtype));
    return value;
}

// The result dict lives in the future's shared state, whose LAST reference may be dropped by a pool thread (the caller
// discarded its InferFuture): the holder's deleter takes the GIL before touching Python reference counts.
using InferResults = std::shared_ptr<py::dict>;
using InferFuture = std::shared_future<InferResults>;
static InferResults make_results() {
    return InferResults(new py::dict(), [](py::dict* p) {
        py::gil_scoped_acquire acquire;
        delete p;
    });
}

struct PyInferRunner : public InferRunner {
    using InferRunner::InferRunner;

    // keyword = input binding name, value = numpy array [batch, ...] of the binding's dtype
    InferFuture Infer(py::kwargs kwargs) {
        const Model& model = GetModel();
        std::shared_ptr<Bindings> bindings;
        {
            // GetBuffers() BLOCKS while every Buffers is in flight, and the post stage of those requests needs the GIL
            // to build their result dicts before it releases them: waiting here with the GIL held would deadlock as soon
            // as more requests are issued than there are Buffers (`[runner.infer(...) for x in xs]`).
            py::gil_scoped_release release;
            auto buffers = Resources().GetBuffers();
            bindings = buffers->CreateBindings(GetModelSmartPtr());
        }
        long batch_size = -1;
        size_t seen = 0;
        for (auto item : kwargs) {
            const std::string key = py::cast<std::string>(item.first);
            // (Model::BindingId aborts on an unknown name, like the reference's CHECK; a Python caller gets an exception)
            bool known = false;
            for (uint32_t i = 0; i < uint32_t(model.GetBindingsCount()); ++i) known = known || model.GetBinding(i).name == key;
            if (!known) throw py::key_error(key + " is not a binding of model " + model.Name());
            const uint32_t id = model.BindingId(key);
            const auto& b = model.GetBinding(id);
            if (!b.isInput) throw py::value_error(key + " is not an input binding");
            py::array arr = py::array::ensure(item.second, py::array::c_style | py::array::forcecast);
            if (!arr) throw py::type_error(key + ": expected a numpy array");
            // a uint8 image binding takes the image bytes: casting normalised floats to uint8 would wrap them silently
            if (b.dtype == B2_DT_UINT8 && !arr.dtype().is(py::dtype::of<std::uint8_t>()))
                throw py::type_error(key + ": this binding takes uint8 images, got dtype " + py::str(arr.dtype()).cast<std::string>());
            arr = py::array::ensure(arr.attr("astype")(numpy_dtype(int(b.dtype)), py::arg("copy") = false), py::array::c_style);
            if (arr.ndim() < 1) throw py::value_error(key + ": expected a leading batch dimension");
            const long batch = long(arr.shape(0));
            if (batch < 1 || batch > long(model.GetMaxBatchSize())) throw py::value_error(key + ": batch outside [1, max_batch_size]");
            if (batch_size == -1) batch_size = batch;
            else if (batch != batch_size) throw py::value_error("input bindings disagree on the batch size");
            if (size_t(arr.nbytes()) != b.bytesPerBatchItem * size_t(batch))
                throw py::value_error(key + ": array size does not match the binding");
            std::memcpy(bindings->HostAddress(id), arr.data(), size_t(arr.nbytes()));
            ++seen;
        }
        if (seen != model.GetInputBindingIds().size()) throw py::value_error("every input binding needs a keyword argument");
        bindings->SetBatchSize(uint32_t(batch_size));
        py::gil_scoped_release release;  // the pipeline's post stage re-acquires the GIL to build the result dict
        auto fut = InferRunner::Infer(bindings, [](std::shared_ptr<Bindings>& b) -> InferResults {
            py::gil_scoped_acquire acquire;
            InferResults results = make_results();
            for (uint32_t id : b->OutputBindings()) {
                const auto& info = b->GetModel()->GetBinding(id);
                std::vector<py::ssize_t> dims;
                dims.push_back(py::ssize_t(b->BatchSize()));
                for (auto d : info.dims) dims.push_back(py::ssize_t(d));
                py::array value(numpy_dtype(int(info.dtype)), dims);
                std::memcpy(value.mutable_data(), b->HostAddress(id), b->BindingSize(id));
                (*results)[py::str(info.name)] = value;
            }
            return results;
        });
        return fut;
    }
    py::dict InputBindings() const {
        py::dict d;
        for (uint32_t id : GetModel().GetInputBindingIds()) d[py::str(GetModel().GetBinding(id).name)] = binding_info(GetModel(), id);
        return d;
    }
    py::dict OutputBindings() const {
        py::dict d;
        for (uint32_t id : GetModel().GetOutputBindingIds()) d[py::str(GetModel().GetBinding(id).name)] = binding_info(GetModel(), id);
        return d;
    }
};

class PyInferenceManager : public InferenceManager {
  public:
    PyInferenceManager(int max_executions, int max_buffers, int pre_threads, int cuda_threads, int post_threads)
        : InferenceManager(max_executions, max_buffers) {
        RegisterThreadPool("pre", std::make_unique<ThreadPool>(size_t(pre_threads)));
        RegisterThreadPool("cuda", std::make_unique<ThreadPool>(size_t(cuda_threads)));
        RegisterThreadPool("post", std::make_unique<ThreadPool>(size_t(post_threads)));
        RegisterRuntime("default", std::make_shared<StandardRuntime>());
        RegisterRuntime("unified", std::make_shared<ManagedRuntime>());
        SetActiveRuntime("default");
    }
    std::shared_ptr<PyInferRunner> RegisterModelByPath(const std::string& name, const std::string& path) {
        auto model = ActiveRuntime().DeserializeEngine(path);
        RegisterModel(name, model);
        return MakeRunner(name);
    }
    std::shared_ptr<PyInferRunner> MakeRunner(const std::string& name) {
        return std::make_shared<PyInferRunner>(GetModel(name), casted_shared_from_this<InferenceManager>());
    }
    py::dict Models() {
        py::dict out;
        ForEachModel([&](const Model& model) {
            py::dict ins, outs;
            for (uint32_t id : model.GetInputBindingIds()) ins[py::str(model.GetBinding(id).name)] = binding_info(model, id);
            for (uint32_t id : model.GetOutputBindingIds()) outs[py::str(model.GetBinding(id).name)] = binding_info(model, id);
            py::dict m;
            m["inputs"] = ins, m["outputs"] = outs, m["max_batch_size"] = model.GetMaxBatchSize();
            out[py::str(model.Name())] = m;
        });
        return out;
    }
};

}  // namespace

PYBIND11_MODULE(trtlab, m) {
    m.doc() = "trtlab Python surface (InferenceManager / InferRunner / InferFuture) on the B200-native runtime";
    py::class_<PyInferenceManager, std::shared_ptr<PyInferenceManager>>(m, "InferenceManager")
        .def(py::init<int, int, int, int, int>(), py::arg("max_exec_concurrency") = 1, py::arg("max_copy_concurrency") = 0,
             py::arg("pre_threads") = 1, py::arg("cuda_threads") = 1, py::arg("post_threads") = 3)
        .def("register_tensorrt_engine", &PyInferenceManager::RegisterModelByPath)
        .def("update_resources", [](PyInferenceManager& self) { self.AllocateResources(); })
        .def("infer_runner", &PyInferenceManager::MakeRunner)
        .def("get_models", &PyInferenceManager::Models)
        .def("metrics_text", [](PyInferenceManager& self) { return self.GetMetrics().Expose(); })
        // infer.cc:411-417: TRTIS GRPCService (Status / Health / Infer) in front of this manager; blocks like the reference's
        // server.Run() unless block=False, in which case the running server object is returned (shutdown() stops it)
        .def("serve", [](std::shared_ptr<PyInferenceManager> self, int port, bool block) {
            return py::module_::import("tensorrt_laboratory_b200.trtis").attr("serve_pybind")(self, port, block);
        }, py::arg("port") = 50052, py::arg("block") = true);
    // infer.cc:547-642: client of a served manager; get_models() / infer_runner(name).infer(**inputs).get()
    m.def("RemoteInferenceManager", [](const std::string& hostname) {
        return py::module_::import("tensorrt_laboratory_b200.trtis").attr("RemoteInferenceManager")(hostname);
    }, py::arg("hostname") = "localhost:50052");
    py::class_<PyInferRunner, std::shared_ptr<PyInferRunner>>(m, "InferRunner")
        .def("infer", &PyInferRunner::Infer)
        .def("input_bindings", &PyInferRunner::InputBindings)
        .def("output_bindings", &PyInferRunner::OutputBindings)
        .def("max_batch_size", &PyInferRunner::MaxBatchSize);
    py::class_<InferFuture, std::shared_ptr<InferFuture>>(m, "InferFuture")
        .def("wait", &InferFuture::wait, py::call_guard<py::gil_scoped_release>())
        .def("get", [](InferFuture& f) {
            {
                py::gil_scoped_release release;
                f.wait();
            }
            return py::dict(*f.get());
        });
}
