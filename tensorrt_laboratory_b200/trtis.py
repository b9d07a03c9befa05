"""TRTIS (TensorRT Inference Server) gRPC protocol front end + remote client -- SURVEY.md 8f N2.

The reference's Python module can ``serve()`` an InferenceManager behind the TRTIS ``GRPCService`` (Status / Health /
Infer; trtlab/pybind/trtlab/infer.cc:124-260) and reach a served one through ``RemoteInferenceManager`` (infer.cc:430-642).
Both are C++ over nvrpc / gRPC C++ there; neither exists in this image, so -- like rpc.py -- the same roles are restated
over grpcio, with messages built at run time from descriptors that carry the reference's package name
(``nvidia.inferenceserver``), message names and FIELD NUMBERS (examples/11_Protos/inference/{nvidia_inference,api,
request_status,server_status,model_config}.proto), i.e. the wire format a TRTIS client or server of that generation
exchanges.  Only the fields the reference's own service fills or reads are declared; unknown fields are preserved by
protobuf.

Server side:   build_trtis_server(backend, address)            (StatusContext, HealthContext, InferContext)
               backend = CapiBackend(capi.InferenceManager) | PybindBackend(trtlab.InferenceManager) | anything with
               ``models()`` and ``infer(model, {input name: array}) -> ({output name: array}, compute seconds)``
Client side:   RemoteInferenceManager(hostname).get_models() / .infer_runner(name).infer(**inputs).get()
"""
from __future__ import annotations

import threading
import time
from concurrent import futures
from typing import Dict, List, Optional, Tuple

import grpc
import numpy as np
from google.protobuf import descriptor_pb2, descriptor_pool, message_factory

from . import rpc

_F = descriptor_pb2.FieldDescriptorProto
_PKG = "nvidia.inferenceserver"
SERVICE = _PKG + ".GRPCService"

# model_config.proto DataType
TYPE_UINT8, TYPE_FP16, TYPE_FP32, TYPE_INT8, TYPE_INT32 = 2, 10, 11, 6, 8
_NP_OF = {TYPE_FP32: np.float32, TYPE_FP16: np.float16, TYPE_INT8: np.int8, TYPE_INT32: np.int32, TYPE_UINT8: np.uint8}
_TYPE_OF = {np.dtype(v): k for k, v in _NP_OF.items()}
# request_status.proto RequestStatusCode
SUCCESS, UNKNOWN, INTERNAL, NOT_FOUND, INVALID_ARG, UNAVAILABLE = 1, 2, 3, 4, 5, 6
SERVER_READY, MODEL_READY = 2, 1


def _build_pool():
    pool = descriptor_pool.DescriptorPool()
    fd = descriptor_pb2.FileDescriptorProto(name="b2/trtis.proto", package=_PKG, syntax="proto3")
    f = rpc._field
    T = "." + _PKG + "."
    # request_status.proto
    e = fd.enum_type.add(name="RequestStatusCode")
    for i, n in enumerate(["INVALID", "SUCCESS", "UNKNOWN", "INTERNAL", "NOT_FOUND", "INVALID_ARG", "UNAVAILABLE", "UNSUPPORTED"]):
        e.value.add(name=n, number=i)
    m = fd.message_type.add(name="RequestStatus")
    f(m, "code", 1, _F.TYPE_ENUM, type_name=T + "RequestStatusCode"), f(m, "msg", 2, _F.TYPE_STRING)
    f(m, "server_id", 3, _F.TYPE_STRING), f(m, "request_id", 4, _F.TYPE_UINT64)
    # api.proto
    m = fd.message_type.add(name="InferRequestHeader")
    n = m.nested_type.add(name="Input")
    f(n, "name", 1, _F.TYPE_STRING), f(n, "byte_size", 2, _F.TYPE_UINT64)
    n = m.nested_type.add(name="Output")
    c = n.nested_type.add(name="Class")
    f(c, "count", 1, _F.TYPE_UINT32)
    f(n, "name", 1, _F.TYPE_STRING), f(n, "byte_size", 2, _F.TYPE_UINT64)
    f(n, "cls", 3, _F.TYPE_MESSAGE, type_name=T + "InferRequestHeader.Output.Class")
    f(m, "batch_size", 1, _F.TYPE_UINT32)
    f(m, "input", 2, _F.TYPE_MESSAGE, _F.LABEL_REPEATED, T + "InferRequestHeader.Input")
    f(m, "output", 3, _F.TYPE_MESSAGE, _F.LABEL_REPEATED, T + "InferRequestHeader.Output")
    m = fd.message_type.add(name="InferResponseHeader")
    n = m.nested_type.add(name="Output")
    r = n.nested_type.add(name="Raw")
    f(r, "byte_size", 1, _F.TYPE_UINT64)
    f(n, "name", 1, _F.TYPE_STRING), f(n, "raw", 2, _F.TYPE_MESSAGE, type_name=T + "InferResponseHeader.Output.Raw")
    f(m, "model_name", 1, _F.TYPE_STRING), f(m, "model_version", 2, _F.TYPE_UINT32), f(m, "batch_size", 3, _F.TYPE_UINT32)
    f(m, "output", 4, _F.TYPE_MESSAGE, _F.LABEL_REPEATED, T + "InferResponseHeader.Output")
    # model_config.proto (the part Status carries)
    e = fd.enum_type.add(name="DataType")
    for i, n in enumerate(["TYPE_INVALID", "TYPE_BOOL", "TYPE_UINT8", "TYPE_UINT16", "TYPE_UINT32", "TYPE_UINT64", "TYPE_INT8", "TYPE_INT16",
                           "TYPE_INT32", "TYPE_INT64", "TYPE_FP16", "TYPE_FP32", "TYPE_FP64"]):
        e.value.add(name=n, number=i)
    m = fd.message_type.add(name="ModelInput")
    e = m.enum_type.add(name="Format")
    for i, n in enumerate(["FORMAT_NONE", "FORMAT_NHWC", "FORMAT_NCHW"]):
        e.value.add(name=n, number=i)
    f(m, "name", 1, _F.TYPE_STRING), f(m, "data_type", 2, _F.TYPE_ENUM, type_name=T + "DataType")
    f(m, "format", 3, _F.TYPE_ENUM, type_name=T + "ModelInput.Format"), f(m, "dims", 4, _F.TYPE_INT64, _F.LABEL_REPEATED)
    m = fd.message_type.add(name="ModelOutput")
    f(m, "name", 1, _F.TYPE_STRING), f(m, "data_type", 2, _F.TYPE_ENUM, type_name=T + "DataType")
    f(m, "dims", 3, _F.TYPE_INT64, _F.LABEL_REPEATED), f(m, "label_filename", 4, _F.TYPE_STRING)
    m = fd.message_type.add(name="ModelConfig")
    f(m, "name", 1, _F.TYPE_STRING), f(m, "platform", 2, _F.TYPE_STRING), f(m, "max_batch_size", 4, _F.TYPE_INT32)
    f(m, "input", 5, _F.TYPE_MESSAGE, _F.LABEL_REPEATED, T + "ModelInput")
    f(m, "output", 6, _F.TYPE_MESSAGE, _F.LABEL_REPEATED, T + "ModelOutput")
    # server_status.proto
    e = fd.enum_type.add(name="ModelReadyState")
    for i, n in enumerate(["MODEL_UNKNOWN", "MODEL_READY", "MODEL_UNAVAILABLE", "MODEL_LOADING", "MODEL_UNLOADING"]):
        e.value.add(name=n, number=i)
    e = fd.enum_type.add(name="ServerReadyState")
    for n, i in (("SERVER_INVALID", 0), ("SERVER_INITIALIZING", 1), ("SERVER_READY", 2), ("SERVER_EXITING", 3), ("SERVER_FAILED_TO_INITIALIZE", 10)):
        e.value.add(name=n, number=i)
    m = fd.message_type.add(name="ModelVersionStatus")
    f(m, "ready_state", 1, _F.TYPE_ENUM, type_name=T + "ModelReadyState")
    m = fd.message_type.add(name="ModelStatus")
    ent = m.nested_type.add(name="VersionStatusEntry")
    ent.options.map_entry = True
    f(ent, "key", 1, _F.TYPE_UINT32), f(ent, "value", 2, _F.TYPE_MESSAGE, type_name=T + "ModelVersionStatus")
    f(m, "config", 1, _F.TYPE_MESSAGE, type_name=T + "ModelConfig")
    f(m, "version_status", 2, _F.TYPE_MESSAGE, _F.LABEL_REPEATED, T + "ModelStatus.VersionStatusEntry")
    m = fd.message_type.add(name="ServerStatus")
    ent = m.nested_type.add(name="ModelStatusEntry")
    ent.options.map_entry = True
    f(ent, "key", 1, _F.TYPE_STRING), f(ent, "value", 2, _F.TYPE_MESSAGE, type_name=T + "ModelStatus")
    f(m, "id", 1, _F.TYPE_STRING), f(m, "version", 2, _F.TYPE_STRING), f(m, "uptime_ns", 3, _F.TYPE_UINT64)
    f(m, "model_status", 4, _F.TYPE_MESSAGE, _F.LABEL_REPEATED, T + "ServerStatus.ModelStatusEntry")
    f(m, "ready_state", 7, _F.TYPE_ENUM, type_name=T + "ServerReadyState")
    # nvidia_inference.proto
    m = fd.message_type.add(name="StatusRequest")
    f(m, "model_name", 1, _F.TYPE_STRING)
    m = fd.message_type.add(name="StatusResponse")
    f(m, "request_status", 1, _F.TYPE_MESSAGE, type_name=T + "RequestStatus"), f(m, "server_status", 2, _F.TYPE_MESSAGE, type_name=T + "ServerStatus")
    m = fd.message_type.add(name="HealthRequest")
    f(m, "mode", 1, _F.TYPE_STRING)
    m = fd.message_type.add(name="HealthResponse")
    f(m, "request_status", 1, _F.TYPE_MESSAGE, type_name=T + "RequestStatus"), f(m, "health", 2, _F.TYPE_BOOL)
    m = fd.message_type.add(name="InferRequest")
    f(m, "model_name", 1, _F.TYPE_STRING), f(m, "version", 2, _F.TYPE_STRING)
    f(m, "meta_data", 3, _F.TYPE_MESSAGE, type_name=T + "InferRequestHeader"), f(m, "raw_input", 4, _F.TYPE_BYTES, _F.LABEL_REPEATED)
    f(m, "batch_id", 100, _F.TYPE_UINT64), f(m, "batch_size", 101, _F.TYPE_UINT32), f(m, "sysv_offset", 102, _F.TYPE_UINT64)
    m = fd.message_type.add(name="InferResponse")
    f(m, "request_status", 1, _F.TYPE_MESSAGE, type_name=T + "RequestStatus")
    f(m, "meta_data", 2, _F.TYPE_MESSAGE, type_name=T + "InferResponseHeader"), f(m, "raw_output", 3, _F.TYPE_BYTES, _F.LABEL_REPEATED)
    f(m, "batch_id", 100, _F.TYPE_UINT64), f(m, "compute_time", 101, _F.TYPE_FLOAT), f(m, "request_time", 102, _F.TYPE_FLOAT)
    pool.Add(fd)
    return pool


_POOL = _build_pool()


def message(name: str):
    """Message class of the TRTIS package, e.g. ``message("InferRequest")``."""
    return message_factory.GetMessageClass(_POOL.FindMessageTypeByName(_PKG + "." + name))


# ------------------------------------------------------------------------------------------------
# backends: what the service needs from an inference manager
# ------------------------------------------------------------------------------------------------
class CapiBackend:
    """capi.InferenceManager (ctypes handle on the C++ InferenceManager / InferRunner pipeline)."""

    def __init__(self, manager):
        self.manager = manager

    def models(self) -> Dict[str, dict]:
        out = {}
        for name, meta in self.manager.models.items():
            out[name] = dict(max_batch=meta.max_batch,
                             inputs={b["name"]: (tuple(b["shape"]), np.dtype(b["np_dtype"])) for b in meta.bindings if b["is_input"]},
                             outputs={b["name"]: (tuple(b["shape"]), np.dtype(np.float32)) for b in meta.bindings if not b["is_input"]})
        return out

    def infer(self, model: str, inputs: Dict[str, np.ndarray]) -> Tuple[Dict[str, np.ndarray], float]:
        meta = self.manager.models[model]
        (x,) = inputs.values()
        y, sec = self.manager.infer_timed(model, x)
        out_name = [b["name"] for b in meta.bindings if not b["is_input"]][0]
        return {out_name: y}, sec


class PybindBackend:
    """The pybind11 ``trtlab.InferenceManager`` (csrc/pybind/trtlab_module.cc): ``serve()`` hands itself to this."""

    def __init__(self, manager):
        self.manager = manager
        self._runners: Dict[str, object] = {}

    def models(self) -> Dict[str, dict]:
        return {name: dict(max_batch=m["max_batch_size"],
                           inputs={k: (tuple(v["shape"]), np.dtype(v["dtype"])) for k, v in m["inputs"].items()},
                           outputs={k: (tuple(v["shape"]), np.dtype(v["dtype"])) for k, v in m["outputs"].items()})
                for name, m in self.manager.get_models().items()}

    def infer(self, model: str, inputs: Dict[str, np.ndarray]):
        runner = self._runners.get(model)
        if runner is None:
            runner = self._runners.setdefault(model, self.manager.infer_runner(model))
        t0 = time.perf_counter()
        res = runner.infer(**inputs).get()
        return {k: np.asarray(v) for k, v in res.items()}, time.perf_counter() - t0


# ------------------------------------------------------------------------------------------------
# server side (infer.cc:131-212)
# ------------------------------------------------------------------------------------------------
class TrtisResources(rpc.Resources):
    def __init__(self, backend, server_id: str = "b200-trtlab"):
        self.backend, self.server_id = backend, server_id
        self.started = time.time()
        self.request_id = 0
        self._lock = threading.Lock()

    def next_id(self) -> int:
        with self._lock:
            self.request_id += 1
            return self.request_id


def _ok(status, res: TrtisResources):
    status.code, status.server_id, status.request_id = SUCCESS, res.server_id, res.next_id()


def _fail(status, res: TrtisResources, code: int, msg: str):
    status.code, status.msg, status.server_id, status.request_id = code, msg, res.server_id, res.next_id()


class StatusContext(rpc.Context):
    """GRPCService/Status: SERVER_READY and one ModelConfig per registered model -- name, max batch size, every input and
    output binding with its dims WITHOUT the batch dimension (infer.cc:131-175); ``model_name`` narrows it to one model."""

    def execute_rpc(self, request, response):
        res: TrtisResources = self.get_resources()
        models = res.backend.models()
        if request.model_name and request.model_name not in models:
            return _fail(response.request_status, res, NOT_FOUND, f"no model named '{request.model_name}'")
        ss = response.server_status
        ss.id, ss.version, ss.ready_state = res.server_id, "b200-trtlab 0.2 (TRTIS GRPCService v1 protocol)", SERVER_READY
        ss.uptime_ns = int((time.time() - res.started) * 1e9)
        for name, meta in models.items():
            if request.model_name and name != request.model_name:
                continue
            ms = ss.model_status[name]
            ms.version_status[1].ready_state = MODEL_READY
            cfg = ms.config
            cfg.name, cfg.platform, cfg.max_batch_size = name, "b200_plan", int(meta["max_batch"])
            for bname, (shape, dt) in meta["inputs"].items():
                i = cfg.input.add()
                i.name, i.data_type = bname, _TYPE_OF[np.dtype(dt)]
                i.dims.extend(int(d) for d in shape)
            for bname, (shape, dt) in meta["outputs"].items():
                o = cfg.output.add()
                o.name, o.data_type = bname, _TYPE_OF[np.dtype(dt)]
                o.dims.extend(int(d) for d in shape)
        _ok(response.request_status, res)


class HealthContext(rpc.Context):
    def execute_rpc(self, request, response):
        res: TrtisResources = self.get_resources()
        if request.mode not in ("", "live", "ready"):
            return _fail(response.request_status, res, INVALID_ARG, f"unknown health mode '{request.mode}'")
        response.health = True
        _ok(response.request_status, res)


class InferContext(rpc.Context):
    """GRPCService/Infer (infer.cc:177-212): ``raw_input[i]`` is the tensor of ``meta_data.input[i]`` for
    ``meta_data.batch_size`` items; the response carries one ``raw_output`` per REQUESTED output in request order.  Failures
    of the request (unknown model / binding, size mismatch, batch out of range) are reported in ``request_status`` the way
    TRTIS does, not as a transport error."""

    def execute_rpc(self, request, response):
        t0 = time.perf_counter()
        res: TrtisResources = self.get_resources()
        st = response.request_status
        response.batch_id = request.batch_id
        models = res.backend.models()
        meta = models.get(request.model_name)
        if meta is None:
            return _fail(st, res, NOT_FOUND, f"no model named '{request.model_name}'")
        hdr = request.meta_data
        n = int(hdr.batch_size)
        if n < 1 or n > meta["max_batch"]:
            return _fail(st, res, INVALID_ARG, f"batch_size {n} outside [1, {meta['max_batch']}]")
        if len(request.raw_input) != len(hdr.input) or len(hdr.input) != len(meta["inputs"]):
            return _fail(st, res, INVALID_ARG, f"{len(request.raw_input)} raw_input for {len(hdr.input)} declared and "
                                               f"{len(meta['inputs'])} model inputs")
        inputs = {}
        for decl, raw in zip(hdr.input, request.raw_input):
            if decl.name not in meta["inputs"]:
                return _fail(st, res, NOT_FOUND, f"model '{request.model_name}' has no input '{decl.name}'")
            shape, dt = meta["inputs"][decl.name]
            want = n * int(np.prod(shape)) * np.dtype(dt).itemsize
            if len(raw) != want or (decl.byte_size and decl.byte_size != want):
                return _fail(st, res, INVALID_ARG, f"input '{decl.name}': {len(raw)} bytes, expected {want}")
            inputs[decl.name] = np.frombuffer(raw, dtype=dt).reshape((n,) + tuple(shape))
        for o in hdr.output:
            if o.name not in meta["outputs"]:
                return _fail(st, res, NOT_FOUND, f"model '{request.model_name}' has no output '{o.name}'")
            if o.HasField("cls"):
                return _fail(st, res, 7, "classification outputs are not provided; request the raw tensor")  # UNSUPPORTED
        try:
            outs, compute_s = res.backend.infer(request.model_name, inputs)
        except Exception as ex:  # the pipeline's failure belongs in the status, the connection stays usable
            return _fail(st, res, INTERNAL, f"{type(ex).__name__}: {ex}")
        out_hdr = response.meta_data
        out_hdr.model_name, out_hdr.model_version, out_hdr.batch_size = request.model_name, 1, n
        for o in hdr.output:
            y = np.ascontiguousarray(outs[o.name])
            m = out_hdr.output.add()
            m.name, m.raw.byte_size = o.name, y.nbytes
            response.raw_output.append(y.tobytes())
        response.compute_time = float(compute_s)
        response.request_time = float(time.perf_counter() - t0)
        _ok(st, res)


def build_trtis_server(backend, address: str = "127.0.0.1:0", contexts: int = 8, executor_threads: int = 8) -> rpc.Server:
    """The reference's BasicInferService (infer.cc:214-260): Status + Health + Infer of ``nvidia.inferenceserver.GRPCService``."""
    server = rpc.Server(address)
    svc = server.register_async_service(SERVICE)
    resources = TrtisResources(backend)
    executor = server.register_executor(rpc.Executor(executor_threads))
    for method, req, resp, ctx, n in (("Status", "StatusRequest", "StatusResponse", StatusContext, 2),
                                      ("Health", "HealthRequest", "HealthResponse", HealthContext, 2),
                                      ("Infer", "InferRequest", "InferResponse", InferContext, contexts)):
        executor.register_contexts(svc.register_rpc(method, message(req), message(resp), ctx), resources, n)
    return server


def serve_pybind(manager, port: int = 50052, block: bool = True):
    """What ``trtlab.InferenceManager.serve(port)`` runs (infer.cc:411-417): the TRTIS service in front of the pybind manager."""
    server = build_trtis_server(PybindBackend(manager), f"0.0.0.0:{port}").async_start()
    if block:  # the reference blocks in server.Run()
        try:
            while server.running():
                time.sleep(0.2)
        except KeyboardInterrupt:
            server.shutdown()
    return server


# ------------------------------------------------------------------------------------------------
# client side (infer.cc:430-642)
# ------------------------------------------------------------------------------------------------
class TrtisError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"TRTIS request failed (code {code}): {msg}")
        self.code = code


class InferFuture:
    def __init__(self, fut: "futures.Future"):
        self._fut = fut

    def get(self, timeout: Optional[float] = None) -> Dict[str, np.ndarray]:
        return self._fut.result(timeout)

    result = get

    def wait(self, timeout: Optional[float] = None):
        futures.wait([self._fut], timeout)


class RemoteInferRunner:
    """PyInferRemoteRunner (infer.cc:430-538): numpy in, future of {output name: numpy} out, over GRPCService/Infer."""

    def __init__(self, name: str, config, client: rpc.ClientUnary):
        self.name, self._client = name, client
        self._max_batch = int(config.max_batch_size)
        self._inputs = {i.name: (tuple(int(d) for d in i.dims), np.dtype(_NP_OF[i.data_type])) for i in config.input}
        self._outputs = {o.name: (tuple(int(d) for d in o.dims), np.dtype(_NP_OF[o.data_type])) for o in config.output}

    def max_batch_size(self) -> int:
        return self._max_batch

    def input_bindings(self) -> Dict[str, dict]:
        return {k: {"shape": list(s), "dtype": d} for k, (s, d) in self._inputs.items()}

    def output_bindings(self) -> Dict[str, dict]:
        return {k: {"shape": list(s), "dtype": d} for k, (s, d) in self._outputs.items()}

    def infer(self, **inputs) -> InferFuture:
        if set(inputs) != set(self._inputs):
            raise ValueError(f"model '{self.name}' takes inputs {sorted(self._inputs)}, got {sorted(inputs)}")
        req = message("InferRequest")()
        req.model_name = self.name
        batch = None
        for k, v in inputs.items():
            shape, dt = self._inputs[k]
            if dt == np.uint8 and np.asarray(v).dtype != np.uint8:
                raise TypeError(f"input '{k}' takes uint8 images, got {np.asarray(v).dtype}")
            a = np.ascontiguousarray(v, dtype=dt)
            if a.shape[1:] != shape:
                if a.shape == shape:  # a single item without its batch dimension, as the reference accepts
                    a = a.reshape((1,) + shape)
                else:
                    raise ValueError(f"input '{k}': shape {a.shape} does not end in {shape}")
            if batch is not None and a.shape[0] != batch:
                raise ValueError("inputs disagree on the batch size")
            batch = a.shape[0]
            i = req.meta_data.input.add()
            i.name, i.byte_size = k, a.nbytes
            req.raw_input.append(a.tobytes())
        if batch > self._max_batch:
            raise ValueError(f"batch {batch} exceeds the model's max batch size {self._max_batch}")
        req.meta_data.batch_size = batch
        for k in self._outputs:
            req.meta_data.output.add().name = k

        def on_complete(request, response, status):
            if status != grpc.StatusCode.OK:
                raise TrtisError(UNAVAILABLE, f"transport: {status}")
            if response.request_status.code != SUCCESS:
                raise TrtisError(response.request_status.code, response.request_status.msg)
            out = {}
            for m, raw in zip(response.meta_data.output, response.raw_output):
                shape, dt = self._outputs[m.name]
                out[m.name] = np.frombuffer(raw, dtype=dt).reshape((response.meta_data.batch_size,) + shape).copy()
            return out

        return InferFuture(self._client.enqueue(req, on_complete))


class RemoteInferenceManager:
    """PyRemoteInferenceManager (infer.cc:547-642): ``get_models()`` asks GRPCService/Status, ``infer_runner(name)``
    returns a runner whose bindings come from the served model's ModelConfig."""

    def __init__(self, hostname: str = "localhost:50052"):
        self.hostname = hostname
        self._status = rpc.ClientUnary(hostname, f"/{SERVICE}/Status", message("StatusRequest"), message("StatusResponse"))
        self._health = rpc.ClientUnary(hostname, f"/{SERVICE}/Health", message("HealthRequest"), message("HealthResponse"))
        self._infer = rpc.ClientUnary(hostname, f"/{SERVICE}/Infer", message("InferRequest"), message("InferResponse"))
        self._configs: Dict[str, object] = {}

    def server_status(self, model_name: str = ""):
        resp = self._status.enqueue(message("StatusRequest")(model_name=model_name)).result(30)
        if resp is None:
            raise TrtisError(UNAVAILABLE, f"no TRTIS service at {self.hostname}")
        if resp.request_status.code != SUCCESS:
            raise TrtisError(resp.request_status.code, resp.request_status.msg)
        return resp.server_status

    def is_healthy(self, mode: str = "ready") -> bool:
        resp = self._health.enqueue(message("HealthRequest")(mode=mode)).result(30)
        return bool(resp is not None and resp.request_status.code == SUCCESS and resp.health)

    def get_models(self) -> List[str]:
        status = self.server_status()
        self._configs = {name: ms.config for name, ms in status.model_status.items()}
        return sorted(self._configs)

    def infer_runner(self, name: str) -> RemoteInferRunner:
        if name not in self._configs:
            self.get_models()
        if name not in self._configs:
            raise KeyError(f"model '{name}' is not served by {self.hostname}")
        return RemoteInferRunner(name, self._configs[name], self._infer)

    def close(self):
        for c in (self._status, self._health, self._infer):
            c.close()
