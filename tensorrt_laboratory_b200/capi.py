"""ctypes binding of the C ABI (``include/b200infer.h`` + ``include/b200cuda.h``).

The shared library is built in-tree by ``__graft_entry__.build()``.  Loading fails LOUDLY when it is
missing -- there is no Python/CPU fallback for any compute entry point.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200infer.so")

_lib = None

# (name, restype, argtypes) -- every symbol declared in include/b200infer.h and include/b200cuda.h
_VP, _I, _SZ, _D, _S = C.c_void_p, C.c_int, C.c_size_t, C.c_double, C.c_char_p
_PVP = C.POINTER(C.c_void_p)
SYMBOLS = [
    ("b2_abi_version", _I, []),
    ("b2_last_error", _S, []),
    ("b2_runtime_create", _I, [_PVP]),
    ("b2_runtime_destroy", None, [_VP]),
    ("b2_runtime_set_allocator", _I, [_VP, _VP, _VP, _VP]),
    ("b2_engine_deserialize", _I, [_VP, _VP, _SZ, _PVP]),
    ("b2_engine_inspect", _I, [_VP, _SZ, _PVP]),
    ("b2_engine_destroy", None, [_VP]),
    ("b2_engine_nb_bindings", _I, [_VP]),
    ("b2_engine_binding_name", _S, [_VP, _I]),
    ("b2_engine_binding_index", _I, [_VP, _S]),
    ("b2_engine_binding_is_input", _I, [_VP, _I]),
    ("b2_engine_binding_dtype", _I, [_VP, _I]),
    ("b2_engine_binding_dims", _I, [_VP, _I, C.POINTER(C.c_int32), C.POINTER(C.c_int)]),
    ("b2_engine_max_batch", _I, [_VP]),
    ("b2_engine_precision", _I, [_VP]),
    ("b2_engine_name", _S, [_VP]),
    ("b2_engine_device_memory_size", _SZ, [_VP]),
    ("b2_engine_weights_size", _SZ, [_VP]),
    ("b2_engine_flops", _D, [_VP, _I]),
    ("b2_engine_nb_layers", _I, [_VP]),
    ("b2_context_create", _I, [_VP, _PVP]),
    ("b2_context_destroy", None, [_VP]),
    ("b2_context_set_device_memory", _I, [_VP, _VP]),
    ("b2_context_enqueue", _I, [_VP, _I, _PVP, _VP, _VP]),
    ("b2_context_nb_launches", _I, [_VP, _I]),
    ("b2_context_set_option", _I, [_VP, _S, _I]),
    ("b2_engine_tune", _I, [_VP, _I, _I]),
    ("b2_engine_refine_tactics", _I, [_VP, _I, _I, C.POINTER(_D)]),
    ("b2_engine_nb_tactics", _I, [_VP]),
    ("b2_engine_get_tactics", _I, [_VP, C.POINTER(C.c_uint32), _I]),
    ("b2_context_prepare", _I, [_VP, _I, _VP]),
    ("b2_context_profile", _I, [_VP, _I, _PVP, _VP, C.POINTER(C.c_float), _I]),
    ("b2_context_launch_name", _S, [_VP, _I, _I]),
    ("b2_context_launch_flops", _D, [_VP, _I, _I]),
    ("b2_context_launch_bytes", _D, [_VP, _I, _I]),
    # b200cuda.h
    ("b2_device_count", _I, []),
    ("b2_device_set", _I, [_I]),
    ("b2_device_get", _I, []),
    ("b2_device_set_blocking_sync", _I, [_I]),
    ("b2_device_info", _I, [_I, _S, _I, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I), C.POINTER(_SZ), C.POINTER(_SZ)]),
    ("b2_device_cpu_affinity", _I, [_I, C.POINTER(C.c_uint64), _I]),
    ("b2_bind_thread_to_device", _I, [_I, C.POINTER(_I)]),
    ("b2_malloc_device", _I, [_PVP, _SZ]),
    ("b2_free_device", _I, [_VP]),
    ("b2_malloc_host", _I, [_PVP, _SZ]),
    ("b2_free_host", _I, [_VP]),
    ("b2_memset_device", _I, [_VP, _I, _SZ, _VP]),
    ("b2_stream_create", _I, [_PVP]),
    ("b2_stream_destroy", _I, [_VP]),
    ("b2_stream_sync", _I, [_VP]),
    ("b2_stream_query", _I, [_VP]),
    ("b2_event_create", _I, [_PVP, _I]),
    ("b2_event_destroy", _I, [_VP]),
    ("b2_event_record", _I, [_VP, _VP]),
    ("b2_event_sync", _I, [_VP]),
    ("b2_event_query", _I, [_VP]),
    ("b2_event_elapsed_ms", _I, [_VP, _VP, C.POINTER(C.c_float)]),
    ("b2_stream_wait_event", _I, [_VP, _VP]),
    ("b2_memcpy_h2d", _I, [_VP, _VP, _SZ, _VP]),
    ("b2_memcpy_d2h", _I, [_VP, _VP, _SZ, _VP]),
    ("b2_memcpy_d2d", _I, [_VP, _VP, _SZ, _VP]),
    ("b2_device_sync", _I, []),
    ("b2_profiler_start", _I, []),
    ("b2_profiler_stop", _I, []),
    # trtlab_host.h
    ("trt_manager_create", _I, [_I, _I, _I, _I, _I, _PVP]),
    ("trt_manager_destroy", None, [_VP]),
    ("trt_manager_register_model", _I, [_VP, _S, _VP, _SZ, _I]),
    ("trt_manager_allocate", _I, [_VP]),
    ("trt_manager_infer", _I, [_VP, _S, _I, _VP, _SZ, _VP, _SZ, C.POINTER(_D)]),
    ("trt_manager_infer_batched", _I, [_VP, _S, _I, _VP, _VP, _I, C.POINTER(_I)]),
    ("trt_manager_bench_batched", _I, [_VP, _S, _I, _VP, _I, _VP, _I, _I, _I, C.POINTER(_D), C.POINTER(_D), C.POINTER(_I)]),
    ("trt_manager_metrics_text", _I, [_VP, C.c_char_p, _SZ]),
    ("trt_manager_serve_metrics", _I, [_VP, _I, C.POINTER(_I)]),
    ("trt_manager_prefill_inputs", _I, [_VP, _S, _VP, _SZ]),
    ("trt_manager_bench", _I, [_VP, _S, _I, _D, _SZ, C.POINTER(_D), C.POINTER(_D), _SZ, C.POINTER(_SZ)]),
    ("trt_manager_bench_window", _I, [_VP, _S, _I, _SZ, _SZ, _SZ, C.POINTER(_D), C.POINTER(_D), _SZ, C.POINTER(_SZ)]),
    ("trt_manager_bench_windows", _I, [_VP, _S, _I, _SZ, _SZ, _SZ, _SZ, C.POINTER(_D), C.POINTER(_D), _SZ, C.POINTER(_SZ)]),
    ("trt_timed_pipeline", _I, [_VP, _SZ, _I, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    ("trt_device_throughput", _I, [_VP, _SZ, _I, _I, _I, _I, _VP, _I, C.POINTER(_D), C.POINTER(_I), _VP, _SZ]),
    ("trt_workspace_infer", _I, [_VP, _SZ, _VP, _SZ, _VP, _SZ, _I, _I]),
    ("trt_cyclic_infer", _I, [_VP, _SZ, _I, _VP, _SZ, _VP, _SZ, _I, _I, C.POINTER(_D)]),
]

NP_DTYPES = {0: np.float32, 1: np.float16, 2: np.int8, 3: np.int32, 5: np.uint8}  # B2_DT_* (same order as utils.cc:40-46)
BENCH_KEYS = ["kMaxExecConcurrency", "kMaxCopyConcurrency", "kBatchSize", "kWalltime", "kBatchesComputed",
              "kBatchesPerSecond", "kInferencesPerSecond", "kSecondsPerBatch", "kExecutionTimePerBatch",
              "kLatencyP50", "kLatencyP90", "kLatencyP99", "kLatencyMax", "kGpuComputeTimePerBatch"]


def as_input(x, dtype) -> np.ndarray:
    """``x`` as a C-contiguous array of an input binding's dtype.  fp32 / fp16 bindings cast; a uint8 image binding takes
    uint8 only (casting normalised floats to uint8 would wrap them into garbage)."""
    if np.dtype(dtype) == np.uint8 and np.asarray(x).dtype != np.uint8:
        raise TypeError(f"this input binding takes uint8 images, got {np.asarray(x).dtype}")
    return np.ascontiguousarray(x, dtype=dtype)


class B2Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200infer error {code}: {msg}")
        self.code = code


def load():
    """dlopen the in-tree library and bind every declared symbol (raises if anything is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built (run `python __graft_entry__.py`). "
            "There is no CPU fallback for this package.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, restype, argtypes in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise B2Error(rc, (load().b2_last_error() or b"").decode(errors="replace"))


def device_count() -> int:
    return load().b2_device_count()


def device_cpu_affinity(device: int = 0) -> List[int]:
    """Host CPUs NVML reports as closest to `device` (reference DeviceInfo::Affinity); [] when unknown."""
    mask = (C.c_uint64 * 16)()
    check(load().b2_device_cpu_affinity(device, mask, 16))
    return [i for i in range(1024) if (mask[i // 64] >> (i % 64)) & 1]


def bind_thread_to_device(device: int = 0) -> int:
    """Bind the calling thread to the GPU's CPUs (no-op when unknown / outside the cpuset); -> CPUs bound, 0 = unchanged."""
    n = _I()
    check(load().b2_bind_thread_to_device(device, C.byref(n)))
    return n.value


def device_info(device: int = 0) -> dict:
    lib = load()
    name = C.create_string_buffer(256)
    maj, mnr, sms = _I(), _I(), _I()
    mem, l2 = _SZ(), _SZ()
    check(lib.b2_device_info(device, name, 256, C.byref(maj), C.byref(mnr), C.byref(sms), C.byref(mem), C.byref(l2)))
    return dict(name=name.value.decode(), cc=(maj.value, mnr.value), sm_count=sms.value, total_mem=mem.value,
                l2_bytes=l2.value)


class DeviceBuffer:
    """RAII device allocation (cuda_malloc)."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        p = _VP()
        check(load().b2_malloc_device(C.byref(p), self.nbytes))
        self.ptr = p.value

    def free(self):
        if self.ptr:
            load().b2_free_device(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedBuffer:
    """RAII pinned host allocation (cuda_malloc_host) exposed as a numpy array."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        p = _VP()
        check(load().b2_malloc_host(C.byref(p), max(self.nbytes, 1)))
        self.ptr = p.value
        self._raw = (C.c_uint8 * max(self.nbytes, 1)).from_address(self.ptr)

    def array(self, dtype, shape) -> np.ndarray:
        a = np.frombuffer(self._raw, dtype=dtype, count=int(np.prod(shape)))
        return a.reshape(shape)

    def free(self):
        if self.ptr:
            self._raw = None
            load().b2_free_host(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Stream:
    def __init__(self):
        p = _VP()
        check(load().b2_stream_create(C.byref(p)))
        self.handle = p.value

    def sync(self):
        check(load().b2_stream_sync(self.handle))

    def destroy(self):
        if self.handle:
            load().b2_stream_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class Event:
    def __init__(self, timing: bool = True):
        p = _VP()
        check(load().b2_event_create(C.byref(p), 1 if timing else 0))
        self.handle = p.value

    def record(self, stream: "Stream"):
        check(load().b2_event_record(self.handle, stream.handle))

    def sync(self):
        check(load().b2_event_sync(self.handle))

    def elapsed_ms(self, stop: "Event") -> float:
        ms = C.c_float()
        check(load().b2_event_elapsed_ms(self.handle, stop.handle, C.byref(ms)))
        return ms.value

    def __del__(self):
        try:
            if self.handle:
                load().b2_event_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class Engine:
    """Deserialized plan on the current device (replaces nvinfer1::ICudaEngine)."""

    def __init__(self, blob: bytes, inspect_only: bool = False):
        lib = load()
        self._lib = lib
        self._blob = blob
        self._rt = _VP()
        self.handle = _VP()
        if inspect_only:
            check(lib.b2_engine_inspect(blob, len(blob), C.byref(self.handle)))
        else:
            check(lib.b2_runtime_create(C.byref(self._rt)))
            check(lib.b2_engine_deserialize(self._rt, blob, len(blob), C.byref(self.handle)))
        self.name = lib.b2_engine_name(self.handle).decode(errors="replace")
        self.max_batch = lib.b2_engine_max_batch(self.handle)
        self.precision = lib.b2_engine_precision(self.handle)
        self.bindings: List[dict] = []
        for i in range(lib.b2_engine_nb_bindings(self.handle)):
            dims = (C.c_int32 * 8)()
            nd = _I()
            check(lib.b2_engine_binding_dims(self.handle, i, dims, C.byref(nd)))
            shape = tuple(int(dims[d]) for d in range(nd.value))
            self.bindings.append(dict(
                name=lib.b2_engine_binding_name(self.handle, i).decode(errors="replace"),
                is_input=bool(lib.b2_engine_binding_is_input(self.handle, i)),
                dtype=lib.b2_engine_binding_dtype(self.handle, i),
                shape=shape,
                item_bytes=int(np.prod(shape)) * NP_DTYPES[lib.b2_engine_binding_dtype(self.handle, i)]().itemsize,
            ))
            self.bindings[-1]["np_dtype"] = NP_DTYPES[self.bindings[-1]["dtype"]]

    @property
    def device_memory_size(self) -> int:
        return self._lib.b2_engine_device_memory_size(self.handle)

    @property
    def weights_size(self) -> int:
        return self._lib.b2_engine_weights_size(self.handle)

    def tune(self, streams: int = 0, all_batches: bool = False) -> int:
        """Time the kernel tactics on this device now (model-registration time), never on the request path.
        -> number of tactics the engine holds."""
        check(self._lib.b2_engine_tune(self.handle, int(streams), 1 if all_batches else 0))
        return self._lib.b2_engine_nb_tactics(self.handle)

    def refine_tactics(self, streams: int = 4, passes: int = 1) -> float:
        """Network-level refinement of the tactic table in the serving regime (`streams` concurrent contexts);
        -> throughput after / before."""
        gain = _D()
        check(self._lib.b2_engine_refine_tactics(self.handle, int(streams), int(passes), C.byref(gain)))
        return gain.value

    def tactics(self) -> np.ndarray:
        """[n, 10] uint32: {op, batch, bn, stages, splits, sps, ws, cn, halo, 0} -- builder.attach_tactics() input."""
        n = self._lib.b2_engine_nb_tactics(self.handle)
        out = np.zeros((max(n, 1), 10), np.uint32)
        got = self._lib.b2_engine_get_tactics(self.handle, out.ctypes.data_as(C.POINTER(C.c_uint32)), n)
        return out[:got]

    def flops(self, batch: int) -> float:
        return self._lib.b2_engine_flops(self.handle, batch)

    def destroy(self):
        if getattr(self, "handle", None) and self.handle.value:
            self._lib.b2_engine_destroy(self.handle)
            self.handle = _VP()
        if getattr(self, "_rt", None) and self._rt.value:
            self._lib.b2_runtime_destroy(self._rt)
            self._rt = _VP()

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def input_np_dtype(blob: bytes):
    """numpy dtype of a plan's (single) input binding: float32, or float16 for plans built with input_dtype="f16"."""
    meta = Engine(blob, inspect_only=True)
    try:
        return [b["np_dtype"] for b in meta.bindings if b["is_input"]][0]
    finally:
        meta.destroy()


class Session:
    """One ExecutionContext + its activation arena + device/pinned binding buffers + a stream:
    the Python-side analogue of the reference's BenchmarkWorkspace (workspace.cc:90-124)."""

    def __init__(self, engine: Engine, options: Optional[Dict[str, int]] = None):
        lib = load()
        self._lib = lib
        self.engine = engine
        self.ctx = _VP()
        check(lib.b2_context_create(engine.handle, C.byref(self.ctx)))
        self.scratch = DeviceBuffer(engine.device_memory_size)
        check(lib.b2_context_set_device_memory(self.ctx, self.scratch.ptr))
        for k, v in (options or {}).items():
            check(lib.b2_context_set_option(self.ctx, k.encode(), int(v)))
        self.stream = Stream()
        self.dev = [DeviceBuffer(b["item_bytes"] * engine.max_batch) for b in engine.bindings]
        self.host = [PinnedBuffer(b["item_bytes"] * engine.max_batch) for b in engine.bindings]
        self._ptrs = (C.c_void_p * len(self.dev))(*[d.ptr for d in self.dev])

    def set_option(self, key: str, value: int):
        check(self._lib.b2_context_set_option(self.ctx, key.encode(), int(value)))

    def host_array(self, i: int, batch: Optional[int] = None) -> np.ndarray:
        b = self.engine.bindings[i]
        n = batch or self.engine.max_batch
        return self.host[i].array(b["np_dtype"], (n,) + b["shape"])

    def h2d(self, batch: int):
        for i, b in enumerate(self.engine.bindings):
            if b["is_input"]:
                check(self._lib.b2_memcpy_h2d(self.dev[i].ptr, self.host[i].ptr, b["item_bytes"] * batch, self.stream.handle))

    def d2h(self, batch: int):
        for i, b in enumerate(self.engine.bindings):
            if not b["is_input"]:
                check(self._lib.b2_memcpy_d2h(self.host[i].ptr, self.dev[i].ptr, b["item_bytes"] * batch, self.stream.handle))

    def enqueue(self, batch: int):
        check(self._lib.b2_context_enqueue(self.ctx, batch, self._ptrs, self.stream.handle, None))

    def infer(self, x: np.ndarray) -> Dict[str, np.ndarray]:
        """Synchronous convenience: pinned H2D -> forward -> D2H.  ``x``: [batch, C, H, W] cast to the binding dtype, or
        uint8 [batch, H, W, C] images for a uint8 binding."""
        inputs = [i for i, b in enumerate(self.engine.bindings) if b["is_input"]]
        if len(inputs) != 1:
            raise ValueError("infer() handles single-input engines")
        x = as_input(x, self.engine.bindings[inputs[0]]["np_dtype"])
        batch = x.shape[0]
        self.host_array(inputs[0], batch)[...] = x
        self.h2d(batch)
        self.enqueue(batch)
        self.d2h(batch)
        self.stream.sync()
        return {b["name"]: self.host_array(i, batch).copy()
                for i, b in enumerate(self.engine.bindings) if not b["is_input"]}

    def profile(self, batch: int) -> List[dict]:
        """Per-launch device times of one (serialised) forward pass."""
        n = self._lib.b2_context_nb_launches(self.ctx, batch)
        if n < 0:
            check(3)
        ms = (C.c_float * n)()
        got = self._lib.b2_context_profile(self.ctx, batch, self._ptrs, self.stream.handle, ms, n)
        if got < 0:
            raise B2Error(3, (self._lib.b2_last_error() or b"").decode())
        return [dict(name=self._lib.b2_context_launch_name(self.ctx, batch, i).decode(), ms=float(ms[i]),
                     flops=self._lib.b2_context_launch_flops(self.ctx, batch, i),
                     bytes=self._lib.b2_context_launch_bytes(self.ctx, batch, i)) for i in range(n)]

    def nb_launches(self, batch: int) -> int:
        return self._lib.b2_context_nb_launches(self.ctx, batch)

    def prepare(self, batch: int):
        """Build the launch plan and instantiate its graph segments ahead of the first request."""
        check(self._lib.b2_context_prepare(self.ctx, batch, self.stream.handle))

    def close(self):
        if self.ctx and self.ctx.value:
            try:
                self.stream.sync()
            except Exception:
                pass
            self._lib.b2_context_destroy(self.ctx)
            self.ctx = _VP()
        for b in self.dev:
            b.free()
        for b in self.host:
            b.free()
        self.scratch.free()
        self.stream.destroy()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class InferenceManager:
    """Python handle on the C++ ``trtlab::TensorRT::InferenceManager`` pipeline (pools of Buffers and
    ExecutionContexts + pre/cuda/post thread pools), the reference's v1 surface
    (trtlab/tensorrt/src/inference_manager.cc:59-327; python flavour: trtlab/pybind/trtlab/infer.cc:683-694)."""

    def __init__(self, max_exec_concurrency: int = 1, max_copy_concurrency: int = 0, pre_threads: int = 1,
                 cuda_threads: int = 1, post_threads: int = 3):
        self._lib = load()
        self.handle = _VP()
        check(self._lib.trt_manager_create(max_exec_concurrency, max_copy_concurrency, pre_threads, cuda_threads,
                                           post_threads, C.byref(self.handle)))
        self._blobs = []
        self.models: Dict[str, Engine] = {}

    def register_model(self, name: str, blob: bytes, max_concurrency: int = 0):
        check(self._lib.trt_manager_register_model(self.handle, name.encode(), blob, len(blob), max_concurrency))
        self._blobs.append(blob)
        self.models[name] = Engine(blob, inspect_only=True)

    def update_resources(self):
        check(self._lib.trt_manager_allocate(self.handle))

    allocate_resources = update_resources

    def infer(self, name: str, x: np.ndarray) -> np.ndarray:
        meta = self.models[name]
        x = as_input(x, [b["np_dtype"] for b in meta.bindings if b["is_input"]][0])
        batch = x.shape[0]
        ob = [b for b in meta.bindings if not b["is_input"]][0]
        out = np.empty((batch,) + ob["shape"], dtype=np.float32)
        sec = _D()
        check(self._lib.trt_manager_infer(self.handle, name.encode(), batch, x.ctypes.data, x.nbytes,
                                          out.ctypes.data, out.nbytes, C.byref(sec)))
        self.last_compute_seconds = sec.value  # device time of the forward pass (ExecutionContext::Synchronize)
        return out

    def infer_timed(self, name: str, x: np.ndarray):
        """-> (output, device seconds of the forward pass), what the reference service reports as compute_time
        (examples/02_TensorRT_GRPC/src/server.cc:169)."""
        meta = self.models[name]
        x = as_input(x, [b["np_dtype"] for b in meta.bindings if b["is_input"]][0])
        batch = x.shape[0]
        ob = [b for b in meta.bindings if not b["is_input"]][0]
        out = np.empty((batch,) + ob["shape"], dtype=np.float32)
        sec = _D()
        check(self._lib.trt_manager_infer(self.handle, name.encode(), batch, x.ctypes.data, x.nbytes,
                                          out.ctypes.data, out.nbytes, C.byref(sec)))
        return out, sec.value

    def infer_batched(self, name: str, x: np.ndarray, window_us: int = 2000):
        """Every image of ``x`` as its own request through BatchedInferRunner -> (outputs [n, ...], merged forward passes)."""
        meta = self.models[name]
        x = as_input(x, [b["np_dtype"] for b in meta.bindings if b["is_input"]][0])
        ob = [b for b in meta.bindings if not b["is_input"]][0]
        out = np.empty((x.shape[0],) + ob["shape"], dtype=np.float32)
        nb = _I(0)
        check(self._lib.trt_manager_infer_batched(self.handle, name.encode(), x.shape[0], x.ctypes.data, out.ctypes.data,
                                                  window_us, C.byref(nb)))
        return out, nb.value

    def bench_batched(self, name: str, ring: np.ndarray, n: int, warm: int, cool: int, window_us: int = 2000):
        """One flood of ``n`` single-image requests (inputs cycle through ``ring``) through BatchedInferRunner ->
        (outputs [n, ...], seconds spanned by the completions of requests [warm, n - cool), total seconds, merged batches)."""
        meta = self.models[name]
        ring = as_input(ring, [b["np_dtype"] for b in meta.bindings if b["is_input"]][0])
        ob = [b for b in meta.bindings if not b["is_input"]][0]
        out = np.empty((n,) + ob["shape"], dtype=np.float32)
        win, tot, nb = _D(), _D(), _I(0)
        check(self._lib.trt_manager_bench_batched(self.handle, name.encode(), n, ring.ctypes.data, ring.shape[0], out.ctypes.data,
                                                  window_us, warm, cool, C.byref(win), C.byref(tot), C.byref(nb)))
        return out, win.value, tot.value, nb.value

    def metrics_text(self) -> str:
        """Prometheus text exposition (request/compute summaries, load-ratio histogram, GPU power gauge)."""
        buf = C.create_string_buffer(1 << 16)
        n = self._lib.trt_manager_metrics_text(self.handle, buf, len(buf))
        if n < 0:
            raise RuntimeError(self._lib.b2_last_error().decode())
        return buf.value.decode()

    def serve_metrics(self, port: int = 0) -> int:
        """Start the Prometheus HTTP endpoint (GET /metrics); -> the bound port."""
        bound = _I()
        check(self._lib.trt_manager_serve_metrics(self.handle, port, C.byref(bound)))
        return bound.value

    def prefill_inputs(self, name: str, ring: np.ndarray):
        ring = as_input(ring, [b["np_dtype"] for b in self.models[name].bindings if b["is_input"]][0])
        check(self._lib.trt_manager_prefill_inputs(self.handle, name.encode(), ring.ctypes.data, ring.shape[0]))

    def bench(self, name: str, batch: int, seconds: float = 5.0, max_batches: int = 0, want_latencies: bool = True):
        res = (C.c_double * 16)()
        cap = max(max_batches, 1 << 20) if want_latencies else 0
        lat = (C.c_double * cap)() if cap else None
        n = _SZ(0)
        check(self._lib.trt_manager_bench(self.handle, name.encode(), batch, seconds, max_batches, res, lat, cap, C.byref(n)))
        out = {k: res[i] for i, k in enumerate(BENCH_KEYS)}
        lats = np.frombuffer(lat, dtype=np.float64, count=n.value).copy() if cap else np.zeros(0)
        return out, lats

    def bench_window(self, name: str, batch: int, warm: int, steps: int, cool: int):
        """One continuous closed loop of warm + steps + cool requests; -> (seconds spanned by the `steps` completions in the
        middle, their latencies)."""
        win = _D()
        lat = (C.c_double * steps)()
        n = _SZ()
        check(self._lib.trt_manager_bench_window(self.handle, name.encode(), batch, warm, steps, cool, C.byref(win), lat, steps, C.byref(n)))
        return win.value, np.array(lat[: n.value])

    def bench_windows(self, name: str, batch: int, warm: int, steps: int, windows: int, cool: int):
        """One continuous closed loop of warm + windows * steps + cool requests; -> (seconds spanned by each of the `windows`
        consecutive groups of `steps` completions [windows], latencies of all their requests)."""
        win = (C.c_double * windows)()
        lat = (C.c_double * (steps * windows))()
        n = _SZ()
        check(self._lib.trt_manager_bench_windows(self.handle, name.encode(), batch, warm, steps, windows, cool, win, lat,
                                                  steps * windows, C.byref(n)))
        return np.array(win[:]), np.array(lat[: n.value])

    def close(self):
        if self.handle and self.handle.value:
            self._lib.trt_manager_destroy(self.handle)
            self.handle = _VP()
        for e in self.models.values():
            e.destroy()
        self.models = {}

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def timed_pipeline(blob: bytes, iters: int = 20):
    a, b, c = C.c_float(), C.c_float(), C.c_float()
    check(load().trt_timed_pipeline(blob, len(blob), iters, C.byref(a), C.byref(b), C.byref(c)))
    return dict(h2d_ms=a.value, compute_ms=b.value, d2h_ms=c.value)


def device_throughput(blob: bytes, contexts: int, batch: int, steps: int, warmup: int, ring: np.ndarray,
                      return_outputs: bool = False):
    """-> (elapsed_ms, kernel launches per step), and with ``return_outputs`` a third item: {output binding name:
    [batch, ...] array} computed by the last timed step (input ``ring[(steps - 1) % R]``).  ``ring``: [R, batch, C, H, W]
    host array (cast to the input dtype)."""
    ring = as_input(ring, input_np_dtype(blob))
    outs = []
    if return_outputs:
        meta = Engine(blob, inspect_only=True)
        outs = [b for b in meta.bindings if not b["is_input"]]
        meta.destroy()
    flat = np.empty(sum(batch * b["item_bytes"] for b in outs), np.uint8)  # the C side writes them back to back
    ms = _D()
    nl = _I()
    check(load().trt_device_throughput(blob, len(blob), contexts, batch, steps, warmup, ring.ctypes.data,
                                       ring.shape[0], C.byref(ms), C.byref(nl),
                                       flat.ctypes.data if return_outputs else None, flat.nbytes))
    if not return_outputs:
        return ms.value, nl.value
    arrays, off = {}, 0
    for b in outs:
        n = batch * b["item_bytes"]
        arrays[b["name"]] = flat[off:off + n].copy().view(b["np_dtype"]).reshape((batch,) + b["shape"])
        off += n
    return ms.value, nl.value, arrays


def _single_io(blob: bytes):
    meta = Engine(blob, inspect_only=True)
    ins = [b for b in meta.bindings if b["is_input"]]
    outs = [b for b in meta.bindings if not b["is_input"]]
    if len(ins) != 1 or len(outs) != 1:
        raise ValueError("single-input single-output engines only")
    return meta, ins[0], outs[0]


def workspace_infer(blob: bytes, x: np.ndarray, managed_runtime: bool = False, iters: int = 2) -> np.ndarray:
    """v2 surface: BenchmarkWorkspace at max batch (caller-captured graph); ``x``: [max_batch, C, H, W]."""
    meta, i, o = _single_io(blob)
    x = as_input(x, i["np_dtype"])
    out = np.zeros((meta.max_batch,) + o["shape"], o["np_dtype"])
    check(load().trt_workspace_infer(blob, len(blob), x.ctypes.data, x.nbytes, out.ctypes.data, out.nbytes, int(managed_runtime), iters))
    return out


def cyclic_infer(blob: bytes, x: np.ndarray, managed_runtime: bool = False, rounds: int = 7):
    """The v1 hot path by hand over CyclicBuffers<CudaPinnedHostMemory, CudaDeviceMemory>; -> (output, device seconds)."""
    meta, i, o = _single_io(blob)
    x = as_input(x, i["np_dtype"])
    out = np.zeros((x.shape[0],) + o["shape"], o["np_dtype"])
    sec = _D()
    check(load().trt_cyclic_infer(blob, len(blob), x.shape[0], x.ctypes.data, x.nbytes, out.ctypes.data, out.nbytes, int(managed_runtime),
                                  rounds, C.byref(sec)))
    return out, sec.value
