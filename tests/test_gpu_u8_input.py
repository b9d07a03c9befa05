"""GPU: uint8 HWC image input bindings.  The engine's first kernel (input_cast_u8_s2d_kernel / input_cast_u8_c8_kernel)
computes builder.preprocess_u8 in fp32 and rounds to fp16 exactly as the fp32 binding's cast does, so a uint8 engine is
BIT-IDENTICAL to the same engine's fp32 binding fed preprocess_u8(x): every comparison here is exact, through the C ABI,
the CUDA graph with re-pointed bindings, the InferenceManager pipelines, pybind and TRTIS."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle.caffe_forward import caffe_forward
from tensorrt_laboratory_b200 import builder, capi, graph, trtis, weights

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "tensorrt_laboratory_b200")
TV = dict(mean=builder.TORCHVISION_MEAN, std=builder.TORCHVISION_STD)
CAFFE_BGR = dict(mean=(104.0, 117.0, 123.0), std=1.0, reverse_channels=True)
CHW = (3, 224, 224)


def _run(blob, x, options=None):
    eng = capi.Engine(blob)
    sess = capi.Session(eng, options)
    try:
        return sess.infer(x)["prob"]
    finally:
        sess.close()
        eng.destroy()


@pytest.fixture(scope="module")
def rn50(gpu):
    net = graph.resnet_caffe(50)
    wts = weights.random_weights(net, 0)
    low = graph.lower(net, wts)
    return dict(net=net, wts=wts, low=low, f32=builder.build_plan(low, builder.PREC_FP16, 8))


def test_u8_engine_equals_fp32_binding_on_preprocessed_images(rn50):
    x = weights.synthetic_image_u8(8, (224, 224), seed=5)
    xp = builder.preprocess_u8(x, CHW, TV)
    blob = builder.build_plan(rn50["low"], builder.PREC_FP16, 8, input_dtype="u8", image=TV)
    eng = capi.Engine(blob)
    sess = capi.Session(eng)
    try:
        assert eng.bindings[0]["dtype"] == 5 and eng.bindings[0]["item_bytes"] == 150528
        got8, got3 = sess.infer(x)["prob"], sess.infer(x[:3])["prob"]
        launch = [capi.load().b2_context_launch_name(sess.ctx, 8, i).decode() for i in range(sess.nb_launches(8))]
    finally:
        sess.close()
        eng.destroy()
    want = _run(rn50["f32"], xp)
    np.testing.assert_array_equal(got8, want)
    np.testing.assert_array_equal(got3, want[:3])
    ref = caffe_forward(rn50["net"], rn50["wts"], xp)
    np.testing.assert_array_equal(got8.argmax(1), ref.reshape(8, -1).argmax(1))
    assert launch[0] == "input_cast:cast:data"          # launch names are "<kind>:<op name>"


@pytest.mark.parametrize("src_hw", [(256, 256), (241, 230)])
def test_crop_and_bgr_order(rn50, src_hw):
    """Centre crop from a larger source (241 x 230: both differences odd, crop_left * C odd) with Caffe BGR means, std 1."""
    img = dict(CAFFE_BGR, src_hw=src_hw)
    x = weights.synthetic_image_u8(8, src_hw, seed=6)
    blob = builder.build_plan(rn50["low"], builder.PREC_FP16, 8, input_dtype="u8", image=img)
    got = _run(blob, x)
    want = _run(rn50["f32"], builder.preprocess_u8(x, CHW, img))
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(_run(blob, x[:5]), want[:5])


def test_c8_kernel_without_space_to_depth(rn50):
    """stem_s2d=False: the stem reads an 8-channel NHWC tensor, written by input_cast_u8_c8_kernel."""
    img = dict(TV, src_hw=(241, 230), reverse_channels=True)
    x = weights.synthetic_image_u8(8, (241, 230), seed=7)
    blob = builder.build_plan(rn50["low"], builder.PREC_FP16, 8, input_dtype="u8", image=img, stem_s2d=False)
    f32 = builder.build_plan(rn50["low"], builder.PREC_FP16, 8, stem_s2d=False)
    want = _run(f32, builder.preprocess_u8(x, CHW, img))
    np.testing.assert_array_equal(_run(blob, x), want)
    np.testing.assert_array_equal(_run(blob, x[:3]), want[:3])


def test_graph_replay_repoints_the_u8_input(rn50):
    """Two different device input buffers through ONE context and its captured graph: the input cast's binding argument is
    re-pointed before each launch (patch_layout).  Each result must equal the direct-launch (graph=0) result."""
    blob = builder.build_plan(rn50["low"], builder.PREC_FP16, 8, input_dtype="u8", image=TV)
    xs = [weights.synthetic_image_u8(8, (224, 224), seed=s) for s in (8, 9)]
    lib = capi.load()
    eng = capi.Engine(blob)
    try:
        direct = [None, None]
        for graph_ in (0, 1):
            sess = capi.Session(eng, {"graph": graph_})
            extra = capi.DeviceBuffer(eng.bindings[0]["item_bytes"] * 8)
            try:
                assert sess.nb_launches(8) == 56
                bufs = [sess.dev[0].ptr, extra.ptr]
                for i, x in enumerate(xs):
                    sess.host_array(0)[...] = x
                    capi.check(lib.b2_memcpy_h2d(bufs[i], sess.host[0].ptr, x.nbytes, sess.stream.handle))
                    sess.stream.sync()
                outs = []
                for rep in range(3):
                    for i in (0, 1):
                        ptrs = (C.c_void_p * 2)(bufs[i], sess.dev[1].ptr)
                        capi.check(lib.b2_context_enqueue(sess.ctx, 8, ptrs, sess.stream.handle, None))
                        sess.d2h(8)
                        sess.stream.sync()
                        outs.append((i, sess.host_array(1).copy()))
                for i, y in outs:
                    if graph_ == 0 and direct[i] is None:
                        direct[i] = y
                    np.testing.assert_array_equal(y, direct[i])
            finally:
                extra.free()
                sess.close()
        assert not np.array_equal(direct[0], direct[1])
    finally:
        eng.destroy()


_ZC_SCRIPT = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from tensorrt_laboratory_b200 import builder, capi, weights
blob = builder.build_resnet_plan(50, builder.PREC_FP16, 8, input_dtype="u8", image=dict(mean=builder.TORCHVISION_MEAN,
                                 std=builder.TORCHVISION_STD))
x = weights.synthetic_image_u8(8, (224, 224), seed=10)
mgr = capi.InferenceManager(max_exec_concurrency=2, max_copy_concurrency=4)
mgr.register_model("rn50u8", blob)
mgr.update_resources()
np.savez(sys.argv[2], *[mgr.infer("rn50u8", x[:b]) for b in (8, 3)])
mgr.close()
"""


def test_manager_pipelines_feed_u8_bytes():
    """InferenceManager + InferRunner (pinned Buffers sized 150 528 B per image), with staged copies and with zero-copy
    input (TRTLAB_ZERO_COPY_INPUT=1, read once per process: in a child), equal the bare C ABI."""
    blob = builder.build_resnet_plan(50, builder.PREC_FP16, 8, input_dtype="u8", image=TV)
    x = weights.synthetic_image_u8(8, (224, 224), seed=10)
    direct = _run(blob, x)
    mgr = capi.InferenceManager(max_exec_concurrency=2, max_copy_concurrency=4)
    try:
        mgr.register_model("rn50u8", blob)
        mgr.update_resources()
        assert mgr.models["rn50u8"].bindings[0]["item_bytes"] == 150528
        np.testing.assert_array_equal(mgr.infer("rn50u8", x), direct)
        np.testing.assert_array_equal(mgr.infer("rn50u8", x[:3]), direct[:3])
        with pytest.raises(TypeError):
            mgr.infer("rn50u8", builder.preprocess_u8(x, CHW, TV))
    finally:
        mgr.close()
    out = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"zc_u8_{os.getpid()}.npz")
    try:
        r = subprocess.run([sys.executable, "-c", _ZC_SCRIPT, ROOT, out], env=dict(os.environ, TRTLAB_ZERO_COPY_INPUT="1"),
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        got = np.load(out)
        np.testing.assert_array_equal(got["arr_0"], direct)
        np.testing.assert_array_equal(got["arr_1"], direct[:3])
    finally:
        if os.path.exists(out):
            os.remove(out)


def test_int8_engine_with_u8_input():
    """ResNet-50 INT8 calibrated on preprocess_u8 images: the uint8 binding equals the same engine's fp32 binding, directly
    and as single-image requests merged by BatchedInferRunner."""
    low = builder.resnet_lowered(50, builder.PREC_INT8, image=TV)
    f32 = builder.build_plan(low, builder.PREC_INT8, 8)
    u8 = builder.build_plan(low, builder.PREC_INT8, 8, input_dtype="u8", image=TV)
    x = weights.synthetic_image_u8(8, (224, 224), seed=12)
    want = _run(f32, builder.preprocess_u8(x, CHW, TV))
    np.testing.assert_array_equal(_run(u8, x), want)
    np.testing.assert_array_equal(_run(u8, x[:3]), want[:3])
    mgr = capi.InferenceManager(max_exec_concurrency=2, max_copy_concurrency=4)
    try:
        mgr.register_model("rn50i8u8", u8)
        mgr.update_resources()
        got, batches = mgr.infer_batched("rn50i8u8", x, window_us=20000)
        assert 1 <= batches <= 8
        np.testing.assert_array_equal(got, want)
    finally:
        mgr.close()


def _trtlab():
    if PKG not in sys.path:
        sys.path.insert(0, PKG)
    import trtlab
    return trtlab


def test_pybind_and_trtis_serve_u8(rn50, tmp_path):
    trtlab = _trtlab()
    blob = builder.build_plan(rn50["low"], builder.PREC_FP16, 8, input_dtype="u8", image=TV)
    plan = tmp_path / "rn50_u8.plan"
    plan.write_bytes(blob)
    x = weights.synthetic_image_u8(8, (224, 224), seed=13)
    direct = _run(blob, x)
    models = trtlab.InferenceManager(max_exec_concurrency=2)
    runner = models.register_tensorrt_engine("rn50u8", str(plan))
    models.update_resources()
    ins = runner.input_bindings()
    assert list(ins) == ["data"] and ins["data"]["shape"] == [224, 224, 3] and ins["data"]["dtype"] == np.uint8
    (y,) = runner.infer(data=x).get().values()
    np.testing.assert_array_equal(np.asarray(y).reshape(8, -1), direct.reshape(8, -1))
    with pytest.raises(TypeError):
        runner.infer(data=x.astype(np.float32))
    srv = models.serve(port=0, block=False)
    try:
        remote = trtlab.RemoteInferenceManager(hostname=f"127.0.0.1:{srv.port}")
        status = remote.server_status("rn50u8")
        (inp,) = status.model_status["rn50u8"].config.input
        assert inp.data_type == trtis.TYPE_UINT8 and list(inp.dims) == [224, 224, 3]
        run = remote.infer_runner("rn50u8")
        for b in (8, 3):
            (val,) = run.infer(data=x[:b]).get(60).values()
            np.testing.assert_array_equal(val.reshape(b, -1), direct[:b].reshape(b, -1))
        with pytest.raises(TypeError):
            run.infer(data=x.astype(np.float32))
        remote.close()
    finally:
        srv.shutdown()
