"""GPU parity of whole networks through the C ABI and through the C++ InferenceManager pipeline.

Tolerances (stated per the north star):
  * MNIST (fp32 engine) vs the reference's golden vectors: abs 1.5e-3 on logits ~1e3 (decimal=3,
    reference examples/30_PyTensorRT/server.py:31), argmax 2/0/9.
  * ResNet-50 fp16 engine vs the fp32 CPU oracle: <= 1e-3 relative on `prob` (relative to the row max),
    identical argmax for every image; vs the fp16-emulating oracle: <= 1e-4.
"""
import numpy as np
import pytest

from oracle.caffe_forward import caffe_forward, lowered_forward_f16emu
from tensorrt_laboratory_b200 import builder, capi, graph, weights
from tests import helpers

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rn50():
    net = graph.resnet_caffe(50)
    wts = weights.random_weights(net, 0)
    low = graph.lower(net, wts)
    x = weights.synthetic_input(8)
    return dict(net=net, wts=wts, low=low, x=x)


@pytest.fixture(scope="module")
def rn50_ref(rn50):
    ref32 = caffe_forward(rn50["net"], rn50["wts"], rn50["x"])  # fp32, unfused Caffe semantics
    emu = lowered_forward_f16emu(rn50["low"], rn50["x"])
    return dict(ref32=ref32, emu=emu)


@pytest.fixture(scope="module")
def rn50_session(gpu, rn50):
    blob = builder.build_plan(rn50["low"], builder.PREC_FP16, 8)
    eng = capi.Engine(blob)
    sess = capi.Session(eng)
    yield dict(blob=blob, eng=eng, sess=sess)
    sess.close()
    eng.destroy()


def test_mnist_known_answer(gpu):
    net, w, xs, ys = helpers.load_mnist_golden()
    low = graph.lower(net, w)
    blob = builder.build_plan(low, builder.PREC_FP32, 4)
    eng = capi.Engine(blob)
    sess = capi.Session(eng)
    try:
        for x, y, am in zip(xs, ys, (2, 0, 9)):
            got = sess.infer(x)[low["output"]]
            assert np.abs(got - y).max() < 1.5e-3
            assert int(got.argmax()) == am
        got = sess.infer(np.concatenate(xs, 0))[low["output"]]
        assert np.abs(got - np.concatenate(ys, 0)).max() < 1.5e-3
    finally:
        sess.close()
        eng.destroy()


def test_resnet50_fp16_matches_oracles_full_batch(rn50, rn50_ref, rn50_session):
    prob = rn50_session["sess"].infer(rn50["x"])["prob"]
    assert prob.shape == (8, 1000)
    np.testing.assert_allclose(prob.sum(1), 1.0, atol=1e-5)
    ref32, emu = rn50_ref["ref32"], rn50_ref["emu"]
    assert (prob.argmax(1) == ref32.argmax(1)).all()  # bit-exact class index
    assert (prob.argmax(1) == emu.argmax(1)).all()
    rowmax = ref32.max(1, keepdims=True)
    assert (np.abs(prob - ref32) / rowmax).max() <= 1e-3
    assert (np.abs(prob - emu) / emu.max(1, keepdims=True)).max() <= 1e-4


def test_resnet50_intermediate_tensors(gpu, rn50):
    taps = ["conv1", "pool1", "res2a", "res3d", "res4f", "res5c", "pool5", "fc1000"]
    x = rn50["x"][:2]
    _, snaps = lowered_forward_f16emu(rn50["low"], x, keep=taps)
    out = helpers.run_engine(rn50["low"], x, builder.PREC_FP16, outputs=taps)
    for name in taps:
        assert helpers.rel_err(out[name].reshape(2, -1), snaps[name].reshape(2, -1)) <= 4e-3, name


def test_resnet50_fp32_engine_matches_fp32_oracle(gpu, rn50):
    x = rn50["x"][:1]
    ref = caffe_forward(rn50["net"], rn50["wts"], x)
    got = helpers.run_engine(rn50["low"], x, builder.PREC_FP32)["prob"]
    assert helpers.rel_err(got, ref) < 1e-5
    assert got.argmax() == ref.argmax()


def test_batch_position_invariance_and_partial_batches(rn50, rn50_session):
    """Size-independent property: an image's result does not depend on the batch it travels in."""
    sess = rn50_session["sess"]
    full = sess.infer(rn50["x"])["prob"]
    perm = np.array([3, 0, 7, 1, 6, 2, 5, 4])
    np.testing.assert_array_equal(sess.infer(rn50["x"][perm])["prob"], full[perm])
    for b in (1, 3, 5):
        np.testing.assert_array_equal(sess.infer(rn50["x"][:b])["prob"], full[:b])


def test_determinism_graph_replay_and_second_context(rn50, rn50_session):
    sess = rn50_session["sess"]
    a = sess.infer(rn50["x"])["prob"]
    b = sess.infer(rn50["x"])["prob"]  # cached CUDA graph replay
    np.testing.assert_array_equal(a, b)
    other = capi.Session(rn50_session["eng"], {"graph": 0})  # second context, direct launches
    try:
        np.testing.assert_array_equal(other.infer(rn50["x"])["prob"], a)
    finally:
        other.close()
    assert sess.nb_launches(8) == 56  # input cast, 53 convs, max pool, fused tail


def test_inference_manager_pipeline_matches_direct_path(rn50, rn50_session):
    """v1 surface: InferenceManager + InferRunner (pre -> cuda -> post thread pools, pooled Buffers /
    ExecutionContexts), results identical to the bare C-ABI path."""
    direct = rn50_session["sess"].infer(rn50["x"])["prob"]
    mgr = capi.InferenceManager(max_exec_concurrency=2, max_copy_concurrency=4)
    try:
        mgr.register_model("rn50", rn50_session["blob"])
        mgr.update_resources()
        for _ in range(3):  # cycles through different pooled Buffers / contexts
            np.testing.assert_array_equal(mgr.infer("rn50", rn50["x"]), direct)
        np.testing.assert_array_equal(mgr.infer("rn50", rn50["x"][:3]), direct[:3])
        res, lats = mgr.bench("rn50", 8, seconds=30.0, max_batches=64)
        assert res["kBatchesComputed"] == 64 and res["kInferencesPerSecond"] > 0
        assert res["kMaxExecConcurrency"] == 2 and res["kMaxCopyConcurrency"] == 4
        assert len(lats) == 64 and (lats > 0).all()
        # observability (SURVEY.md 8f N4): the reference service's four series, Prometheus text format
        text = mgr.metrics_text()
        assert 'yais_inference_compute_duration_ms_count{model="rn50"} 64' in text
        assert 'yais_inference_request_duration_ms{model="rn50",quantile="0.99"}' in text
        assert 'yais_inference_load_ratio_bucket{le="+Inf"} 64' in text
        assert 0 < res["kGpuComputeTimePerBatch"] < 0.05
    finally:
        mgr.close()


def test_fp16_input_binding_matches_fp32_binding(rn50, rn50_session):
    """Secondary mode: the input binding declared fp16.  The engine rounds fp32 inputs to fp16 in its first kernel anyway,
    so feeding the pre-rounded values through an fp16 binding gives bit-identical results -- via the bare C ABI and via
    the InferenceManager pipeline (pinned Buffers sized by the binding dtype)."""
    direct = rn50_session["sess"].infer(rn50["x"])["prob"]
    blob = builder.build_resnet_plan(50, builder.PREC_FP16, 8, input_dtype="f16")
    eng = capi.Engine(blob)
    assert [b["dtype"] for b in eng.bindings if b["is_input"]] == [1]
    assert [b["item_bytes"] for b in eng.bindings if b["is_input"]] == [3 * 224 * 224 * 2]
    sess = capi.Session(eng)
    try:
        np.testing.assert_array_equal(sess.infer(rn50["x"])["prob"], direct)
        np.testing.assert_array_equal(sess.infer(rn50["x"][:3])["prob"], direct[:3])
    finally:
        sess.close()
        eng.destroy()
    mgr = capi.InferenceManager(max_exec_concurrency=2, max_copy_concurrency=4)
    try:
        mgr.register_model("rn50h", blob)
        mgr.update_resources()
        np.testing.assert_array_equal(mgr.infer("rn50h", rn50["x"]), direct)
    finally:
        mgr.close()


def test_side_branches_run_forked_and_change_nothing(rn50, rn50_session):
    """The shortcut convolutions of the four "a" blocks run on a forked stream (a parallel branch of the captured graph)
    while branch2a/2b execute; results are bit-identical to the linear schedule, with and without graph replay."""
    eng = capi.Engine(rn50_session["blob"])
    outs = {}
    try:
        for fork, graph_ in ((1, 1), (0, 1), (1, 0)):
            sess = capi.Session(eng, {"fork": fork, "graph": graph_})
            try:
                outs[(fork, graph_)] = sess.infer(rn50["x"])["prob"]
                for _ in range(3):
                    np.testing.assert_array_equal(sess.infer(rn50["x"])["prob"], outs[(fork, graph_)])
                n = sess.nb_launches(8)
                names = [capi.load().b2_context_launch_name(sess.ctx, 8, i).decode() for i in range(n)]
                assert sum(1 for s_ in names if s_.endswith(" side")) == 4
            finally:
                sess.close()
    finally:
        eng.destroy()
    np.testing.assert_array_equal(outs[(1, 1)], outs[(0, 1)])
    np.testing.assert_array_equal(outs[(1, 0)], outs[(0, 1)])
    np.testing.assert_array_equal(outs[(1, 1)], rn50_session["sess"].infer(rn50["x"])["prob"])


def test_dynamic_batching_runner(rn50, rn50_session):
    """BatchedInferRunner: 13 single-image requests -> one full batch of 8 + one window-closed batch of 5; every image's
    result is bit-identical to the direct batch-8 path (results do not depend on the batch an image travels in)."""
    x = np.concatenate([rn50["x"], rn50["x"][:5]], axis=0)
    direct = rn50_session["sess"].infer(rn50["x"])["prob"]
    want = np.concatenate([direct, direct[:5]], axis=0)
    mgr = capi.InferenceManager(max_exec_concurrency=2, max_copy_concurrency=4)
    try:
        mgr.register_model("rn50", rn50_session["blob"])
        mgr.update_resources()
        got, batches = mgr.infer_batched("rn50", x, window_us=20000)
        assert batches == 2
        np.testing.assert_array_equal(got, want)
    finally:
        mgr.close()


def test_timed_benchmark_workspace(rn50_session):
    t = capi.timed_pipeline(rn50_session["blob"], iters=5)
    assert t["h2d_ms"] > 0 and t["compute_ms"] > 0 and t["d2h_ms"] > 0
    assert t["h2d_ms"] < 5 and t["compute_ms"] < 50


def test_device_throughput_harness(rn50_session):
    ring = weights.synthetic_input(8, ring=2)
    ms, launches = capi.device_throughput(rn50_session["blob"], contexts=2, batch=8, steps=8, warmup=4, ring=ring)
    assert ms > 0 and launches == 56


def test_device_throughput_returns_the_last_steps_outputs(rn50_session):
    """What `bench.py --dump-outputs` writes: step 7 of 8 ran on context 1 with input ring[7 % 3]."""
    ring = weights.synthetic_input(8, seed=7, ring=3)
    ms, _, outs = capi.device_throughput(rn50_session["blob"], contexts=2, batch=8, steps=8, warmup=4, ring=ring,
                                         return_outputs=True)
    assert ms > 0 and list(outs) == ["prob"] and outs["prob"].shape == (8, 1000) and outs["prob"].dtype == np.float32
    want = rn50_session["sess"].infer(ring[1])["prob"]
    assert (outs["prob"].argmax(1) == want.argmax(1)).all()
    assert (np.abs(outs["prob"] - want) / want.max(1, keepdims=True)).max() <= 1e-4


def test_enqueue_argument_validation(rn50_session):
    import ctypes as C
    lib = capi.load()
    sess = rn50_session["sess"]
    assert lib.b2_context_enqueue(sess.ctx, 9, sess._ptrs, sess.stream.handle, None) == 1  # batch > max
    assert lib.b2_context_enqueue(sess.ctx, 0, sess._ptrs, sess.stream.handle, None) == 1
    nulls = (C.c_void_p * 2)(None, None)
    assert lib.b2_context_enqueue(sess.ctx, 1, nulls, sess.stream.handle, None) == 1
    assert lib.b2_context_set_option(sess.ctx, b"nonsense", 1) == 1


def test_resnet152_fp16_matches_oracle(gpu):
    """The reference's other in-tree deploy net (models/ResNet-152-deploy.prototxt, 155 convs).
    With these weights the logits reach ~90 and the softmax is NOT saturated (p_max ~0.5-0.7), so `prob` inherits the
    fp16 noise of the logits: the fp16-EMULATING oracle itself is 7e-3 away from the fp32 oracle on `prob`.  The bar is
    therefore stated on the logits (<= 1e-3 relative, the north-star tolerance), identical argmax, and `prob` within the
    fp16 noise floor measured by the two oracles."""
    net = graph.resnet_caffe(152)
    wts = weights.random_weights(net, 0)
    low = graph.lower(net, wts)
    x = weights.synthetic_input(2, seed=7)
    emu, emu_t = lowered_forward_f16emu(low, x, keep=["fc1000"])
    ref32, ref_t = caffe_forward(net, wts, x, keep=["fc1000"])
    out = helpers.run_engine(low, x, builder.PREC_FP16, outputs=["fc1000", "prob"], max_batch=2)
    prob, logits = out["prob"], out["fc1000"].reshape(2, -1)
    assert (prob.argmax(1) == ref32.argmax(1)).all() and (prob.argmax(1) == emu.argmax(1)).all()
    assert helpers.rel_err(logits, ref_t["fc1000"].reshape(2, -1)) <= 1e-3
    assert helpers.rel_err(logits, emu_t["fc1000"].reshape(2, -1)) <= 1e-3
    floor = float((np.abs(emu - ref32) / ref32.max(1, keepdims=True)).max())  # fp16 noise floor of this network
    e_32 = float((np.abs(prob - ref32) / ref32.max(1, keepdims=True)).max())
    assert e_32 <= max(2.0 * floor, 2e-3), (e_32, floor)
    np.testing.assert_allclose(prob.sum(1), 1.0, atol=1e-5)


def test_tactic_cache_roundtrip(gpu, tmp_path, monkeypatch):
    """B2_TUNE_CACHE: tactics timed by one engine instance (b2_engine_tune, model-registration time) are reused by the
    next (no re-timing, same results)."""
    cache = tmp_path / "tactics.txt"
    monkeypatch.setenv("B2_TUNE_CACHE", str(cache))
    _, _, low = helpers.conv_case(64, 28, 28, 128, 3, 1, 1)
    x = np.random.default_rng(0).standard_normal((2, 64, 28, 28), dtype=np.float32)
    blob = builder.build_plan(low, builder.PREC_FP16, 2)

    def run():
        eng = capi.Engine(blob)
        assert eng.tune(streams=2) == 1
        sess = capi.Session(eng)
        try:
            return list(sess.infer(x).values())[0]
        finally:
            sess.close()
            eng.destroy()

    a = run()
    lines = cache.read_text().strip().splitlines()
    assert len(lines) == 1 and len(lines[0].split()) == 10
    b = run()
    assert cache.read_text().strip().splitlines() == lines  # nothing re-tuned
    np.testing.assert_array_equal(a, b)
