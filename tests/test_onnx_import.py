"""ONNX front-end (SURVEY.md 8f N4): generic importer for CNN classifiers + the exporter used to round-trip it."""
import os

import numpy as np
import pytest

from oracle.caffe_forward import caffe_forward
from tensorrt_laboratory_b200 import builder, graph, onnx_import, onnx_lite, weights
from tests import helpers

MNIST_ONNX = os.path.join(helpers.GOLDEN, "mnist_v1_3_model.onnx")


def _same_lowering(a, b, tol=1e-6):
    assert [o["type"] for o in a["ops"]] == [o["type"] for o in b["ops"]]
    for x, y in zip(a["ops"], b["ops"]):
        for k in ("cin", "cout", "k", "stride", "pad", "relu"):
            assert x.get(k) == y.get(k), (x["name"], k)
        assert (x.get("residual") is None) == (y.get("residual") is None)
        if "W" in x:
            assert np.abs(x["W"] - y["W"]).max() <= tol and np.abs(x["bias"] - y["bias"]).max() <= tol, x["name"]


def test_resnet50_round_trips_through_onnx():
    """Caffe-v1 ResNet-50 -> ONNX bytes (Conv / BatchNormalization / Relu / Add / MaxPool(ceil) / GlobalAveragePool /
    Flatten / Gemm / Softmax) -> importer: the lowered graph (fused ops, folded weights) is the same."""
    net = graph.resnet_caffe(50)
    w = weights.random_weights(net, 0)
    model = onnx_lite.parse_model(onnx_import.export_onnx(net, w))
    assert model["input_shapes"] == {"data": [1, 3, 224, 224]} and len(model["nodes"]) == 176
    net2, w2 = onnx_import.import_onnx(model, name="ResNet-50")
    _same_lowering(graph.lower(net, w), graph.lower(net2, w2))
    # and the plan builder accepts it (same blob size: same tensors, ops, payload)
    assert len(builder.build_plan(graph.lower(net2, w2), builder.PREC_FP16, 2)) == len(builder.build_plan(graph.lower(net, w), builder.PREC_FP16, 2))


def test_round_trip_preserves_the_forward_pass():
    net = builder.single_conv_net(8, 12, 12, 16, 3, 1, 1, relu=True, residual=True)
    net["layers"].append(dict(name="pool", type="Pooling", bottoms=[net["layers"][-1]["tops"][0]], tops=["pool"], pool="MAX",
                              kernel_size=3, stride=2, pad=0))
    net["layers"].append(dict(name="gap", type="Pooling", bottoms=["pool"], tops=["gap"], pool="AVE", kernel_size=6, stride=1, pad=0))
    net["layers"].append(dict(name="fc", type="InnerProduct", bottoms=["gap"], tops=["fc"], num_output=5, bias_term=True))
    net["layers"].append(dict(name="prob", type="Softmax", bottoms=["fc"], tops=["prob"]))
    w = weights.random_weights(net, 3)
    x = np.random.default_rng(0).standard_normal((2,) + tuple(net["input_dims"][1:])).astype(np.float32)
    net2, w2 = onnx_import.import_onnx(onnx_lite.parse_model(onnx_import.export_onnx(net, w)))
    np.testing.assert_allclose(caffe_forward(net2, w2, x), caffe_forward(net, w, x), rtol=1e-5, atol=1e-6)


def test_reference_mnist_model_through_the_generic_importer():
    model = onnx_lite.load_model(MNIST_ONNX)
    net, w = onnx_import.import_onnx(model, name="mnist-v1.3")     # Conv(SAME_UPPER)+Add, Relu, MaxPool, Reshape, MatMul+Add
    net0, w0 = onnx_lite.mnist_to_caffe_like(model)
    _same_lowering(graph.lower(net, w), graph.lower(net0, w0), tol=0.0)
    _, _, xs, ys = helpers.load_mnist_golden()
    for x, y, want in zip(xs, ys, (2, 0, 9)):
        got = caffe_forward(net, w, x)
        np.testing.assert_almost_equal(got.reshape(1, 10), y.reshape(1, 10), decimal=3)
        assert int(got.argmax()) == want


def test_unsupported_operators_are_reported():
    net = builder.single_conv_net(8, 8, 8, 8, 1, 1, 0)
    w = weights.random_weights(net, 0)
    model = onnx_lite.parse_model(onnx_import.export_onnx(net, w))
    model["nodes"].append({"inputs": [model["nodes"][-1]["outputs"][0]], "outputs": ["y"], "name": "lstm", "op": "LSTM", "attrs": {}})
    with pytest.raises(ValueError, match="unsupported operator LSTM"):
        onnx_import.import_onnx(model)
    with pytest.raises(ValueError, match="input shape"):
        onnx_import.import_onnx({**model, "nodes": model["nodes"][:-1], "input_shapes": {}})


def test_corrupt_onnx_files_are_value_errors_never_crashes():
    """Random truncations and byte flips of a valid ModelProto either parse (payload bytes changed) or raise ValueError."""
    import random
    sys_path_net = builder.single_conv_net(64, 8, 8, 64, 3, 1, 1, residual=True)
    buf = onnx_import.export_onnx(sys_path_net, weights.random_weights(sys_path_net, 0))
    rnd = random.Random(2)
    outcomes = {"ok": 0, "ValueError": 0}
    for t in range(400):
        b = bytearray(buf)
        if t % 2:
            b = b[:rnd.randrange(1, len(b))]
        else:
            for _ in range(3):
                b[rnd.randrange(len(b))] = rnd.randrange(256)
        try:
            model = onnx_lite.parse_model(bytes(b))
            try:
                onnx_import.import_onnx(model)
            except (ValueError, KeyError, NotImplementedError):
                pass  # a well-formed protobuf that no longer describes a supported CNN
            outcomes["ok"] += 1
        except ValueError:
            outcomes["ValueError"] += 1
    assert outcomes["ValueError"] > 100 and sum(outcomes.values()) == 400
