"""CPU: model front-ends (prototxt parser, generated ResNets, ONNX-lite) and the lowering pass."""
import gzip
import os

import numpy as np
import pytest

from tensorrt_laboratory_b200 import graph, onnx_lite, weights
from tests.helpers import GOLDEN


@pytest.mark.parametrize("depth,nlayers", [(50, 228), (152, 670)])
def test_generated_resnet_equals_reference_prototxt(depth, nlayers):
    with gzip.open(os.path.join(GOLDEN, f"ResNet-{depth}-deploy.prototxt.gz"), "rt") as f:
        parsed = graph.parse_prototxt(f.read())
    gen = graph.resnet_caffe(depth)
    assert parsed["input_dims"] == gen["input_dims"] == [1, 3, 224, 224]
    assert len(parsed["layers"]) == len(gen["layers"]) == nlayers
    for a, b in zip(parsed["layers"], gen["layers"]):
        for k in set(a) | set(b):
            if k in ("eps", "operation"):
                continue
            assert a.get(k) == b.get(k), (a["name"], k)


def test_parser_on_inline_prototxt():
    txt = '''name: "t" input: "data" input_dim: 1 input_dim: 3 input_dim: 8 input_dim: 8
    layer { bottom: "data" top: "c" name: "c" type: "Convolution"
            convolution_param { num_output: 4 kernel_size: 3 pad: 1 stride: 2 bias_term: false } }  # comment
    layer { bottom: "c" top: "c" name: "r" type: "ReLU" }
    layer { bottom: "c" top: "p" name: "p" type: "Pooling" pooling_param { kernel_size: 2 stride: 2 pool: AVE } }'''
    net = graph.parse_prototxt(txt)
    c = net["layers"][0]
    assert (c["num_output"], c["kernel_size"], c["pad"], c["stride"], c["bias_term"]) == (4, 3, 1, 2, False)
    assert net["layers"][2]["pool"] == "AVE"
    assert graph.infer_shapes(net)["p"] == (4, 2, 2)
    with pytest.raises(ValueError):
        graph.parse_prototxt('layer { name: "x" type: "LSTM" }')


def test_resnet50_known_layers_and_lowering():
    net = graph.resnet_caffe(50)
    by = {L["name"]: L for L in net["layers"]}
    assert (by["conv1"]["kernel_size"], by["conv1"]["stride"], by["conv1"]["pad"], by["conv1"]["bias_term"]) == (7, 2, 3, True)
    assert by["res3a_branch1"]["stride"] == 2 and by["res3a_branch2a"]["stride"] == 2  # Caffe-v1: stride on the 1x1
    assert by["res3a_branch2b"]["stride"] == 1 and by["res2a_branch2a"]["stride"] == 1
    shapes = graph.infer_shapes(net)
    assert shapes["pool1"] == (64, 56, 56)  # ceil-mode pooling
    assert shapes["res5c"] == (2048, 7, 7) and shapes["prob"] == (1000, 1, 1)
    low = graph.lower(net)
    kinds = [o["type"] for o in low["ops"]]
    assert kinds.count("conv") == 53 and kinds.count("maxpool") == 1 and kinds.count("avgpool") == 1
    assert kinds[-2:] == ["fc", "softmax"]
    assert abs(graph.conv_flops(low) - 7.716e9) < 1e6  # SURVEY.md 8(d): 7.716 GFLOP / image
    fused = [o for o in low["ops"] if o["type"] == "conv" and o["residual"]]
    assert len(fused) == 16 and all(o["name"].endswith("branch2c") and o["relu"] for o in fused)
    assert low["ops"][5]["residual"] == "res2a_branch1" and low["ops"][5]["output"] == "res2a"


def test_resnet152_flops():
    low = graph.lower(graph.resnet_caffe(152))
    assert abs(graph.conv_flops(low) - 22.565e9) < 2e6
    assert sum(o["type"] == "conv" for o in low["ops"]) == 155


def test_weights_are_deterministic_and_specified():
    net = graph.resnet_caffe(50)
    a, b = weights.random_weights(net, 0), weights.random_weights(net, 0)
    assert all(np.array_equal(a[k][f], b[k][f]) for k in a for f in a[k])
    c = weights.random_weights(net, 1)
    assert not np.array_equal(a["conv1"]["W"], c["conv1"]["W"])
    assert a["conv1"]["W"].shape == (64, 3, 7, 7) and "b" in a["conv1"] and "b" not in a["res2a_branch1"]
    g = a["scale2a_branch2c"]["gamma"]
    assert 0.1 <= g.min() and g.max() <= 0.3
    g = a["scale2a_branch2a"]["gamma"]
    assert 0.8 <= g.min() and g.max() <= 1.2
    x = weights.synthetic_input(2, ring=3)
    assert x.shape == (3, 2, 3, 224, 224) and x.dtype == np.float32


def test_onnx_lite_reads_reference_mnist():
    model = onnx_lite.load_model(os.path.join(GOLDEN, "mnist_v1_3_model.onnx"))
    assert [n["op"] for n in model["nodes"]] == ["Reshape", "Conv", "Add", "Relu", "MaxPool", "Conv", "Add", "Relu",
                                                 "MaxPool", "Reshape", "MatMul", "Add"]
    net, w = onnx_lite.mnist_to_caffe_like(model)
    assert graph.infer_shapes(net)[net["layers"][-1]["tops"][0]] == (10, 1, 1)
    x = onnx_lite.load_tensor(os.path.join(GOLDEN, "mnist_v1_3_input_0.pb"))
    assert x.shape == (1, 1, 28, 28)
    # the committed fixture is exactly what the decoder produces
    from tests import helpers
    _, gw, gx, _ = helpers.load_mnist_golden()
    np.testing.assert_array_equal(gx[0], x)
    for lname in w:
        for f in w[lname]:
            np.testing.assert_array_equal(gw[lname][f], w[lname][f])


def test_same_upper_padding():
    assert onnx_lite.same_upper_pads(28, 5) == (2, 2)
    assert onnx_lite.same_upper_pads(28, 4) == (1, 2)  # extra pad at the end
    assert onnx_lite.same_upper_pads(7, 3, 2) == (1, 1)
