"""CPU: uint8 HWC image input bindings -- plan records, builder validation, the engine reader's checks of the
normalisation record, the numpy specification (builder.preprocess_u8), tools/build_engine.py and the TRTIS type."""
import os
import struct
import subprocess
import sys

import numpy as np
import pytest

from tensorrt_laboratory_b200 import builder, capi, graph, trtis, weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TV = dict(mean=builder.TORCHVISION_MEAN, std=builder.TORCHVISION_STD)
HDR, OP, BIND, TENS = builder._HEADER, builder._OP, builder._BINDING, builder._TENSOR


def _stem_low(cin=3, h=32, w=32):
    """One 7x7 / stride-2 convolution on a thin input: the fp16 builder packs it space-to-depth (the ResNet stem)."""
    net = builder.single_conv_net(cin, h, w, 64, 7, 2, 3)
    return graph.lower(net, weights.random_weights(net, 0))


def _offsets(blob):
    n_t, n_o, n_b = struct.unpack_from("<III", blob, 20)
    payload_off, payload_bytes = struct.unpack_from("<QQ", blob, 32)
    op0 = HDR.size + n_t * TENS.size
    b0 = op0 + n_o * OP.size
    return dict(op0=op0, bind0=b0, payload=payload_off, payload_bytes=payload_bytes, n_ops=n_o)


def _cast_op(blob):
    o = _offsets(blob)
    rec = OP.unpack_from(blob, o["op0"])
    assert rec[1] == builder.OP_INPUT_CAST
    return dict(zip(["w_off", "w_bytes", "b_off", "b_bytes"], rec[17:21]))


def _norm_rec(blob):
    c = _cast_op(blob)
    assert c["b_bytes"] == 48
    v = builder._INPUT_NORM.unpack_from(blob, _offsets(blob)["payload"] + c["b_off"])
    return dict(mean=np.float32(v[0:4]), inv_std=np.float32(v[4:8]), top=v[8], left=v[9], perm=v[10:14])


def test_u8_plan_records_round_trip(lib):
    img = dict(mean=(10.0, 20.0, 30.0), std=(2.0, 3.0, 7.0), reverse_channels=True, src_hw=(41, 38))
    blob = builder.build_plan(_stem_low(), builder.PREC_FP16, 4, input_dtype="u8", image=img)
    eng = capi.Engine(blob, inspect_only=True)
    try:
        b = eng.bindings[0]
        assert b["is_input"] and b["dtype"] == 5 and b["shape"] == (41, 38, 3) and b["item_bytes"] == 41 * 38 * 3
        assert b["np_dtype"] is np.uint8
    finally:
        eng.destroy()
    r = _norm_rec(blob)
    np.testing.assert_array_equal(r["mean"], np.float32([10, 20, 30, 0]))
    np.testing.assert_array_equal(r["inv_std"], np.float32([1 / 2.0, 1 / 3.0, 1 / 7.0, 0]))
    assert r["inv_std"][1] == np.float32(1.0 / 3.0)        # 1/std in float64, rounded once
    assert (r["top"], r["left"]) == (round(9 / 2), round(6 / 2)) == (4, 3)
    assert r["perm"] == (2, 1, 0, 0)


def test_existing_plans_unchanged_and_the_u8_plan_differs_only_locally():
    low = _stem_low()
    for prec, dtypes in ((builder.PREC_FP16, ("f32", "f16")), (builder.PREC_FP32, ("f32",))):
        for dt in dtypes:
            blob = builder.build_plan(low, prec, 4, input_dtype=dt)
            assert _cast_op(blob)["b_bytes"] == 0 and _cast_op(blob)["b_off"] == 0
            assert blob == builder.build_plan(low, prec, 4, input_dtype=dt, image=None)
    f32 = builder.build_plan(low, builder.PREC_FP16, 4)
    u8 = builder.build_plan(low, builder.PREC_FP16, 4, input_dtype="u8", image=TV)
    o = _offsets(f32)
    assert _offsets(u8)["payload"] == o["payload"] and len(u8) > len(f32)
    assert len(u8) - len(f32) <= 48 + 15 and u8[-48:] == builder._INPUT_NORM.pack(*_norm_rec(u8)["mean"], *_norm_rec(u8)["inv_std"],
                                                                                0, 0, 0, 1, 2, 0)
    allowed = set(range(40, 48))                                     # header payload_bytes
    allowed |= set(range(o["op0"], o["op0"] + OP.size))              # the input cast op record
    allowed |= set(range(o["bind0"], o["bind0"] + BIND.size))        # the input binding record
    diff = {i for i in range(len(f32)) if f32[i] != u8[i]}
    assert diff and diff <= allowed, sorted(diff - allowed)[:10]
    assert _offsets(u8)["payload_bytes"] == len(u8) - o["payload"]


def test_builder_rejects_what_the_engine_cannot_run():
    low = _stem_low()
    cases = {
        "fp32 engine": dict(precision=builder.PREC_FP32, input_dtype="u8", image=TV),
        "std 0": dict(input_dtype="u8", image=dict(mean=0, std=(1, 0, 1))),
        "crop larger than the source": dict(input_dtype="u8", image=dict(src_hw=(31, 40))),
        "image without u8": dict(input_dtype="f32", image=TV),
        "image with f16": dict(input_dtype="f16", image=TV),
        "wrong number of means": dict(input_dtype="u8", image=dict(mean=(1, 2))),
        "non-finite mean": dict(input_dtype="u8", image=dict(mean=float("nan"))),
        "unknown key": dict(input_dtype="u8", image=dict(scale=2)),
    }
    for name, kw in cases.items():
        prec = kw.pop("precision", builder.PREC_FP16)
        with pytest.raises(ValueError):
            builder.build_plan(low, prec, 4, **kw)
            pytest.fail(name)
    with pytest.raises(ValueError):                                   # C > 4
        builder.build_plan(_stem_low(cin=5), builder.PREC_FP16, 4, input_dtype="u8")
    with pytest.raises(ValueError):                                   # BGR order of a 4-channel input
        builder.build_plan(_stem_low(cin=4), builder.PREC_FP16, 4, input_dtype="u8", image=dict(reverse_channels=True))
    with pytest.raises(ValueError):
        builder.build_plan(low, builder.PREC_FP16, 4, input_dtype="u16")
    # INT8 engines have the fp16 stem: legal
    blob = builder.build_resnet_plan(50, builder.PREC_INT8, 8, input_dtype="u8", image=TV)
    assert _norm_rec(blob)["perm"] == (0, 1, 2, 0)


def _u8_blob():
    return builder.build_plan(_stem_low(), builder.PREC_FP16, 4, input_dtype="u8",
                              image=dict(mean=(1, 2, 3), std=(4, 5, 6), src_hw=(40, 36)))


def test_engine_reader_rejects_every_bad_normalisation_field(lib):
    blob = _u8_blob()
    o = _offsets(blob)
    cast = _cast_op(blob)
    rec = o["payload"] + cast["b_off"]
    cast_b = o["op0"] + 144                                            # OpRec.b_off
    bind = o["bind0"] + 64

    def mutated(offset, fmt, *vals, base=blob):
        bad = bytearray(base)
        struct.pack_into(fmt, bad, offset, *vals)
        return bytes(bad)

    capi.Engine(blob, inspect_only=True).destroy()                   # the unmodified plan loads
    f32 = builder.build_plan(_stem_low(), builder.PREC_FP16, 4)
    f32_fp32 = builder.build_plan(_stem_low(), builder.PREC_FP32, 4)
    cases = {
        "perm repeats a channel": mutated(rec + 40, "<4B", 0, 0, 2, 0),
        "perm names channel 3 of 3": mutated(rec + 40, "<4B", 0, 1, 3, 0),
        "perm entry past C not 0": mutated(rec + 40, "<4B", 0, 1, 2, 3),
        "inv_std entry past C not 0": mutated(rec + 16 + 12, "<f", 1.0),
        "crop_top outside the source": mutated(rec + 32, "<I", 40 - 32 + 1),
        "crop_left outside the source": mutated(rec + 36, "<I", 36 - 32 + 1),
        "crop_top wraps": mutated(rec + 32, "<I", 2 ** 32 - 1),
        "inv_std 0": mutated(rec + 16 + 4, "<f", 0.0),
        "inv_std nan": mutated(rec + 16, "<f", float("nan")),
        "inv_std inf": mutated(rec + 16 + 8, "<f", float("inf")),
        "mean inf": mutated(rec + 4, "<f", float("-inf")),
        "b_bytes 0 on a uint8 binding": mutated(cast_b + 8, "<Q", 0),
        "b_bytes 47": mutated(cast_b + 8, "<Q", 47),
        "record outside the payload": mutated(cast_b, "<Q", o["payload_bytes"] - 40),
        "record offset wraps": mutated(cast_b, "<Q", 2 ** 64 - 8),
        "b_bytes 48 on an fp32 binding": mutated(_offsets(f32)["op0"] + 152, "<Q", 48, base=f32),
        "uint8 binding of an fp32 engine": mutated(_offsets(f32_fp32)["bind0"] + 68, "<I", 5, base=f32_fp32),
        "uint8 output binding": mutated(o["bind0"] + BIND.size + 68, "<I", 5),
        "5 channels": mutated(bind + 16 + 8, "<i", 5),
        "channels disagree with the tensor": mutated(bind + 16 + 8, "<i", 2),
        "rank 2": mutated(bind + 12, "<I", 2),
        "source height 0": mutated(bind + 16, "<i", 0),
        "source smaller than the crop": mutated(bind + 16 + 4, "<i", 31),
        "dtype 4 (kBOOL)": mutated(bind + 4, "<I", 4),
    }
    for name, bad in cases.items():
        with pytest.raises(capi.B2Error) as ei:
            capi.Engine(bad, inspect_only=True)
        assert ei.value.code == 1, name


_U8_FUZZ = r"""
import random, struct, sys
sys.path.insert(0, sys.argv[1])
from tensorrt_laboratory_b200 import builder, capi, graph, weights
net = builder.single_conv_net(3, 32, 32, 64, 7, 2, 3)
blob = builder.build_plan(graph.lower(net, weights.random_weights(net, 0)), builder.PREC_FP16, 2, input_dtype="u8",
                          image=dict(mean=(1, 2, 3), std=(4, 5, 6), src_hw=(40, 36)))
n_t, n_o = struct.unpack_from("<II", blob, 20)
op0 = builder._HEADER.size + n_t * builder._TENSOR.size
bind0 = op0 + n_o * builder._OP.size
payload = struct.unpack_from("<Q", blob, 32)[0]
b_off = struct.unpack_from("<Q", blob, op0 + 144)[0]      # OpRec.b_off
regions = [(payload + b_off, 48), (op0, builder._OP.size), (bind0 + 64, 48)]   # record, cast op, binding fields
rnd = random.Random(int(sys.argv[2]))
ok = err = 0
for t in range(int(sys.argv[3])):
    b = bytearray(blob)
    for _ in range(rnd.randrange(1, 4)):
        start, size = regions[t % 3]
        i = start + rnd.randrange(size)
        b[i] = rnd.choice([0, 1, 2, 3, 4, 5, 0x7f, 0x80, 0xff, rnd.randrange(256)])
    try:
        capi.Engine(bytes(b), inspect_only=True).destroy()
        ok += 1
    except capi.B2Error:
        err += 1
print("ok", ok, "rejected", err)
"""


def test_normalisation_record_survives_random_corruption():
    """400 seeded random corruptions of a uint8 plan's normalisation record, input cast op and binding, parsed in a child
    process (a crash of the C parser fails the test instead of ending the run): each is accepted or rejected with B2_EINVAL."""
    out = subprocess.run([sys.executable, "-c", _U8_FUZZ, ROOT, "11", "400"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, (out.returncode, out.stderr[-1500:])
    ok, rejected = int(out.stdout.split()[1]), int(out.stdout.split()[3])
    assert ok + rejected == 400 and rejected > 100


def test_preprocess_u8_is_the_torchvision_formula():
    """((x / 255 - m) / s) in float64 against the float32 subtract-then-multiply of preprocess_u8.  The float32 means carry
    a representation error of up to half an ulp of ~124, which dominates close to the mean, so the bound is 2 float32 ulp
    of the largest value in the output."""
    rng = np.random.default_rng(3)
    x = rng.integers(0, 256, size=(2, 9, 8, 3), dtype=np.uint8)
    x[0, 0, :, :] = np.arange(24, dtype=np.uint8).reshape(8, 3) + 110      # values next to the means
    y = builder.preprocess_u8(x, (3, 9, 8), TV)
    assert y.dtype == np.float32 and y.shape == (2, 3, 9, 8)
    m, s = np.array([0.485, 0.456, 0.406]), np.array([0.229, 0.224, 0.225])
    ref = ((x.astype(np.float64) / 255 - m) / s).transpose(0, 3, 1, 2)
    tol = 2 * np.spacing(np.float32(np.abs(ref).max()))
    assert np.abs(y - ref).max() <= tol
    # exactly one subtract and one multiply in float32
    nrm = builder.image_norm(TV, (3, 9, 8))
    want = (x.astype(np.float32) - nrm["mean"]) * nrm["inv_std"]
    np.testing.assert_array_equal(y, want.transpose(0, 3, 1, 2))
    # BGR: output channel c is source channel 2 - c
    bgr = builder.preprocess_u8(x, (3, 9, 8), dict(mean=(104, 117, 123), std=1, reverse_channels=True))
    np.testing.assert_array_equal(bgr[:, 0], x[..., 2].astype(np.float32) - 104)


@pytest.mark.parametrize("src_hw,hw", [((256, 256), (224, 224)), ((241, 230), (224, 224)), ((5, 6), (2, 2)),
                                       ((7, 4), (4, 1)), ((224, 224), (224, 224))])
def test_center_crop_offsets_follow_round(src_hw, hw):
    top, left = builder.center_crop_offsets(src_hw, hw)
    assert (top, left) == (int(round((src_hw[0] - hw[0]) / 2)), int(round((src_hw[1] - hw[1]) / 2)))
    x = np.arange(src_hw[0] * src_hw[1], dtype=np.int64).reshape(src_hw) % 256
    img = np.repeat(x.astype(np.uint8)[None, :, :, None], 3, axis=3)
    y = builder.preprocess_u8(img, (3,) + hw, dict(src_hw=src_hw))
    np.testing.assert_array_equal(y[0, 1], x[top:top + hw[0], left:left + hw[1]].astype(np.float32))


def test_build_engine_tool_writes_the_builder_plan(tmp_path):
    out = tmp_path / "rn50_u8.plan"
    cmd = [sys.executable, os.path.join(ROOT, "tools", "build_engine.py"), "--model", "resnet50", "--input", "u8",
           "--mean", "123.675,116.28,103.53", "--std", "58.395,57.12,57.375", "--bgr", "--source-size", "256x240", "-o", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    img = dict(mean=(123.675, 116.28, 103.53), std=(58.395, 57.12, 57.375), reverse_channels=True, src_hw=(256, 240))
    assert out.read_bytes() == builder.build_resnet_plan(50, builder.PREC_FP16, 8, input_dtype="u8", image=img)
    r = subprocess.run(cmd[:2] + ["--model", "resnet50", "--bgr", "-o", str(tmp_path / "x.plan")], capture_output=True, text=True)
    assert r.returncode != 0 and "--input u8" in r.stderr


def test_capi_refuses_float_arrays_for_a_uint8_binding():
    x = np.zeros((2, 4, 4, 3), np.float32)
    with pytest.raises(TypeError):
        capi.as_input(x, np.uint8)
    u = np.zeros((2, 4, 4, 3), np.uint8)
    assert capi.as_input(u, np.uint8) is u or np.array_equal(capi.as_input(u, np.uint8), u)
    np.testing.assert_array_equal(capi.as_input(np.ones(3), np.float32), np.ones(3, np.float32))   # fp32 still casts


def test_trtis_uint8_model_input_wire_bytes():
    # model_config.proto: ModelInput{name=1, data_type=2 (TYPE_UINT8 = 2), format=3, dims=4 (packed int64)}
    m = trtis.message("ModelInput")(name="data", data_type=trtis.TYPE_UINT8)
    m.dims.extend([224, 224, 3])
    assert m.SerializeToString() == b"\x0a\x04data" + b"\x10\x02" + b"\x22\x05\xe0\x01\xe0\x01\x03"
    assert trtis._NP_OF[trtis.TYPE_UINT8] is np.uint8 and trtis._TYPE_OF[np.dtype(np.uint8)] == 2
