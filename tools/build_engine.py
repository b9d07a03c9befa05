#!/usr/bin/env python
"""Build a B2ENGINE plan file -- the step the reference performs with `trtexec` (reference models/setup.py:32-56,
examples/ONNX/resnet50/build.py:35-67).

  python tools/build_engine.py --model resnet50 --precision fp16 --batch 8 -o rn50_b8_fp16.plan
  python tools/build_engine.py --prototxt /path/ResNet-152-deploy.prototxt --precision fp16 --batch 32 -o rn152.plan
  python tools/build_engine.py --model mnist --precision fp32 --batch 1 -o mnist.plan
  python tools/build_engine.py --prototxt deploy.prototxt --caffemodel weights.caffemodel --precision int8 --batch 32 -o rn.plan
  python tools/build_engine.py --model resnet50 --batch 8 --tune -o rn50_tuned.plan      (on a GPU box: tactics in the file)
Weights: deterministic synthetic weights (the reference's benchmark engines are weightless too, models/README.md:6-7),
unless --caffemodel names a binary NetParameter (trtexec --model=...); MNIST and --onnx carry their own weights.
--precision int8: post-training quantization, max-abs calibration on --calib (an .npy [N,C,H,W] fp32) or on synthetic images.
--input u8: the input binding takes decoded images, uint8 [H, W, C] per item (a quarter of the fp32 bytes); the engine's
first kernel centre-crops them from --source-size, reorders RGB -> BGR with --bgr and normalises (x - mean) / std with
--mean / --std in pixel units (0..255), e.g. torchvision: --mean 123.675,116.28,103.53 --std 58.395,57.12,57.375.
  python tools/build_engine.py --model resnet50 --input u8 --mean 123.675,116.28,103.53 --std 58.395,57.12,57.375 \
      --source-size 256x256 -o rn50_u8.plan
--tune: time the kernel configurations on this machine's GPU (what trtexec does while building) and store the tactic table
in the plan file; an engine deserialized from it never tunes at load.
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tensorrt_laboratory_b200 import builder, graph, weights  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", choices=["resnet50", "resnet152", "mnist"])
    ap.add_argument("--prototxt")
    ap.add_argument("--onnx", help="ONNX CNN classifier (Conv / BatchNormalization / Relu / Add / MaxPool / AveragePool / "
                                   "GlobalAveragePool / Flatten / Reshape / Gemm / MatMul / Softmax), e.g. an ONNX-zoo ResNet")
    ap.add_argument("--precision", choices=["fp16", "fp32", "int8"], default="fp16")
    ap.add_argument("--caffemodel", help="binary caffe NetParameter with the weights of --prototxt / --model resnetNN")
    ap.add_argument("--calib", help="int8: .npy of calibration inputs [N, C, H, W] fp32 (default: 8 synthetic images)")
    ap.add_argument("--tune", action="store_true", help="needs a GPU: tune kernel tactics now and embed them in the plan")
    ap.add_argument("--tune-all-batches", action="store_true", help="with --tune: one tactic set per batch size 1..max")
    ap.add_argument("--input", choices=["f32", "f16", "u8"], default="f32",
                    help="input binding dtype: fp32 NCHW (default), fp16 NCHW (fp16 engines) or uint8 HWC images (fp16 / int8)")
    ap.add_argument("--mean", help="--input u8: per-channel mean in pixel units, comma separated (default 0)")
    ap.add_argument("--std", help="--input u8: per-channel std in pixel units, comma separated (default 1)")
    ap.add_argument("--bgr", action="store_true", help="--input u8: the network takes the channels in reverse (BGR) order")
    ap.add_argument("--source-size", help="--input u8: HxW of the images; the network input is centre-cropped from them")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("-o", "--output", required=True)
    a = ap.parse_args()
    prec = {"fp16": builder.PREC_FP16, "fp32": builder.PREC_FP32, "int8": builder.PREC_INT8}[a.precision]
    image = None
    if a.input == "u8":
        image = dict(reverse_channels=a.bgr)
        if a.mean:
            image["mean"] = [float(v) for v in a.mean.split(",")]
        if a.std:
            image["std"] = [float(v) for v in a.std.split(",")]
        if a.source_size:
            image["src_hw"] = tuple(int(v) for v in a.source_size.lower().split("x"))
    elif a.mean or a.std or a.bgr or a.source_size:
        ap.error("--mean / --std / --bgr / --source-size describe a uint8 input: add --input u8")

    def weights_for(net):
        if a.caffemodel:
            from tensorrt_laboratory_b200 import caffemodel
            return caffemodel.load_caffemodel(a.caffemodel, net)
        return weights.random_weights(net, a.seed)

    if a.prototxt:
        with open(a.prototxt) as f:
            net = graph.parse_prototxt(f.read())
        wts = weights_for(net)
    elif a.onnx:
        from tensorrt_laboratory_b200 import onnx_import, onnx_lite
        net, wts = onnx_import.import_onnx(onnx_lite.load_model(a.onnx), name=os.path.splitext(os.path.basename(a.onnx))[0])
    elif a.model == "mnist":
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        from tests import helpers
        net, wts, _, _ = helpers.load_mnist_golden()
    else:
        net = graph.resnet_caffe(int(a.model[6:]))
        wts = weights_for(net)
    low = graph.lower(net, wts)
    if prec == builder.PREC_INT8:
        import numpy as np
        from tensorrt_laboratory_b200 import quantize
        chw = tuple(net["input_dims"][1:])
        if a.calib:
            calib = np.load(a.calib).astype(np.float32)
        elif image is not None:  # calibrate on what the uint8 binding feeds the network
            src_hw = builder.image_norm(image, chw)["src_hw"]
            calib = builder.preprocess_u8(weights.synthetic_image_u8(8, src_hw, chw[0], seed=4321), chw, image)
        else:
            calib = weights.synthetic_input(8, chw=chw, seed=4321)
        low = quantize.quantize_lowered(low, calib)
    blob = builder.build_plan(low, prec, a.batch, input_dtype=a.input, image=image)
    if a.tune:
        from tensorrt_laboratory_b200 import capi
        eng = capi.Engine(blob)
        n = eng.tune(streams=4, all_batches=a.tune_all_batches)
        blob = builder.attach_tactics(blob, eng.tactics())
        print(f"tuned {n} tactics on this GPU")
    with open(a.output, "wb") as f:
        f.write(blob)
    print(f"wrote {a.output}: {len(blob) / 1e6:.1f} MB, {net['name']}, {a.precision}, max batch {a.batch}")


if __name__ == "__main__":
    main()
