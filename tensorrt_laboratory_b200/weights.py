"""Deterministic synthetic weights for raw Caffe layer lists.

The reference's benchmark engines carry random weights (reference ``models/README.md:6-7``,
``models/setup.py:53`` builds from the prototxt with no caffemodel), so the benchmark/parity weights
are DEFINED here, reproducibly, and consumed identically by the CPU oracle and the GPU engine
(SURVEY.md section 8(d)):

  ``numpy.random.default_rng(seed)``, layers visited in prototxt order;
  Convolution / InnerProduct  W ~ N(0, sqrt(2/(Cin*k*k)))  (He), bias ~ N(0, 0.01) where present;
  BatchNorm   mean ~ N(0, 0.1), var ~ U(0.5, 1.5);
  Scale       gamma ~ U(0.8, 1.2)  (U(0.1, 0.3) on the last BN of a bottleneck, ``*_branch2c``, so the
              residual stream stays bounded in fp16), beta ~ N(0, 0.1).
"""
from __future__ import annotations

import numpy as np

from .graph import infer_shapes


def random_weights(net: dict, seed: int = 0) -> dict:
    rng = np.random.default_rng(seed)
    shapes = infer_shapes(net)
    # infer_shapes reports the shape after the last writer; walk again to know each layer's input C,H,W
    cur = {net["input"]: tuple(net["input_dims"][1:])}
    out = {}
    for L in net["layers"]:
        t = L["type"]
        name = L["name"]
        c, h, w = cur[L["bottoms"][0]]
        if t == "Convolution":
            k = L["kernel_size"]
            std = np.sqrt(2.0 / (c * k * k))
            rec = {"W": (rng.standard_normal((L["num_output"], c, k, k)) * std).astype(np.float32)}
            if L["bias_term"]:
                rec["b"] = (rng.standard_normal(L["num_output"]) * 0.01).astype(np.float32)
            out[name] = rec
            from .graph import conv_out
            cur[L["tops"][0]] = (L["num_output"], conv_out(h, k, L["pad"], L["stride"]),
                                 conv_out(w, k, L["pad"], L["stride"]))
        elif t == "BatchNorm":
            out[name] = {
                "mean": (rng.standard_normal(c) * 0.1).astype(np.float32),
                "var": rng.uniform(0.5, 1.5, c).astype(np.float32),
            }
            cur[L["tops"][0]] = (c, h, w)
        elif t == "Scale":
            lo, hi = (0.1, 0.3) if name.endswith("_branch2c") else (0.8, 1.2)
            rec = {"gamma": rng.uniform(lo, hi, c).astype(np.float32)}
            if L.get("bias_term"):
                rec["beta"] = (rng.standard_normal(c) * 0.1).astype(np.float32)
            out[name] = rec
            cur[L["tops"][0]] = (c, h, w)
        elif t == "InnerProduct":
            kdim = c * h * w
            std = np.sqrt(2.0 / kdim)
            rec = {"W": (rng.standard_normal((L["num_output"], kdim)) * std).astype(np.float32)}
            if L["bias_term"]:
                rec["b"] = (rng.standard_normal(L["num_output"]) * 0.01).astype(np.float32)
            out[name] = rec
            cur[L["tops"][0]] = (L["num_output"], 1, 1)
        else:
            cur[L["tops"][0]] = shapes[L["tops"][0]]
    return out


def synthetic_input(batch: int, chw=(3, 224, 224), seed: int = 1234, ring: int = 1) -> np.ndarray:
    """fp32 NCHW N(0,1) input batches (the reference binding contract: fp32, batch-major NCHW)."""
    rng = np.random.default_rng(seed)
    shape = (ring, batch) + tuple(chw) if ring > 1 else (batch,) + tuple(chw)
    return rng.standard_normal(shape, dtype=np.float32)


def synthetic_image_u8(batch: int, src_hw=(224, 224), channels: int = 3, seed: int = 1234, ring: int = 1) -> np.ndarray:
    """uint8 [batch, src_h, src_w, C] images, uniform over 0..255 (what a JPEG decoder hands a uint8 image binding)."""
    rng = np.random.default_rng(seed)
    shape = (ring, batch) + tuple(src_hw) + (channels,) if ring > 1 else (batch,) + tuple(src_hw) + (channels,)
    return rng.integers(0, 256, size=shape, dtype=np.uint8)
