"""Plan builder: lowered graph (+ folded weights) -> B2ENGINE blob.

This is the offline step the reference performs with ``trtexec`` (reference ``models/setup.py:32-56``,
``examples/ONNX/resnet50/build.py:35-67``): it fixes precision and max batch, lays weights out in the
kernel-native format and writes one self-contained file that ``Runtime::DeserializeEngine`` loads
(reference ``trtlab/tensorrt/src/runtime.cc:62-95``).  Binary layout: ``csrc/plan_format.h``.
"""
from __future__ import annotations

import struct
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import graph as G

PREC_FP32, PREC_FP16, PREC_INT8 = 0, 1, 2
OP_INPUT_CAST, OP_CONV, OP_MAXPOOL, OP_AVGPOOL, OP_FC, OP_SOFTMAX, OP_OUTPUT_CAST, OP_QUANTIZE = range(8)
T_ACT, T_VEC = 0, 1
MAGIC = b"B2ENGINE"
VERSION = 1

_HEADER = struct.Struct("<8sIIIIIIQQ64s16x")
_TENSOR = struct.Struct("<64sIIIIIif4x")  # ... binding, scale (INT8 tensors: real value = q * scale; 0 = fp16 / fp32 tensor)
_OP = struct.Struct("<64sIiiiiIIIIIIIIIIIQQQQIIII")
_BINDING = struct.Struct("<64sIIiI8i16x")
_INPUT_NORM = struct.Struct("<4f4fII4B4x")  # mean[4], inv_std[4], crop_top, crop_left, perm[4]
assert _HEADER.size == 128 and _TENSOR.size == 96 and _OP.size == 176 and _BINDING.size == 128 and _INPUT_NORM.size == 48
DT_FLOAT, DT_HALF, DT_UINT8 = 0, 1, 5  # B2_DT_* of include/b200infer.h (5 = TensorRT's kUINT8)

# torchvision's ImageNet normalisation in pixel units (0..255): ToTensor's /255 folded into mean and std
TORCHVISION_MEAN = tuple(255.0 * v for v in (0.485, 0.456, 0.406))
TORCHVISION_STD = tuple(255.0 * v for v in (0.229, 0.224, 0.225))


def center_crop_offsets(src_hw: Sequence[int], hw: Sequence[int]):
    """(top, left) of an H x W crop centred in a src_h x src_w image, rounded like torchvision's CenterCrop."""
    return int(round((src_hw[0] - hw[0]) / 2.0)), int(round((src_hw[1] - hw[1]) / 2.0))


def image_norm(image: Optional[dict], chw: Sequence[int]) -> dict:
    """Validated normalisation of a uint8 image binding feeding a [C, H, W] input:
    ``image`` = dict(mean=..., std=..., reverse_channels=False, src_hw=None) in pixel units (a scalar or C values each;
    defaults mean 0, std 1, src_hw = (H, W)).  -> dict(mean, inv_std: float32 [C], perm, src_hw, top, left)."""
    c, h, w = (int(v) for v in chw)
    image = dict(image or {})
    unknown = set(image) - {"mean", "std", "reverse_channels", "src_hw"}
    if unknown:
        raise ValueError(f"image: unknown keys {sorted(unknown)}")
    if not 1 <= c <= 4:
        raise ValueError(f"uint8 image inputs carry 1..4 channels, this network takes {c}")

    def per_channel(key, dflt):
        v = np.asarray(image.get(key, dflt), dtype=np.float64).reshape(-1)
        if v.size == 1:
            v = np.repeat(v, c)
        if v.size != c or not np.all(np.isfinite(v)):
            raise ValueError(f"image: {key} needs 1 or {c} finite values, got {image.get(key)!r}")
        return v

    mean, std = per_channel("mean", 0.0), per_channel("std", 1.0)
    if np.any(std == 0):
        raise ValueError("image: std must be non-zero")
    inv_std = (1.0 / std).astype(np.float32)  # computed in float64, rounded once
    if not np.all(np.isfinite(inv_std)) or np.any(inv_std == 0):
        raise ValueError("image: 1/std is not a finite non-zero float32")
    reverse = bool(image.get("reverse_channels", False))
    if reverse and c != 3:
        raise ValueError("image: reverse_channels (RGB <-> BGR) needs 3 channels")
    src_hw = tuple(int(v) for v in (image.get("src_hw") or (h, w)))
    if len(src_hw) != 2 or src_hw[0] < h or src_hw[1] < w:
        raise ValueError(f"image: a {h}x{w} crop does not fit a source of {src_hw}")
    top, left = center_crop_offsets(src_hw, (h, w))
    return dict(mean=mean.astype(np.float32), inv_std=inv_std, perm=tuple(range(c))[::-1] if reverse else tuple(range(c)),
                src_hw=src_hw, top=top, left=left, chw=(c, h, w))


def preprocess_u8(x: np.ndarray, chw: Sequence[int], image: Optional[dict] = None) -> np.ndarray:
    """The semantics of a uint8 image binding, in numpy: uint8 [N, src_h, src_w, C] -> float32 [N, C, H, W], what the
    fp32 binding of the same engine receives.  Centre crop, channel order ``perm``, then per channel
    ``(float32(x) - mean) * inv_std`` in float32 (one subtract, one multiply); the engine's first kernel computes these exact
    values before rounding them to fp16."""
    nrm = image_norm(image, chw)
    c, h, w = nrm["chw"]
    x = np.asarray(x)
    if x.dtype != np.uint8 or x.ndim != 4 or x.shape[1:] != nrm["src_hw"] + (c,):
        raise ValueError(f"expected uint8 [N, {nrm['src_hw'][0]}, {nrm['src_hw'][1]}, {c}], got {x.dtype} {x.shape}")
    crop = x[:, nrm["top"]:nrm["top"] + h, nrm["left"]:nrm["left"] + w, :][..., list(nrm["perm"])].astype(np.float32)
    y = (crop - nrm["mean"]) * nrm["inv_std"]
    return np.ascontiguousarray(y.transpose(0, 3, 1, 2))


def _roundup(v: int, m: int) -> int:
    return (v + m - 1) // m * m


def phys_channels(c: int, precision: int) -> int:
    """Channel padding policy of activation tensors.  fp16/tcgen05: 8 (one 16-byte TMA element row,
    un-swizzled K-chunks) for thin inputs, otherwise a multiple of 64 (one 128-byte swizzle row)."""
    if precision == PREC_FP32:
        return c
    return 8 if c <= 8 else _roundup(c, 64)


def stem_s2d_transform(W: np.ndarray, k: int, pad: int, w_in: int):
    """Re-express a stride-2, thin-input (Cin <= 4) convolution on a horizontally space-to-depth packed input.

    The packed tensor holds pixel pairs: X2[n, h, w2, dw*4 + c] = X[n, c, h, 2*w2 + dw].  Column 2q - pad + s of
    the original becomes packed column q + a with a = floor((s - pad)/2), dw = (s - pad) mod 2, so the
    kxk / stride-2 conv turns into a k x kw2 conv with stride (2, 1) over 8 channels -- 4/7 of the im2col TMA
    loads and of the zero-padded K for the 7x7 stem.  Returns (W2 [cout, k, kw2, 8], kw2, pad_lo, pad_hi).
    """
    cout, kh, kw, cin = W.shape
    assert kh == kw == k and cin <= 4 and w_in % 2 == 0
    a_min = (0 - pad) // 2
    a_max = (k - 1 - pad) // 2
    kw2 = a_max - a_min + 1
    W2 = np.zeros((cout, kh, kw2, 8), dtype=W.dtype)
    for s_ in range(k):
        a = (s_ - pad) // 2
        dw = (s_ - pad) - 2 * a
        W2[:, :, a - a_min, dw * 4:dw * 4 + cin] = W[:, :, s_, :]
    q = (w_in + 2 * pad - k) // 2 + 1
    pad_lo = -a_min
    pad_hi = q - 1 + kw2 - w_in // 2 - pad_lo
    assert pad_hi >= 0
    return W2, kw2, pad_lo, pad_hi


def pack_weights_sw128(W: np.ndarray) -> np.ndarray:
    """[Cout_phys, K] fp16 (K % 64 == 0, Cout_phys % 32 == 0) -> blocks [K/64][Cout/32][32 rows][128 B] whose bytes are
    exactly what the kernel wants in shared memory for a 64-K weight sub-tile under the 128-byte swizzle (16-byte
    chunk j of row r sits at chunk j ^ (r % 8)).  The N tile of ANY width BN in {32, 64, 128} for k-block kb is then
    ONE contiguous run of BN*128 bytes = one `cp.async.bulk` instruction (instruction issue, ~200 cycles per TMA op
    from a single thread, is what paces the main loop -- profiles/phase_timing)."""
    cout, K = W.shape
    assert cout % 32 == 0 and K % 64 == 0 and W.dtype == np.float16
    blk = W.reshape(cout // 32, 32, K // 64, 8, 8)            # [nb, r, kb, chunk, elem]
    blk = blk.transpose(2, 0, 1, 3, 4)                         # [kb, nb, r, chunk, elem]
    out = np.empty_like(blk)
    r = np.arange(32)
    for j in range(8):
        out[:, :, r, j ^ (r % 8), :] = blk[:, :, r, j, :]
    return np.ascontiguousarray(out).reshape(-1)


def pack_weights_sw128_i8(W: np.ndarray) -> np.ndarray:
    """INT8 twin of :func:`pack_weights_sw128`: [Cout_phys, K] int8 (K % 128 == 0) -> blocks [K/128][Cout/32][32 rows][128 B],
    16-byte chunk j of row r at chunk j ^ (r % 8): the shared-memory image of a 128-K weight sub-tile."""
    cout, K = W.shape
    assert cout % 32 == 0 and K % 128 == 0 and W.dtype == np.int8
    blk = W.reshape(cout // 32, 32, K // 128, 8, 16).transpose(2, 0, 1, 3, 4)   # [kb, nb, r, chunk, 16 bytes]
    out = np.empty_like(blk)
    r = np.arange(32)
    for j in range(8):
        out[:, :, r, j ^ (r % 8), :] = blk[:, :, r, j, :]
    return np.ascontiguousarray(out).reshape(-1)


def _name(s: str) -> bytes:
    b = s.encode()
    if len(b) > 63:
        b = b[:63]
    return b


def build_plan(lowered: dict, precision: int = PREC_FP16, max_batch: int = 8,
               outputs: Optional[Sequence[str]] = None, name: Optional[str] = None, stem_s2d: bool = True,
               pack_weights: bool = True, input_dtype: str = "f32", image: Optional[dict] = None) -> bytes:
    """Serialize ``lowered`` (from :func:`graph.lower` with weights) into a plan blob.

    ``input_dtype``: "f32" = the reference's binding contract (pybind casts inputs to float, infer.cc:435-441);
    "f16" (fp16 engines only) = the secondary mode of SURVEY.md §8(d): half the H2D bytes per request;
    "u8" (fp16 and INT8 engines, 1..4 channels) = decoded images, uint8 [src_h, src_w, C] per item, a quarter of the fp32
    bytes: the input cast crops, orders and normalises them as :func:`preprocess_u8` with ``image`` (see
    :func:`image_norm`) specifies.

    ``outputs``: tensor names to expose as output bindings (default: the graph output).  4-D activation
    outputs get an ``OUTPUT_CAST`` to fp32 NCHW; vector outputs (fc / softmax) are written in place.
    """
    if precision not in (PREC_FP32, PREC_FP16, PREC_INT8):
        raise ValueError("precision must be PREC_FP32, PREC_FP16 or PREC_INT8")
    int8 = precision == PREC_INT8
    if int8 != bool(lowered.get("int8")):
        raise ValueError("PREC_INT8 takes a graph quantized by quantize.quantize_lowered (and only that precision does)")
    tscale = lowered.get("tensor_scales", {})   # INT8 tensors: name -> scale
    if int8:  # the fp16 part of an INT8 engine follows the fp16 engine's layout rules
        precision_fp = PREC_FP16
    else:
        precision_fp = precision
    wdtype = np.float16 if precision_fp == PREC_FP16 else np.float32
    outputs = list(outputs) if outputs else [lowered["output"]]
    shapes: Dict[str, tuple] = dict(lowered["tensors"])
    vec_tensors = {op["output"] for op in lowered["ops"] if op["type"] in (G.OP_FC, G.OP_SOFTMAX)}

    tensors: List[dict] = []
    tindex: Dict[str, int] = {}

    def add_tensor(tname: str) -> int:
        if tname in tindex:
            return tindex[tname]
        c, h, w = shapes[tname]
        if tname in vec_tensors:
            rec = dict(name=tname, kind=T_VEC, h=1, w=1, c=c * h * w, c_phys=c * h * w, binding=-1)
        elif tname in tscale:  # INT8 activations: one 128-byte swizzle row = 128 channels
            rec = dict(name=tname, kind=T_ACT, h=h, w=w, c=c, c_phys=_roundup(c, 128), binding=-1, scale=float(np.float32(tscale[tname])))
        else:
            rec = dict(name=tname, kind=T_ACT, h=h, w=w, c=c, c_phys=phys_channels(c, precision_fp), binding=-1)
        tindex[tname] = len(tensors)
        tensors.append(rec)
        return tindex[tname]

    bindings: List[dict] = []
    ops: List[dict] = []
    payload = bytearray()

    def add_payload(arr: np.ndarray):
        while len(payload) % 256:
            payload.append(0)
        off = len(payload)
        raw = np.ascontiguousarray(arr).tobytes()
        payload.extend(raw)
        return off, len(raw)

    # input binding + cast
    cin, hin, win = lowered["input_shape"]
    t_in = add_tensor(lowered["input"])
    if input_dtype not in ("f32", "f16", "u8") or (input_dtype != "f32" and precision_fp != PREC_FP16):
        raise ValueError("input_dtype is 'f32' (the reference's binding contract) or, for fp16 / INT8 engines, 'f16' or 'u8'")
    if image is not None and input_dtype != "u8":
        raise ValueError("image= describes a uint8 input binding: pass input_dtype='u8'")
    norm = image_norm(image, (cin, hin, win)) if input_dtype == "u8" else None
    if norm is not None:
        bindings.append(dict(name=lowered["input"], is_input=1, dtype=DT_UINT8, tensor=t_in, dims=[*norm["src_hw"], cin]))
    else:
        bindings.append(dict(name=lowered["input"], is_input=1, dtype=DT_HALF if input_dtype == "f16" else DT_FLOAT, tensor=t_in,
                             dims=[cin, hin, win]))
    ops.append(dict(name="cast:" + lowered["input"], type=OP_INPUT_CAST, inp=-1, res=-1, out=t_in, binding=0))
    # fp16 stem: a stride-2 conv that is the only reader of a thin (<= 4 channel) even-width input runs on a
    # horizontally space-to-depth packed copy of the input (see stem_s2d_transform)
    readers = [o for o in lowered["ops"] if o["input"] == lowered["input"] or o.get("residual") == lowered["input"]]
    s2d_op = None
    if (precision_fp == PREC_FP16 and stem_s2d and len(readers) == 1 and readers[0]["type"] == G.OP_CONV
            and readers[0]["stride"] == 2 and cin <= 4 and win % 2 == 0 and lowered["input"] not in outputs
            and readers[0]["k"] >= 3):
        s2d_op = readers[0]
        _, _, s2d_lo, s2d_hi = stem_s2d_transform(s2d_op["W"], s2d_op["k"], s2d_op["pad"], win)
        # the horizontal padding is made PHYSICAL (zero pixels written by the cast), so the conv has pad_w = 0 and its
        # kw taps are contiguous in memory: the engine reads a whole filter row as one 64-byte TMA "pixel"
        tensors[t_in].update(w=win // 2 + s2d_lo + s2d_hi, c=8, c_phys=8)
        ops[0].update(k=2, pad=s2d_lo, stride=s2d_hi)

    for op in lowered["ops"]:
        t = op["type"]
        ti = add_tensor(op["input"])
        to = add_tensor(op["output"])
        rec = dict(name=op["name"], inp=ti, res=-1, out=to, binding=-1)
        if t == "quantize":
            rec.update(type=OP_QUANTIZE)
        elif t == G.OP_CONV and op.get("int8"):
            cin_phys, cout_phys = tensors[ti]["c_phys"], tensors[to]["c_phys"]
            k = op["k"]
            taps = k * k
            Wq = np.zeros((cout_phys, taps, cin_phys), dtype=np.int8)
            Wq[:op["cout"], :, :op["cin"]] = op["Wq"].reshape(op["cout"], taps, op["cin"])
            w_off, w_bytes = add_payload(pack_weights_sw128_i8(Wq.reshape(cout_phys, taps * cin_phys)))
            rq = np.zeros(2 * cout_phys + 4, dtype=np.float32)   # [m | b | r 0 0 0]; padded channels requantise to 0
            rq[:op["cout"]] = op["m"]
            rq[cout_phys:cout_phys + op["cout"]] = op["b"]
            rq[2 * cout_phys] = op["r"] if op["r"] is not None else 0.0
            b_off, b_bytes = add_payload(rq)
            rec.update(type=OP_CONV, k=k, stride=op["stride"], pad=op["pad"], relu=int(op["relu"]) | 2 | 4,
                       cin=op["cin"], cout=op["cout"], cin_phys=cin_phys, cout_phys=cout_phys, taps=taps, taps_phys=taps,
                       w_off=w_off, w_bytes=w_bytes, b_off=b_off, b_bytes=b_bytes)
            if op["residual"] is not None:
                rec["res"] = add_tensor(op["residual"])
        elif t == G.OP_CONV:
            if "W" not in op:
                raise ValueError(f"conv {op['name']}: lowered graph carries no weights")
            cin_phys = tensors[ti]["c_phys"]
            cout_phys = tensors[to]["c_phys"]
            k = op["k"]
            Wsrc, cin_eff, extra = op["W"], op["cin"], {}
            taps = k * k
            if op is s2d_op:
                Wsrc, kw2, pad_lo, pad_hi = stem_s2d_transform(op["W"], k, op["pad"], win)
                cin_eff, taps = 8, k * kw2
                extra = dict(kw=kw2, stride_w=1, pad_w_lo=0, pad_w_hi=0, ceil_mode=op["cin"] * k * k)
            taps_phys = _roundup(taps, 2) if (precision_fp == PREC_FP16 and cin_phys == 8) else taps
            W = np.zeros((cout_phys, taps_phys, cin_phys), dtype=np.float32)
            W[:op["cout"], :taps, :cin_eff] = Wsrc.reshape(op["cout"], taps, cin_eff)
            bias = np.zeros(cout_phys, dtype=np.float32)
            bias[:op["cout"]] = op["bias"]
            packed = precision_fp == PREC_FP16 and cin_phys % 64 == 0 and cout_phys % 32 == 0 and pack_weights
            if packed:
                w_off, w_bytes = add_payload(pack_weights_sw128(W.astype(np.float16).reshape(cout_phys, taps_phys * cin_phys)))
            else:
                w_off, w_bytes = add_payload(W.astype(wdtype))
            b_off, b_bytes = add_payload(bias)
            rec.update(type=OP_CONV, k=k, stride=op["stride"], pad=op["pad"], relu=int(op["relu"]) | (2 if packed else 0),
                       cin=cin_eff, cout=op["cout"], cin_phys=cin_phys, cout_phys=cout_phys,
                       taps=taps, taps_phys=taps_phys, w_off=w_off, w_bytes=w_bytes, b_off=b_off, b_bytes=b_bytes)
            rec.update(extra)
            if op["residual"] is not None:
                rec["res"] = add_tensor(op["residual"])
        elif t == G.OP_MAXPOOL:
            rec.update(type=OP_MAXPOOL, k=op["k"], stride=op["stride"], pad=op["pad"], ceil_mode=int(op["ceil_mode"]))
        elif t == G.OP_AVGPOOL:
            rec.update(type=OP_AVGPOOL, k=op["k"], stride=op["stride"])
        elif t == G.OP_FC:
            c, h, w = op["in_chw"]
            c_phys = tensors[ti]["c_phys"]
            Wf = np.zeros((op["cout"], h * w, c_phys), dtype=np.float32)
            Wf[:, :, :c] = op["W"].reshape(op["cout"], h * w, c)
            w_off, w_bytes = add_payload(Wf.astype(wdtype))
            b_off, b_bytes = add_payload(op["bias"].astype(np.float32))
            rec.update(type=OP_FC, cin=op["cin"], cout=op["cout"], cin_phys=h * w * c_phys, cout_phys=op["cout"],
                       w_off=w_off, w_bytes=w_bytes, b_off=b_off, b_bytes=b_bytes)
        elif t == G.OP_SOFTMAX:
            rec.update(type=OP_SOFTMAX)
        else:
            raise ValueError(f"unsupported lowered op {t}")
        ops.append(rec)

    for oname in outputs:
        if oname not in tindex:
            raise ValueError(f"output tensor {oname!r} is not produced by the graph")
        ti = tindex[oname]
        trec = tensors[ti]
        bidx = len(bindings)
        if trec["kind"] == T_VEC:
            if trec["binding"] >= 0:
                raise ValueError(f"tensor {oname} bound twice")
            trec["binding"] = bidx
            bindings.append(dict(name=oname, is_input=0, dtype=0, tensor=ti, dims=[trec["c"]]))
        else:
            bindings.append(dict(name=oname, is_input=0, dtype=0, tensor=ti, dims=[trec["c"], trec["h"], trec["w"]]))
            ops.append(dict(name="cast:" + oname, type=OP_OUTPUT_CAST, inp=ti, res=-1, out=-1, binding=bidx))

    if norm is not None:  # behind every weight, so the weight offsets are those of the fp32-binding plan
        while len(payload) % 16:
            payload.append(0)
        perm = list(norm["perm"]) + [0] * (4 - cin)
        ops[0].update(b_off=len(payload), b_bytes=_INPUT_NORM.size)
        payload.extend(_INPUT_NORM.pack(*np.pad(norm["mean"], (0, 4 - cin)).tolist(), *np.pad(norm["inv_std"], (0, 4 - cin)).tolist(),
                                        norm["top"], norm["left"], *perm))

    tables = _HEADER.size + len(tensors) * _TENSOR.size + len(ops) * _OP.size + len(bindings) * _BINDING.size
    payload_offset = _roundup(tables, 256)
    blob = bytearray()
    blob += _HEADER.pack(MAGIC, VERSION, precision, max_batch, len(tensors), len(ops), len(bindings),
                         payload_offset, len(payload), _name(name or lowered["name"]))
    for t in tensors:
        blob += _TENSOR.pack(_name(t["name"]), t["kind"], t["h"], t["w"], t["c"], t["c_phys"], t["binding"], t.get("scale", 0.0))
    for o in ops:
        blob += _OP.pack(_name(o["name"]), o["type"], o["inp"], o["res"], o["out"], o["binding"],
                         o.get("k", 0), o.get("stride", 0), o.get("pad", 0), o.get("relu", 0), o.get("ceil_mode", 0),
                         o.get("cin", 0), o.get("cout", 0), o.get("cin_phys", 0), o.get("cout_phys", 0),
                         o.get("taps", 0), o.get("taps_phys", 0),
                         o.get("w_off", 0), o.get("w_bytes", 0), o.get("b_off", 0), o.get("b_bytes", 0),
                         o.get("kw", 0), o.get("stride_w", 0), o.get("pad_w_lo", 0), o.get("pad_w_hi", 0))
    for b in bindings:
        dims = list(b["dims"]) + [0] * (8 - len(b["dims"]))
        blob += _BINDING.pack(_name(b["name"]), b["is_input"], b["dtype"], b["tensor"], len(b["dims"]), *dims)
    blob += b"\0" * (payload_offset - len(blob))
    blob += payload
    return bytes(blob)


def resnet_lowered(depth: int = 50, precision: int = PREC_FP16, seed: int = 0, calib_batch: int = 8,
                   image: Optional[dict] = None) -> dict:
    """Generated Caffe-v1 ResNet + deterministic weights, lowered.  PREC_INT8: quantized, calibrated (max-abs) on
    ``calib_batch`` synthetic inputs (seed 4321) -- with ``image``, on :func:`preprocess_u8` of synthetic uint8 images, the
    values a uint8 binding feeds the network."""
    from . import weights as Wt
    net = G.resnet_caffe(depth)
    low = G.lower(net, Wt.random_weights(net, seed))
    if precision == PREC_INT8:
        from . import quantize
        if image is None:
            calib = Wt.synthetic_input(calib_batch, seed=4321)
        else:
            chw = low["input_shape"]
            src_hw = image_norm(image, chw)["src_hw"]
            calib = preprocess_u8(Wt.synthetic_image_u8(calib_batch, src_hw, chw[0], seed=4321), chw, image)
        low = quantize.quantize_lowered(low, calib)
    return low


def build_resnet_plan(depth: int = 50, precision: int = PREC_FP16, max_batch: int = 8, seed: int = 0,
                      input_dtype: str = "f32", calib_batch: int = 8, image: Optional[dict] = None) -> bytes:
    """Convenience: :func:`resnet_lowered` -> plan (``input_dtype`` / ``image`` as in :func:`build_plan`)."""
    low = resnet_lowered(depth, precision, seed, calib_batch, image if input_dtype == "u8" else None)
    return build_plan(low, precision, max_batch, input_dtype=input_dtype, image=image)


def single_conv_net(cin: int, h: int, w: int, cout: int, k: int, stride: int, pad: int, relu: bool = True,
                    residual: bool = False, bias: bool = True) -> dict:
    """Raw layer list of a one-convolution network (kernel-level parity tests go through the public ABI).
    With ``residual`` the net is  y = relu(conv_b(x) + conv_a(x))  so the fused add path is exercised."""
    L = []
    if residual:
        L.append(dict(name="short", type="Convolution", bottoms=["data"], tops=["short"], num_output=cout,
                      kernel_size=k, pad=pad, stride=stride, bias_term=bias))
    L.append(dict(name="conv", type="Convolution", bottoms=["data"], tops=["conv"], num_output=cout,
                  kernel_size=k, pad=pad, stride=stride, bias_term=bias))
    top = "conv"
    if residual:
        L.append(dict(name="sum", type="Eltwise", bottoms=["short", "conv"], tops=["sum"], operation="SUM"))
        top = "sum"
    if relu:
        L.append(dict(name="relu", type="ReLU", bottoms=[top], tops=[top]))
    return {"name": f"conv{k}x{k}s{stride}_{cin}x{h}x{w}_{cout}", "input": "data", "input_dims": [1, cin, h, w],
            "layers": L}


def attach_tactics(blob: bytes, tactics: np.ndarray) -> bytes:
    """Append a tactic table (``capi.Engine.tactics()`` after ``Engine.tune()``: [n, 10] uint32 records
    {op, batch, bn, stages, splits, sps, ws, cn, halo, 0}) to a plan blob -- the role of the tactics a TensorRT plan file
    carries (reference models/setup.py:53-55: trtexec tunes offline).  An engine deserialized from the result never tunes."""
    tactics = np.ascontiguousarray(tactics, dtype=np.uint32).reshape(-1, 10)
    hdr = list(_HEADER.unpack_from(blob, 0))
    base = blob
    old_n, _, old_off = struct.unpack_from("<IIQ", blob, _HEADER.size - 16)
    if old_n:  # replace an existing table
        base = blob[:old_off]
    off = (len(base) + 63) // 64 * 64
    out = bytearray(base) + bytes(off - len(base)) + tactics.tobytes()
    struct.pack_into("<IIQ", out, _HEADER.size - 16, tactics.shape[0], 0, off)
    del hdr
    return bytes(out)
