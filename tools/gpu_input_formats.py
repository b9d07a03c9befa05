#!/usr/bin/env python
"""End-to-end cost of the input binding format: fp32 NCHW, fp16 NCHW and uint8 HWC images (one GPU run, one JSON).

  python tools/gpu_input_formats.py --out profiles/input_formats_<tag>.json [--steps 20]

* e2e: the closed loop of bench.py's e2e leg (InferenceManager, 4 contexts, 8 pinned Buffers, batch 8, ResNet-50 fp16;
  InferBench::Run, median of 5 consecutive windows of --steps completions) for the three bindings of ONE engine (same
  weights and tactic table), alternated f32, f16, u8, f32, f16, u8.  Inputs: 32 batches of seeded uint8 images; the
  fp32 / fp16 legs feed builder.preprocess_u8 of the same images.
* zero copy: the u8 leg once more with TRTLAB_ZERO_COPY_INPUT=1 (read once per process: a child process).
* cast: per-launch device time of the input cast from Session.profile(8) (serialised launches, CUDA events), median of
  30 forward passes, fp32 and u8 engines.
* configs[2]: ResNet-152 INT8 batch 32, single-image requests flooded through BatchedInferRunner (bench.py run_config2),
  fp32 against u8 bindings of one engine.
The card's name, power limit and maximum SM clock are read (never set) with nvidia-smi in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tensorrt_laboratory_b200 import builder, capi, weights  # noqa: E402

BATCH, CONTEXTS, BUFFERS, RING = 8, 4, 8, 32
TV = dict(mean=builder.TORCHVISION_MEAN, std=builder.TORCHVISION_STD)
CHW = (3, 224, 224)


def card():
    q = "name,power.limit,clocks.max.sm,driver_version"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), (v.strip() for v in out.split(","))))
    except Exception as ex:  # reported, not guessed
        return {"error": f"nvidia-smi: {ex}"}


def rn50_blobs():
    """The three bindings of one ResNet-50 fp16 engine, all carrying the tactic table tuned once on this GPU."""
    low = builder.resnet_lowered(50, builder.PREC_FP16)
    blobs = {dt: builder.build_plan(low, builder.PREC_FP16, BATCH, input_dtype=dt, image=TV if dt == "u8" else None)
             for dt in ("f32", "f16", "u8")}
    eng = capi.Engine(blobs["f32"])
    eng.tune(streams=CONTEXTS)
    tactics = eng.tactics()
    eng.destroy()
    return {dt: builder.attach_tactics(b, tactics) for dt, b in blobs.items()}


def rings():
    u8 = weights.synthetic_image_u8(BATCH, (224, 224), seed=1234, ring=RING)
    f32 = np.stack([builder.preprocess_u8(r, CHW, TV) for r in u8])
    return {"u8": u8, "f32": f32, "f16": f32.astype(np.float16)}


def e2e_leg(blob, ring, steps):
    warm = max(3 * CONTEXTS, 2 * BUFFERS * 2)
    mgr = capi.InferenceManager(CONTEXTS, BUFFERS, pre_threads=1, cuda_threads=1, post_threads=3)
    try:
        mgr.register_model("rn50", blob)
        mgr.update_resources()
        mgr.prefill_inputs("rn50", ring[:BUFFERS])
        mgr.bench("rn50", BATCH, seconds=600.0, max_batches=warm, want_latencies=False)
        res, lats = mgr.bench("rn50", BATCH, seconds=600.0, max_batches=steps, want_latencies=True)
        win_s, win_lat = mgr.bench_windows("rn50", BATCH, warm=warm, steps=steps, windows=5, cool=2 * BUFFERS)
    finally:
        mgr.close()
    rates = [steps * BATCH / float(w) for w in win_s]
    return {"value": float(np.median(rates)), "windows": rates, "p50_ms": float(np.percentile(win_lat, 50) * 1e3),
            "p99_ms": float(np.percentile(win_lat, 99) * 1e3), "bracketed": steps * BATCH / res["kWalltime"],
            "h2d_bytes_per_batch": int(ring[0].nbytes)}


def cast_time(blob, x, reps=30):
    eng = capi.Engine(blob)
    sess = capi.Session(eng)
    try:
        sess.infer(x)
        ms = []
        for _ in range(reps):
            prof = sess.profile(BATCH)
            assert prof[0]["name"].startswith("input_cast:"), prof[0]["name"]
            ms.append(prof[0]["ms"])
        return {"name": prof[0]["name"], "median_us": float(np.median(ms) * 1e3), "min_us": float(np.min(ms) * 1e3),
                "bytes": prof[0]["bytes"]}
    finally:
        sess.close()
        eng.destroy()


def config2():
    batch, contexts = 32, 8
    low = builder.resnet_lowered(152, builder.PREC_INT8, image=TV)
    f32 = builder.build_plan(low, builder.PREC_INT8, batch)
    u8 = builder.build_plan(low, builder.PREC_INT8, batch, input_dtype="u8", image=TV)
    eng = capi.Engine(f32)
    eng.tune(streams=contexts)
    tactics = eng.tactics()
    eng.destroy()
    xs = weights.synthetic_image_u8(256, (224, 224), seed=4242)
    out = {}
    for name, blob, x in (("f32", f32, builder.preprocess_u8(xs, CHW, TV)), ("u8", u8, xs),
                          ("f32_again", f32, builder.preprocess_u8(xs, CHW, TV)), ("u8_again", u8, xs)):
        mgr = capi.InferenceManager(contexts, 2 * contexts, pre_threads=1, cuda_threads=1, post_threads=3)
        try:
            mgr.register_model("rn152i8", builder.attach_tactics(blob, tactics))
            mgr.update_resources()
            mgr.infer_batched("rn152i8", x, window_us=2000)
            n_img, warm, cool = 6144, 1024, 1024
            _, win, dt, nb = mgr.bench_batched("rn152i8", x, n_img, warm, cool, window_us=2000)
        finally:
            mgr.close()
        out[name] = {"value": (n_img - warm - cool) / win, "bracketed": n_img / dt, "merged_batches": nb,
                     "h2d_bytes_per_request": int(x[0].nbytes)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "input_formats.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--zero-copy-leg", help=argparse.SUPPRESS)  # child: write the zero-copy u8 leg to this file
    a = ap.parse_args()
    if capi.device_count() < 1:
        raise SystemExit("gpu_input_formats.py: no CUDA device (there is no CPU fallback to measure)")
    if a.zero_copy_leg:
        r = rings()
        with open(a.zero_copy_leg, "w") as f:
            json.dump(e2e_leg(rn50_blobs()["u8"], r["u8"], a.steps), f)
        return
    t0 = time.time()
    result = {"card": card(), "steps": a.steps, "batch": BATCH, "contexts": CONTEXTS, "buffers": BUFFERS}
    blobs, r = rn50_blobs(), rings()
    legs = []
    for dt in ("f32", "f16", "u8") * 2:
        leg = e2e_leg(blobs[dt], r[dt], a.steps)
        leg["binding"] = dt
        legs.append(leg)
        print(dt, round(leg["value"]), "inf/s", flush=True)
    result["e2e_legs"] = legs
    result["e2e_median"] = {dt: float(np.median([l["value"] for l in legs if l["binding"] == dt])) for dt in ("f32", "f16", "u8")}
    zc_path = a.out + ".zc.tmp"
    env = dict(os.environ, TRTLAB_ZERO_COPY_INPUT="1")
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--steps", str(a.steps), "--zero-copy-leg", zc_path], env=env,
                       capture_output=True, text=True, timeout=1800)
    if p.returncode == 0:
        with open(zc_path) as f:
            result["e2e_u8_zero_copy"] = json.load(f)
        os.remove(zc_path)
    else:
        result["e2e_u8_zero_copy"] = {"error": p.stderr[-2000:]}
    x8 = r["u8"][0]
    result["cast_kernel"] = {"f32": cast_time(blobs["f32"], r["f32"][0]), "u8": cast_time(blobs["u8"], x8)}
    result["config2_rn152_int8_b32_batched"] = config2()
    result["card_after"] = card()
    result["seconds"] = time.time() - t0
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("card", "e2e_median")}))


if __name__ == "__main__":
    main()
