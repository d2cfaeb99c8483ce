"""A/B timing of per-tile quantizer steps (DESIGN §3 item 13) against the scalar step on one GPU, in one process,
alternating the two forms: standalone quantize, the fused denoise_quantized (whole call, and its norm2 stage from
last_timings) and dequantize.  Volume: 1024^3 uint16 (default), the periodic synthetic clean field plus Gaussian noise
of sigma 24, generated on the device; the table holds kappa * noise_sigma of the raw volume per 64^3 tile, the scalar
step kappa * the whole volume's noise_sigma.  Times are CUDA events on the handle's stream around each call (medians
over the repetitions).  Prints the card's name and power limit and writes JSON.  Developer tool.

  python tools/step_table_time.py --out profiles/step_table_time_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "aind-exaspim-image-compression_b200"))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import b4d  # noqa: E402
from b4d import synth  # noqa: E402

SIGMA, SEED, KAPPA, TILE = 24.0, 5, 0.5, (64, 64, 64)


def make_volume(n, dev):
    clean = torch.from_numpy(synth.clean_tile(SEED)).to(dev)
    T = clean.shape[0]
    g = torch.Generator(device=dev)
    g.manual_seed(SEED)
    vol = torch.empty((n, n, n), dtype=torch.uint16, device=dev)
    reps = (n + T - 1) // T
    for z in range(0, n, 16):
        z1 = min(n, z + 16)
        base = clean[torch.arange(z, z1, device=dev) % T].repeat(1, reps, reps)[:, :n, :n]
        v = base + torch.randn((z1 - z, n, n), generator=g, device=dev) * SIGMA
        vol[z:z1] = torch.clamp(torch.round(v), 0, 65535).to(torch.int32).to(torch.uint16)
    return vol


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "step_table_time_b200.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    dev = torch.device("cuda", 0)
    dn = b4d.Denoiser(0)
    raw = make_volume(args.size, dev)
    sig = dn.noise_sigma(raw, tile=TILE)["sigma"]
    table = b4d.noise_scaled_steps(sig, KAPPA, TILE)
    step = b4d.noise_scaled_step(dn.noise_sigma(raw)["sigma"], KAPPA)
    y = dn.denoise(raw, SIGMA)
    ext = torch.cuda.ExternalStream(dn.stream_ptr(), device=dev)

    def timed(call):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(ext)
        out = call()
        e1.record(ext)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    pairs = {
        "quantize": (lambda: dn.quantize(y, 37.0, 0.0, step), lambda: dn.quantize(y, 37.0, 0.0, table)),
        "denoise_quantized": (lambda: dn.denoise_quantized(raw, SIGMA, 37.0, 0.0, step),
                              lambda: dn.denoise_quantized(raw, SIGMA, 37.0, 0.0, table)),
    }
    res = {k: {"scalar_ms": [], "table_ms": []} for k in ("quantize", "denoise_quantized", "dequantize")}
    res["denoise_quantized"].update({"scalar_norm2_ms": [], "table_norm2_ms": []})
    q_scalar = q_table = None
    for rep in range(args.reps + 1):  # the first round warms every shape up and is dropped
        for name, (a, b) in pairs.items():
            for form, call in (("scalar", a), ("table", b)):
                ms, out = timed(call)
                norm2 = dn.last_timings()["norm2"][0] if name == "denoise_quantized" else None
                if name == "quantize":
                    if form == "scalar":
                        q_scalar = out
                    else:
                        q_table = out
                del out
                if rep:
                    res[name][form + "_ms"].append(ms)
                    if norm2 is not None:
                        res[name][form + "_norm2_ms"].append(norm2)
        for form, call in (("scalar", lambda: dn.dequantize(q_scalar, step, 37.0)),
                           ("table", lambda: dn.dequantize(q_table, table, 37.0))):
            ms, out = timed(call)
            del out
            if rep:
                res["dequantize"][form + "_ms"].append(ms)
    n = args.size ** 3
    summary = {}
    for name, r in res.items():
        summary[name] = {k: float(np.median(v)) for k, v in r.items()}
    for name in ("quantize", "dequantize"):  # 4 B float32 + 2 B uint16 per voxel
        summary[name]["table_TB_per_s"] = 6.0 * n / (summary[name]["table_ms"] * 1e-3) / 1e12
    d = summary["denoise_quantized"]
    d["norm2_table_over_scalar"] = d["table_norm2_ms"] / d["scalar_norm2_ms"]
    name, limits = card()
    out = {
        "tool": "tools/step_table_time.py", "card": name, "power_limit_and_max_sm_clock": limits,
        "volume": "%d^3 uint16, synthetic, sigma %g" % (args.size, SIGMA), "tile": TILE, "kappa": KAPPA,
        "scalar_step": step, "table_steps_min_max": [float(table.steps.min()), float(table.steps.max())],
        "reps": args.reps, "median": summary, "all": res,
        "timing": "CUDA events on the handle's stream around each call, tensors on the device; the table calls "
                  "include their table upload",
    }
    print(json.dumps(out, indent=1), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    dn.close()


if __name__ == "__main__":
    main()
