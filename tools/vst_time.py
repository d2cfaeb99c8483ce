"""Times the Poisson-Gaussian path (DESIGN §3.12) on a Poisson-Gaussian version of the 1024^3 bench volume, resident
on the device, against the uint16 path on the same volume.

The volume: the bench's clean field (synth.clean_tile(4), period 128) as the expected count, z = gain Poisson((c -
offset)/gain) + N(offset, read_sigma^2) with gain 2, offset 37, read sigma 3, drawn on the device with a seeded
generator, rounded and clipped to uint16.  Timed, with CUDA events on the handle's stream after warm-up calls:
noise_level_function (default bins), gat_forward and gat_inverse (device in and out), denoise_vst with the model
from the estimate, and denoise(u16) at sigma = noise_sigma.  Each call includes its stream synchronise.  Also the
byte-tile share of the matcher (byte tiles over the tiles of both stages) of the two denoise paths, their RMSE
against the clean field, and the device name and power limit from the same run.  Developer tool: needs a CUDA
device.
"""
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "aind-exaspim-image-compression_b200"))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import b4d  # noqa: E402
from b4d import _lib, synth  # noqa: E402

GAIN, OFFSET, READ_SIGMA = 2.0, 37.0, 3.0


def pg_bench_volume(n, seed=4):
    """(noisy uint16 CUDA tensor, clean float32 CUDA tensor) of side n."""
    tile = torch.from_numpy(synth.clean_tile(seed)).cuda()
    reps = -(-n // tile.shape[0])
    clean = tile.repeat(reps, reps, reps)[:n, :n, :n].contiguous()
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    lam = torch.clamp(clean.double() - OFFSET, min=0.0) / GAIN
    z = GAIN * torch.poisson(lam, generator=g) + OFFSET
    del lam
    z += READ_SIGMA * torch.randn(z.shape, generator=g, device="cuda", dtype=torch.float64)
    z = torch.clamp(torch.round(z), 0, 65535).to(torch.int32).to(torch.int16)  # the uint16 bits
    return z.view(torch.uint16), clean


def timed(d, fn, calls, warmup):
    ext = torch.cuda.ExternalStream(d.stream_ptr(), device=torch.device("cuda", 0))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(warmup):
        r = fn()
    torch.cuda.synchronize()
    e0.record(ext)
    for _ in range(calls):
        r = fn()
    e1.record(ext)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls, r


def rmse(y, clean):
    if y.dtype == torch.uint16:
        y = y.view(torch.int16).to(torch.int32) & 0xFFFF
    return float(torch.sqrt(torch.mean((y.double() - clean.double()) ** 2)))


def main():
    if not torch.cuda.is_available():
        raise SystemExit("vst_time.py needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": gpu}), flush=True)
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    z, clean = pg_bench_volume(n)
    d = b4d.Denoiser(0)
    refs = d.lib.b4d_num_refs(_lib.shape3((n, n, n)))
    tiles = 2 * math.ceil(round(refs ** (1.0 / 3.0)) / 4) ** 3  # matcher tiles of both stages

    ms, nlf = timed(d, lambda: d.noise_level_function(z), 10, 2)
    offset = d.tile_stats(z)["offset"]
    model = b4d.PoissonGaussian.from_nlf(nlf["a"], nlf["b"], offset)
    print(json.dumps({"case": "noise_level_function", "ms": round(ms, 3), "a": nlf["a"], "b": nlf["b"],
                      "usable_bins": nlf["usable"], "offset": offset, "model": model._asdict()}), flush=True)
    ms, f = timed(d, lambda: d.gat_forward(z, model), 10, 2)
    print(json.dumps({"case": "gat_forward", "ms": round(ms, 3), "bytes": 6 * z.numel()}), flush=True)
    ms, _ = timed(d, lambda: d.gat_inverse(f, model), 10, 2)
    print(json.dumps({"case": "gat_inverse", "ms": round(ms, 3), "bytes": 8 * z.numel()}), flush=True)
    del f
    sigma = float(d.noise_sigma(z)["sigma"])
    for name, fn in (("denoise_vst", lambda: d.denoise_vst(z, model)), ("denoise_u16", lambda: d.denoise(z, sigma))):
        ms, y = timed(d, fn, 3, 1)
        st = d.last_match_stats()
        t = {k: round(v[0], 2) for k, v in d.last_timings().items()}
        print(json.dumps({"case": name, "ms": round(ms, 2), "sigma": 1.0 if name == "denoise_vst" else sigma,
                          "byte_tiles": st["byte_tiles"], "tiles": tiles,
                          "byte_tile_share": round(st["byte_tiles"] / tiles, 4), "match_stats": st,
                          "timings_ms": t, "rmse_vs_clean": rmse(y, clean)}), flush=True)
        del y
    print(json.dumps({"case": "noisy", "rmse_vs_clean": rmse(z, clean)}), flush=True)


if __name__ == "__main__":
    main()
