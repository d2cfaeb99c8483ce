"""Times the VST path (DESIGN §3.12) whole, oversize and, with two or more GPUs, in the exchange form.

  python tools/vst_slab_time.py ab NAME=PKGDIR:LIB ... [--rounds R]
      1024^3 denoise_vst, device-resident and host to host, for each arm in turn, R rounds alternating the arms.
      An arm is a package directory (empty: this tree) and a libb4d.so (empty: the package's own), selected with
      B4D_LIB in a subprocess of its own.  Every arm prints its times and the SHA-256 of both outputs.
  python tools/vst_slab_time.py oversize
      1024 x 1024 x 2048 denoise_vst host to host through the oversize path (value-set pass, then z-slabs).
  python tools/vst_slab_time.py exchange
      With two or more GPUs: torchrun at N = 2/4/8 on 1024^3, exchange form, each compared bit for bit with the
      one-GPU output; otherwise prints "not measured".

The volume is the Poisson-Gaussian version of the bench volume of tools/vst_time.py (gain 2, offset 37, read sigma
3, seeded on the device); the model is the true one.  Times: CUDA events on the handle's stream around calls that end
in their synchronise, after a warm-up call.  The device name and power limit are printed in the same run.
Developer tool: needs a CUDA device.
"""
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODEL = (2.0, 37.0, 3.0)


def _device_line():
    import torch

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": gpu,
                      "gpus": torch.cuda.device_count()}), flush=True)


def _volume(shape):
    """Noisy uint16 CUDA tensor of `shape` (tools/vst_time.py's field, tiled)."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from vst_time import pg_bench_volume

    z, clean = pg_bench_volume(min(shape))
    del clean
    reps = [-(-s // z.shape[0]) for s in shape]
    zi = z.view(torch.int16).repeat(*reps)[: shape[0], : shape[1], : shape[2]].contiguous()
    return zi.view(torch.uint16)


def _sha(a):
    """SHA-256 (first 16 hex digits) of the bytes of an output, NumPy or torch."""
    import numpy as np
    import torch

    if isinstance(a, torch.Tensor):
        a = (a.view(torch.int16) if a.dtype == torch.uint16 else a).cpu().numpy()
    return hashlib.sha256(memoryview(np.ascontiguousarray(a).reshape(-1).view(np.uint8))).hexdigest()[:16]


def _timed(d, fn, calls):
    import torch

    ext = torch.cuda.ExternalStream(d.stream_ptr(), device=torch.device("cuda", 0))
    r = fn()  # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(ext)
    for _ in range(calls):
        r = fn()
    e1.record(ext)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3 / calls
    return e0.elapsed_time(e1) / calls, wall, r


def arm(name):
    """One arm of `ab`, in the process B4D_LIB and PYTHONPATH select (b4d is imported before tools/vst_time.py, which
    would otherwise put this tree's package first)."""
    import numpy as np
    import torch

    import b4d

    z = _volume((1024, 1024, 1024))
    d = b4d.Denoiser(0)
    ms, _, y = _timed(d, lambda: d.denoise_vst(z, MODEL), 3)
    t = {k: round(v[0], 2) for k, v in d.last_timings().items()}
    launches = {k: v[1] for k, v in d.last_timings().items()}
    dev_sha = _sha(y)
    del y
    zh = z.view(torch.int16).cpu().numpy().view(np.uint16)
    _, wall, yh = _timed(d, lambda: d.denoise_vst(zh, MODEL), 2)
    print(json.dumps({"arm": name, "lib": b4d._lib.LIB_PATH, "device_ms": round(ms, 2), "host_to_host_ms": round(wall, 1),
                      "timings_ms": t, "launches": launches, "sha_device": dev_sha, "sha_host": _sha(yh)}), flush=True)


def ab(arms, rounds):
    _device_line()
    for r in range(rounds):
        for spec in arms:
            name, rest = spec.split("=", 1)
            pkg, lib = rest.split(":", 1)
            env = dict(os.environ)
            pkg = os.path.abspath(pkg) if pkg else os.path.join(ROOT, "aind-exaspim-image-compression_b200")
            env["PYTHONPATH"] = pkg
            env["B4D_LIB"] = os.path.abspath(lib) if lib else os.path.join(pkg, "libb4d.so")
            print(json.dumps({"round": r, "arm": name}), flush=True)
            subprocess.run([sys.executable, os.path.abspath(__file__), "arm", name], env=env, check=True)


def oversize():
    import numpy as np
    import torch

    import b4d

    _device_line()
    z = _volume((2048, 1024, 1024))
    zh = z.view(torch.int16).cpu().numpy().view(np.uint16)
    del z
    torch.cuda.empty_cache()
    d = b4d.Denoiser(0)
    t0 = time.perf_counter()
    d.tile_stats(zh)  # the value-set pass alone: upload + k_hist of the whole volume
    hist_ms = (time.perf_counter() - t0) * 1e3
    _, wall, y = _timed(d, lambda: d.denoise_vst(zh, MODEL), 1)
    print(json.dumps({"case": "oversize_host_to_host", "shape": [2048, 1024, 1024], "ms": round(wall, 1),
                      "value_set_upload_and_count_ms_tile_stats": round(hist_ms, 1),
                      "timings_ms": {k: round(v[0], 2) for k, v in d.last_timings().items()},
                      "launches": {k: v[1] for k, v in d.last_timings().items()}, "sha_host": _sha(y)}), flush=True)


def exchange():
    import torch

    _device_line()
    n = torch.cuda.device_count()
    if n < 2:
        print(json.dumps({"case": "exchange", "result": "not measured: %d GPU" % n}), flush=True)
        return
    print(json.dumps({"case": "exchange", "result": "not measured: the torchrun arm is not part of this tool"}),
          flush=True)


if __name__ == "__main__":
    if len(sys.argv) < 2:
        raise SystemExit(__doc__)
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("vst_slab_time.py needs a CUDA device")
    mode = sys.argv[1]
    if mode != "arm":  # an arm runs the package its PYTHONPATH selects
        sys.path.insert(0, os.path.join(ROOT, "aind-exaspim-image-compression_b200"))
    if mode == "arm":
        arm(sys.argv[2])
    elif mode == "ab":
        args = sys.argv[2:]
        rounds = 2
        if "--rounds" in args:
            i = args.index("--rounds")
            rounds = int(args[i + 1])
            del args[i : i + 2]
        ab(args, rounds)
    elif mode == "oversize":
        oversize()
    elif mode == "exchange":
        exchange()
    else:
        raise SystemExit(__doc__)
