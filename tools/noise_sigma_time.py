"""Times b4d.noise_sigma (DESIGN §3.11) on the 1024^3 bench volume (synth.vol(1024, 1024, 1024, seed=4)) resident
on the device, for tile 64^3, one tile per volume, and one tile per volume with the whole-call histogram.

Per case: ms per call from CUDA events over 20 calls after 3 warm-up calls (the call includes its stream
synchronise and the host arithmetic of the result), the bytes the kernels read, computed from the shape
(2 B per voxel per pass: two select passes, plus one for the histogram), GB/s and the share of the 6553.9 GB/s
copy bandwidth the project uses as its HBM peak (BASELINE.md).  The volume (2 GiB) is 16x the L2, so every pass
reads HBM.  Also prints the device name and power limit from the same run.  Developer tool: needs a CUDA device.
"""
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

HBM_PEAK_GBS = 6553.9
CALLS, WARMUP = 20, 3


def main():
    if not torch.cuda.is_available():
        raise SystemExit("noise_sigma_time.py needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": gpu}))
    shape = (1024, 1024, 1024)
    vol = synth.vol(*shape, seed=4)
    x = torch.from_numpy(vol.view(np.int16)).cuda().view(torch.uint16)
    voxels = int(np.prod(shape))
    d = b4d.Denoiser(0)
    ext = torch.cuda.ExternalStream(d.stream_ptr(), device=x.device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, tile, hist, passes in (("tile64", (64, 64, 64), False, 2), ("whole", None, False, 2),
                                     ("whole+hist", None, True, 3)):
        for _ in range(WARMUP):
            r = d.noise_sigma(x, tile=tile, return_hist=hist)
        torch.cuda.synchronize()
        e0.record(ext)
        for _ in range(CALLS):
            r = d.noise_sigma(x, tile=tile, return_hist=hist)
        e1.record(ext)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / CALLS
        nbytes = passes * 2 * voxels
        gbs = nbytes / (ms * 1e-3) / 1e9
        s = r[0]["sigma"] if hist else r["sigma"]
        print(json.dumps({"case": name, "tile": tile, "hist": hist, "ms": round(ms, 4), "bytes_read": nbytes,
                          "GB/s": round(gbs, 1), "share_of_hbm_peak": round(gbs / HBM_PEAK_GBS, 3),
                          "sigma_median": float(np.median(s)), "calls": CALLS}))


if __name__ == "__main__":
    main()
