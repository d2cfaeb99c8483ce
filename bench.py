#!/usr/bin/env python
"""bench.py — BM4D denoise voxels/s on a synthetic uint16 1024^3 ExaSPIM-like
volume, z-slab sharded over N B200s (BASELINE.json metric, configs[3]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--size S] [--dump-outputs DIR]

One step = one full two-stage BM4D denoise (hard threshold + Wiener) of the
whole volume: every rank denoises its z-slab (+ halos on the global grid, no
volume data crosses GPUs), after the path's only collective — the all-gather of
per-slab uint16 histograms for the global offset / sigma statistics.

  value   voxels/s with the slab already resident in HBM (device in, device out)
  e2e     voxels/s through the public API with HOST buffers (pinned): H2D of the
          slab and D2H of the owned planes inside the timed region
  roofline  the matching kernel (dominant): algorithmic integer ops
          2*Ns^3*L^3*R per launch / its CUDA-event duration, against the
          (sub, mad) issue-rate peak measured live by the shipped microbenchmark
  cpu_baseline  the CPU oracle (float32 path, OpenMP, all host cores) on a
          bounded sub-volume of the same data — "port", not the closed bm4d wheel

--impl reference times the reference arm: the reference's BM4D is the closed
third-party wheel bm4d==4.2.5 (absent from this image and un-installable, no
network), so the arm runs this repo's CPU restatement (oracle/) — labelled as such.

--dump-outputs DIR writes what the last timed step returned, so that two builds
can be compared output for output on the same seeded input:
  denoised.npy    float32, the denoised volume at DUMP_VOXELS seeded flat
                  positions (every voxel when the volume is smaller), ascending
  tile_stats.npy  float64, the step's tile statistics in b4d_stats field order
                  (n, n_nonzero, offset, median, mad, sigma, vmin, vmax)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
# torch.distributed.run exports OMP_NUM_THREADS=1 to every rank.  Rank 0 runs the CPU legs (cpu_baseline,
# --impl reference) on all the host cores it may use, so the OpenMP runtime has to see that count BEFORE any
# library that carries one (NumPy, torch, liboracle.so) is loaded; oracle_threads() reports what was used.
if int(os.environ.get("RANK", "0")) == 0:
    os.environ["OMP_NUM_THREADS"] = str(len(os.sched_getaffinity(0)))
    os.environ.pop("OMP_THREAD_LIMIT", None)
for _p in (os.path.join(ROOT, "aind-exaspim-image-compression_b200"), ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

SIGMA = 24.0  # scripts/precompute.py:284
SEED = 4  # SURVEY §8d config 4
NS, LBLK, K_HT, K_WIE = 11, 4, 16, 32
DUMP_VOXELS = 1 << 22  # --dump-outputs: 16 MiB of float32 at most


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------- data ------
def make_slab_device(size, zb, ze, device):
    """uint16 planes [zb, ze) of the seeded size^3 volume, generated on the GPU:
    the clean 128^3 tile of b4d.synth repeated periodically + white Gaussian
    noise (sigma 24) seeded per 128-plane chunk, so any rank can regenerate any
    plane without materialising the whole volume."""
    import torch

    from b4d import synth

    clean = torch.from_numpy(synth.clean_tile(SEED)).to(device)  # (128,128,128) float32
    T = clean.shape[0]
    reps = (size + T - 1) // T
    plane_tile = clean.repeat(1, reps, reps)[:, :size, :size]  # (128, size, size)
    out = torch.empty((ze - zb, size, size), dtype=torch.uint16, device=device)
    for c in range(zb // T, (ze - 1) // T + 1):
        a, b = max(zb, c * T), min(ze, (c + 1) * T)
        g = torch.Generator(device=device)
        g.manual_seed(SEED * 1000003 + c)
        noise = torch.randn((T, size, size), generator=g, device=device, dtype=torch.float32) * SIGMA
        v = (plane_tile + noise)[a - c * T : b - c * T]
        out[a - zb : b - zb] = torch.clamp(torch.round(v), 0, 65535).to(torch.int32).to(torch.uint16)
        del noise, v
    return out


def make_sample_host(shape):
    from b4d import synth

    return synth.vol(shape[0], shape[1], shape[2], seed=SEED, sigma=SIGMA)


def dump_sample_index(size):
    """Ascending flat indices into the size^3 volume of the voxels --dump-outputs writes: all of them up to
    DUMP_VOXELS, else a draw seeded by SEED, so that it depends on the size alone (not on the run or the world size)."""
    n = size ** 3
    if n <= DUMP_VOXELS:
        return np.arange(n, dtype=np.int64)
    return np.unique(np.random.default_rng(SEED).integers(0, n, DUMP_VOXELS, dtype=np.int64))


def dump_outputs(path, y, stats, size, own_b, own_e, world, rank, device):
    """Write the sampled denoised volume and the tile statistics of one step to path (rank 0).  Each rank fills
    the sampled voxels of its owned planes [own_b, own_e); the others stay 0, so an integer sum over the ranks
    assembles the float32 bit patterns unchanged."""
    import torch
    import torch.distributed as dist

    from b4d import _lib

    idx = dump_sample_index(size)
    plane = size * size
    lo, hi = (int(i) for i in np.searchsorted(idx, (own_b * plane, own_e * plane)))
    bits = torch.zeros(idx.size, dtype=torch.int32, device=device)
    mine = torch.from_numpy(idx[lo:hi] - own_b * plane).to(device)
    bits[lo:hi] = y.reshape(-1)[mine].view(torch.int32)
    if world > 1:
        dist.all_reduce(bits)
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        np.save(os.path.join(path, "denoised.npy"), bits.cpu().numpy().view(np.float32))
        np.save(os.path.join(path, "tile_stats.npy"), np.array([stats[k] for k, _ in _lib.Stats._fields_], np.float64))
        log("outputs of the last timed step written to %s (%d sampled voxels)" % (path, idx.size))


# --------------------------------------------------------------- clocks ------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL,
                text=True,
            )
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------- reference -----
def probe_real_bm4d():
    """Version of an importable closed `bm4d` wheel (plain, then baseline/_ref), or
    None.  This repo's own import-name shim does not count."""
    saved = list(sys.path)
    try:
        sys.path[:] = [p for p in saved if "aind-exaspim-image-compression_b200" not in p]
        sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
        sys.modules.pop("bm4d", None)
        import bm4d as real

        v = getattr(real, "__version__", "?")
        return None if "b4d" in str(v) else str(v)
    except Exception:
        return None
    finally:
        sys.modules.pop("bm4d", None)
        sys.path[:] = saved


def workload_config(S, halo, exchange=False):
    return {
        "workload": "BM4D HT+Wiener denoise of one uint16 %d^3 volume (BASELINE configs[3]), z-slabs + halo %d%s"
        % (S, halo, " + one neighbour exchange of basic-estimate planes between the stages" if exchange else ""),
        "sigma": SIGMA, "Ns": NS, "K_ht": K_HT, "K_wiener": K_WIE,
    }


def xform_roofline(mac_per_voxel, voxels, ms, peaks):
    if not ms or not peaks.get("ffma"):
        return None
    ach = mac_per_voxel * voxels / (ms * 1e-3)
    return {"bound": "fp32", "achieved": ach / 1e12, "peak": peaks["ffma"] / 1e12, "unit": "TMAC/s",
            "frac": ach / peaks["ffma"], "ms_per_launch": ms}


def traffic_per_launch(size, world):
    """dram__bytes_read.sum + dram__bytes_write.sum of one k_match launch, from the committed
    `ncu --set full` capture of this workload (profiles/traffic.json), or None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        return t.get("k_match", {}).get("%d^3/%d" % (size, world))
    except Exception:
        return None


def oracle_threads():
    """Pin the oracle's OpenMP team to the cores this process may run on and return the team size
    actually used (omp_get_max_threads after the call) — never os.cpu_count()."""
    from oracle import np_oracle

    return np_oracle.set_threads(len(os.sched_getaffinity(0)))


def cpu_port_throughput(sample_shape, repeats=1, dn=None):
    """voxels/s of the CPU oracle (float32 path, OpenMP over all host cores).  With a Denoiser the oracle also acts
    as the checker: the GPU result on the same sample is compared with the oracle's, and a 64^3 crop with the
    float64 oracle (max-abs, and how many stage-2 groups differ between the float32 and the float64 pipeline)."""
    from oracle import np_oracle

    vol = make_sample_host(sample_shape)
    o = np_oracle.Oracle("mirror")
    best = None
    for _ in range(repeats):
        t = time.perf_counter()
        ref = o.denoise(vol, SIGMA)
        dt = time.perf_counter() - t
        best = dt if best is None else min(best, dt)
    parity = None
    if dn is not None:
        from oracle import parity_util

        y = np.asarray(dn.denoise(vol, SIGMA))
        diff = np.abs(y.astype(np.float64) - ref.astype(np.float64))
        parity = {"vs_float32_mirror": {"voxels": int(vol.size), "bit_equal": bool((y.view(np.uint32) == ref.view(np.uint32)).all()),
                                        "voxels_differing": int((y.view(np.uint32) != ref.view(np.uint32)).sum()),
                                        "max_abs": float(diff.max())}}
        crop = np.ascontiguousarray(vol[:64, :64, :64])
        of = np_oracle.Oracle("f64")
        f = of.denoise(crop, SIGMA)
        o.denoise(crop, SIGMA)
        yc = np.asarray(dn.denoise(crop, SIGMA))
        try:
            rep = parity_util.check_against_f64(yc, f, o.stage2_matches(crop.shape), of.stage2_matches(crop.shape), 0.5, 0.05, NS)
            rep["within_bar"] = True
        except AssertionError as e:  # report, never hide
            rep = dict(e.args[0]) if e.args and isinstance(e.args[0], dict) else {"error": str(e)}
            rep["within_bar"] = False
        rl2 = float(np.linalg.norm(yc.astype(np.float64) - f) / np.linalg.norm(f))
        parity["vs_float64_oracle"] = dict(rep, voxels=int(crop.size), rel_l2=rl2,
                                           bar="max-abs <= 0.5 except under flipped stage-2 matches; rel-L2 <= 1e-3")
    return vol.size / best, best, parity


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    shape = (128, 192, 192)
    cores = oracle_threads()
    real = probe_real_bm4d()
    from oracle import np_oracle

    vol = make_sample_host(shape)
    o = np_oracle.Oracle("mirror")
    for _ in range(args.warmup):
        o.denoise(vol, SIGMA)
    t = time.perf_counter()
    for _ in range(args.steps):
        o.denoise(vol, SIGMA)
    dt = (time.perf_counter() - t) / args.steps
    val = vol.size / dt
    sample = "%dx%dx%d sub-volume of the seeded 1024^3 volume per step (CPU restatement oracle/, float32 path, OpenMP)" % shape
    line = {
        "impl": "reference",
        "metric": "bm4d_denoise_voxels_per_s",
        "value": val,
        "unit": "voxels/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": dt * 1e3,
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": dict(workload_config(args.size, 2 * (NS - 1 + LBLK - 1)), sample=sample),
        "cpu_baseline": {"value": val, "unit": "voxels/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference bm4d==4.2.5 (closed wheel) absent -> parity vs closed binary NOT measured; "
        "this arm times the repo's CPU restatement" + ("" if real is None else " (an importable bm4d %s was found but is not used here)" % real),
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------ main -----
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b4d", choices=["b4d", "reference"])
    ap.add_argument("--size", type=int, default=1024, help="volume side (default 1024: the metric's config)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stats", action="store_true", help="diagnostic: leave the statistics pass out of the step")
    ap.add_argument("--no-exchange", action="store_true",
                    help="N > 1: 26-plane halos and no data-path exchange instead of 13-plane halos + one "
                         "neighbour exchange of basic-estimate planes between the stages")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned to DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs dumps the GPU path; --impl reference has no such output")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import b4d
    from b4d.sharding import denoise_slab_exchange, exchange_halo, halo_planes, slab_plan, stats_from_hist_lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world != args.gpus:
        log("bench.py: --gpus %d needs torchrun with WORLD_SIZE=%d (got %d)" % (args.gpus, args.gpus, world))
        return 2
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = b4d.bind_to_gpu_numa(local) if world > 1 else None  # before any host buffer exists
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    S = args.size
    exchange = world > 1 and not args.no_exchange
    halo = exchange_halo(NS, NS) if exchange else halo_planes(NS, NS, 2)
    own_b, own_e, zb, ze = slab_plan(S, world, rank, halo)
    dn = b4d.Denoiser(local)
    t0 = time.perf_counter()
    slab_dev = make_slab_device(S, zb, ze, dev)
    torch.cuda.synchronize()
    slab_pin = torch.empty(slab_dev.shape, dtype=torch.uint16, pin_memory=True)
    slab_pin.copy_(slab_dev)
    out_pin = torch.empty((own_e - own_b, S, S), dtype=torch.float32, pin_memory=True)
    outq_pin = torch.empty((own_e - own_b, S, S), dtype=torch.uint16, pin_memory=True)
    torch.cuda.synchronize()
    if rank == 0:
        log("data: slab %s generated in %.1fs" % (tuple(slab_dev.shape), time.perf_counter() - t0))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def stats_begin():
        # the path's only collective: all-gather of per-slab histograms.  N > 1: started asynchronously, it
        # travels while the slab is denoised; stats_end() sums the parts and evaluates the statistics.
        st, hist = dn.tile_stats(slab_dev[own_b - zb : own_e - zb], 0.1, return_hist=True)
        if world == 1:
            return st
        mine = torch.from_numpy(hist).to(dev)
        parts = torch.empty((world,) + tuple(mine.shape), dtype=mine.dtype, device=dev)
        return (dist.all_gather_into_tensor(parts, mine, async_op=True), parts, mine)

    def stats_end(tok):
        if world == 1:
            return tok
        tok[0].wait()
        return stats_from_hist_lib(tok[1].sum(0).cpu().numpy(), 0.1)

    host_ms = {"stats_begin": 0.0, "denoise": 0.0, "stats_end": 0.0}

    def step_resident():
        t0 = time.perf_counter()
        if args.no_stats and stats is not None:
            tok = None
        else:
            tok = stats_begin()
        t1 = time.perf_counter()
        if exchange:  # stage 1, neighbour exchange of basic-estimate planes (NCCL p2p), stage 2
            y = denoise_slab_exchange(dn, slab_dev, zb, S, own_b, own_e, SIGMA, rank, world, device=dev)
        else:
            y = dn.denoise_slab(slab_dev, zb, S, own_b, own_e, SIGMA)
        t2 = time.perf_counter()
        st = stats if tok is None else stats_end(tok)
        t3 = time.perf_counter()
        host_ms["stats_begin"] += (t1 - t0) * 1e3
        host_ms["denoise"] += (t2 - t1) * 1e3
        host_ms["stats_end"] += (t3 - t2) * 1e3
        return st, y

    # end to end, host in -> host out through the public API; H2D and D2H happen inside the call.  The path named
    # by BASELINE.json ends in the quantizer: the fused form returns the uint16 volume (denoise -> background-offset
    # subtract -> quantize, 2 bytes per voxel back to the host); the float32 form (the bm4d() return value, 4 bytes
    # per voxel) is timed as well and reported as e2e_float32.
    def step_e2e(quant=None, host_in=None, host_out=None):
        src = slab_pin.numpy() if host_in is None else host_in
        dst = (outq_pin.numpy() if quant is not None else out_pin.numpy()) if host_out is None else host_out
        if exchange:
            denoise_slab_exchange(dn, src, zb, S, own_b, own_e, SIGMA, rank, world, device=dev, out=dst, quantize=quant)
        else:
            dn.denoise_slab(src, zb, S, own_b, own_e, SIGMA, out=dst, quantize=quant)

    # ---- warm-up (also sizes the scratch buffers)
    stats = None
    for _ in range(max(args.warmup, 3)):
        stats, y = step_resident()
        del y
    barrier()

    # ---- timed: resident inputs.  CUDA events on the library's own stream (every kernel and
    # copy of the handle is enqueued there; torch.cuda.Event only sees the stream it is
    # recorded on), bracketed by barrier + synchronize.
    ext = torch.cuda.ExternalStream(dn.stream_ptr(), device=dev)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    fam = {}
    launches = 0
    barrier()
    ev0.record(ext)
    for i in range(args.steps):
        stats, y = step_resident()
        if i + 1 < args.steps:  # the last step's output stays for --dump-outputs
            del y
        tm = dn.last_timings()
        for k, (ms, nl) in tm.items():
            fam[k] = fam.get(k, 0.0) + ms
            launches += nl
        launches += 1  # histogram kernel
    ev1.record(ext)
    barrier()
    dt = ev0.elapsed_time(ev1) * 1e-3
    log("rank %d host ms per step (warm-up included): %s" % (rank, {k: round(v / (args.steps + max(args.warmup, 3)), 2) for k, v in host_ms.items()}))
    clocks = sampler.stop() if rank == 0 else None
    mstats = dn.last_match_stats()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, y, stats, S, own_b, own_e, world, rank, dev)
    del y

    # ---- the HBM-bound tail of the path: fused offset-subtract + noise-scaled quantize (K7) on the
    # denoised slab, device in / device out, timed alone (burst) with CUDA events
    _, y_last = step_resident()
    step_q = b4d.noise_scaled_step(stats["sigma"], 0.5)
    q_ms = None
    for _ in range(4):
        ev0.record(ext)
        qv = dn.quantize(y_last, offset_sub=float(stats["offset"]), offset_add=0.0, step=step_q)
        ev1.record(ext)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        q_ms = ms if q_ms is None else min(q_ms, ms)
    q_vox = float(y_last.numel())
    # ---- K9: chunk gather + byte shuffle + byte counts of the quantized slab (64^3 pieces), same way
    c_ms = cb_ms = None
    for _ in range(4):
        ev0.record(ext)
        cby, chist = dn.chunk_shuffle(qv, (64, 64, 64))
        ev1.record(ext)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        c_ms = ms if c_ms is None else min(c_ms, ms)
        ev0.record(ext)
        cby, _ = dn.chunk_shuffle(qv, (64, 64, 64), want_hist=False)
        ev1.record(ext)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        cb_ms = ms if cb_ms is None else min(cb_ms, ms)
    cratio_est = b4d.estimate_cratio(chist.cpu().numpy()) if rank == 0 else None
    del y_last, qv, cby, chist

    # ---- timed: end to end with host buffers (pinned): quantized uint16 result, then the float32 result
    quant = (float(stats["offset"]), 0.0, 1.0)
    step_e2e(quant)
    barrier()
    ev0.record(ext)
    for _ in range(args.steps):
        step_e2e(quant)
    ev1.record(ext)
    barrier()
    dt_e2e = ev0.elapsed_time(ev1) * 1e-3
    step_e2e()
    barrier()
    ev0.record(ext)
    for _ in range(args.steps):
        step_e2e()
    ev1.record(ext)
    barrier()
    dt_e2e_f32 = ev0.elapsed_time(ev1) * 1e-3

    # ---- the same with ordinary (pageable) NumPy arrays, what the reference's callers hand over: the
    # library stages them through its pinned ring (HostMover).  Wall clock between barriers (the call
    # returns when the output array is complete).
    slab_np = np.array(slab_pin.numpy(), copy=True)
    out_np = np.empty(tuple(out_pin.shape), dtype=np.float32)

    step_e2e(None, slab_np, out_np)
    barrier()
    t_pg = time.perf_counter()
    for _ in range(args.steps):
        step_e2e(None, slab_np, out_np)
    barrier()
    dt_pg = time.perf_counter() - t_pg
    del slab_np, out_np

    times = torch.tensor([dt, dt_e2e, dt_pg, dt_e2e_f32], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dt, dt_e2e, dt_pg, dt_e2e_f32 = (float(t) for t in times)
    h2d = torch.tensor([slab_pin.numel() * 2, out_pin.numel() * 4, launches], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(h2d, op=dist.ReduceOp.SUM)

    if rank == 0:
        V = float(S) ** 3
        # reference blocks this rank processed per stage (slab grid), for the roofline
        from b4d.api import _lib as L

        peaks = dn.measure_pipe_peaks()
        r_slab = dn.lib.b4d_num_refs(L.shape3((ze - zb, S, S)))
        ops_per_launch = 2.0 * NS ** 3 * LBLK ** 3 * r_slab  # upper bound: slab-edge refs are skipped
        t_match = (fam.get("match1", 0.0) + fam.get("match2", 0.0)) / (2.0 * args.steps) * 1e-3
        achieved = ops_per_launch / t_match if t_match > 0 else 0.0
        hbm_peak = 6553.9
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        except Exception:
            pass
        t_norm = (fam.get("norm1", 0.0) + fam.get("norm2", 0.0)) / (2.0 * args.steps) * 1e-3
        slab_vox = float(ze - zb) * S * S
        t_k0 = fam.get("k0", 0.0) / (2.0 * args.steps) * 1e-3
        kernels = {
            "match": {"bound": "int32", "achieved": achieved / 1e12, "peak": peaks["sub_mad"] / 1e12, "unit": "TOP/s",
                      "frac": achieved / peaks["sub_mad"] if peaks["sub_mad"] else None,
                      "ms_per_launch": t_match * 1e3},
            # SURVEY 8d: K3 / K6 count 8 B read + 4 B write per voxel (the kernel itself moves more: int64
            # numerator, uint32 weight map, float32 out = 16 B/voxel; the fallback is read only where den = 0)
            "normalise": {"bound": "hbm", "achieved": 12.0 * slab_vox / t_norm / 1e9 if t_norm > 0 else None,
                          "peak": hbm_peak, "unit": "GB/s",
                          "frac": 12.0 * slab_vox / t_norm / 1e9 / hbm_peak if t_norm > 0 else None,
                          "moved_bytes_per_voxel": 16.0,
                          "ms_per_launch": t_norm * 1e3},
            # K0: uint16 read + {S2, S1} table write = 10 B/voxel, two launches per step (TMA-fed)
            "block_energy": {"bound": "hbm", "achieved": 10.0 * slab_vox / t_k0 / 1e9 if t_k0 > 0 else None,
                             "peak": hbm_peak, "unit": "GB/s",
                             "frac": 10.0 * slab_vox / t_k0 / 1e9 / hbm_peak if t_k0 > 0 else None,
                             "ms_per_launch": t_k0 * 1e3},
            # K7: float32 read + uint16 write = 6 B/voxel (SURVEY §8d)
            "quantize": {"bound": "hbm", "achieved": 6.0 * q_vox / (q_ms * 1e-3) / 1e9, "peak": hbm_peak,
                         "unit": "GB/s", "frac": 6.0 * q_vox / (q_ms * 1e-3) / 1e9 / hbm_peak, "ms_per_launch": q_ms},
            # K9: uint16 read + 2 bytes written = 4 B/voxel
            "chunk_shuffle": {"bound": "hbm", "achieved": 4.0 * q_vox / (c_ms * 1e-3) / 1e9, "peak": hbm_peak,
                              "unit": "GB/s", "frac": 4.0 * q_vox / (c_ms * 1e-3) / 1e9 / hbm_peak,
                              "ms_per_launch": c_ms, "entropy_cratio_of_quantized_slab": cratio_est,
                              "bytes_only_ms": cb_ms, "bytes_only_frac": 4.0 * q_vox / (cb_ms * 1e-3) / 1e9 / hbm_peak},
            "filter_ht_ms": fam.get("filter1", 0.0) / args.steps,
            "filter_wiener_ms": fam.get("filter2", 0.0) / args.steps,
            # SURVEY 8d: dense-matrix MAC count of the transforms, K (2*768 + 4*64) / 27 per voxel (hard threshold)
            # and K (3*768 + 6*64) / 27 (Wiener), against the measured FFMA issue rate.  The Haar stage needs no
            # multiplies and the kernels are bound by shuffles / shared-memory reductions, so this is a low bar.
            "filter_ht": xform_roofline(K_HT * (2 * 768 + 4 * 64) / 27.0, slab_vox, fam.get("filter1", 0.0) / args.steps, peaks),
            "filter_wiener": xform_roofline(K_WIE * (3 * 768 + 6 * 64) / 27.0, slab_vox, fam.get("filter2", 0.0) / args.steps, peaks),
        }
        line = {
            "metric": "bm4d_denoise_voxels_per_s",
            "value": V * args.steps / dt,
            "unit": "voxels/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": max(args.warmup, 3),
            "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": None,
            "dtype": "int32+f32",
            "data": "synthetic",
            "config": dict(
                workload_config(S, halo, exchange),
                l2="inputs larger than L2 (%.2f GiB slab per rank)" % (slab_pin.numel() * 2 / 2 ** 30),
                timing="CUDA events on the library stream around the K steps, between barrier + synchronize, max over ranks",
            ),
            "e2e": {"value": V * args.steps / dt_e2e, "unit": "voxels/s",
                    "h2d_bytes_per_step": int(h2d[0]), "d2h_bytes_per_step": int(h2d[1]) // 2,
                    "host_buffers": "pinned",
                    "result": "uint16 volume of the fused denoise -> offset subtract -> quantize call (the path's output)"},
            "e2e_float32": {"value": V * args.steps / dt_e2e_f32, "unit": "voxels/s",
                            "h2d_bytes_per_step": int(h2d[0]), "d2h_bytes_per_step": int(h2d[1]),
                            "host_buffers": "pinned", "result": "float32 volume (the bm4d() return value)"},
            "e2e_pageable": {"value": V * args.steps / dt_pg, "unit": "voxels/s",
                             "h2d_bytes_per_step": int(h2d[0]), "d2h_bytes_per_step": int(h2d[1]),
                             "host_buffers": "pageable NumPy arrays (the reference's call surface), float32 result, wall clock"},
            "cpus_bound_to_gpu_numa_node": numa_cpus,
            "gpu_launches": int(h2d[2]),
            "clocks": clocks,
            "roofline": {"bound": "int32", "achieved": achieved / 1e12, "peak": peaks["sub_mad"] / 1e12,
                         "unit": "TOP/s", "frac": achieved / peaks["sub_mad"] if peaks["sub_mad"] else None,
                         "traffic": traffic_per_launch(S, world),
                         "kernel": "k_match<11> (byte-tile + general launch of one stage; stage 1 and 2 averaged)",
                         "peak_source": "shipped microbenchmark, dependent (sub, mad) pairs at the IMAD issue rate, "
                                        "measured in this run; IDP.4A/IDP.2A retire 4/2 pairs per issue slot, so "
                                        "byte tiles can exceed it"},
            "roofline_kernels": kernels,
            "device_ms_per_step": {k: v / args.steps for k, v in fam.items()},
            "pipe_peaks_ops_per_s": peaks,
            "match_stats": mstats,
            "tile_stats": stats,
        }
        if not args.no_cpu_baseline and world == 1:  # rank 0 at N = 1 only (the other ranks would idle in a barrier)
            shape = (192, 256, 256)
            threads = oracle_threads()
            v, secs, parity = cpu_port_throughput(shape, dn=dn)
            line["cpu_baseline"] = {
                "value": v, "unit": "voxels/s", "cores": threads, "kind": "port",
                "sample": "%dx%dx%d sub-volume of the same seeded volume, one pass (%.1f s); CPU restatement, not the closed bm4d binary" % (shape + (secs,)),
                "parity_of_the_gpu_path_on_the_sample": parity,
            }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
