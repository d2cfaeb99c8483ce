"""z-slab sharding of one large volume across the GPUs of one box (SURVEY §8e).

One process per GPU.  Every rank denoises its slab plus halos; reference blocks
sit on the GLOBAL grid, so the union of the owned planes equals the
whole-volume result and no volume data crosses GPUs.  The only exchange is the
all-gather of per-slab uint16 histograms (256 KiB per rank) from which every
rank derives the same global offset percentile / median / MAD sigma — a
percentile is not decomposable from per-rank percentiles, a histogram is
(transforms.py:433-438, metrics.py:54-58).  The VST path (DESIGN §3.12) uses the
same merged histogram as the value set of the whole volume, from which every rank
derives the same matching map.
"""
import os

import numpy as np

L = 4


def halo_planes(search_ht=11, search_wie=11, stages=2):
    """Planes needed beyond the owned range on each interior face for exact
    slab == whole equality: (Ns - 1 + L - 1) per stage (SURVEY Appendix C)."""
    h = search_ht - 1 + L - 1
    if stages == 2:
        h += search_wie - 1 + L - 1
    return h


def slab_plan(z_total, world, rank, halo):
    """Owned planes [own_begin, own_end) and slab planes [z_begin, z_end) of `rank`."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad world/rank")
    base, rem = divmod(int(z_total), int(world))
    own_begin = rank * base + min(rank, rem)
    own_end = own_begin + base + (1 if rank < rem else 0)
    if own_end <= own_begin:
        raise ValueError("more ranks than planes")
    z_begin = max(0, own_begin - halo)
    z_end = min(z_total, own_end + halo)
    if z_end - z_begin < L:
        raise ValueError("slab thinner than one block")
    return own_begin, own_end, z_begin, z_end


def exchange_halo(search_ht=11, search_wie=11):
    """Halo per interior face when neighbours swap basic-estimate planes between the stages
    (SURVEY §8e, "one exchange step"): the larger of the two per-stage halos."""
    return max(search_ht, search_wie) - 1 + L - 1


def exchange_planes(send_down, send_up, recv_below, recv_above, rank, world, group=None):
    """Neighbour exchange of z-planes between consecutive ranks: `send_down` goes to rank - 1
    (which receives it as its `recv_above`), `send_up` to rank + 1.  Tensors on the rank's CUDA
    device (NCCL point-to-point over NVLink) or on the CPU (gloo); None where there is no
    neighbour.  Returns when the received planes are complete."""
    import torch.distributed as dist

    ops = []
    if rank > 0:
        ops.append(dist.P2POp(dist.isend, send_down, rank - 1, group))
        ops.append(dist.P2POp(dist.irecv, recv_below, rank - 1, group))
    if rank < world - 1:
        ops.append(dist.P2POp(dist.isend, send_up, rank + 1, group))
        ops.append(dist.P2POp(dist.irecv, recv_above, rank + 1, group))
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()


def _process_group_ready():
    import torch.distributed as dist

    return dist.is_available() and dist.is_initialized()


def vst_value_hist(denoiser, owned, world, value_hist=None, device=None, group=None):
    """The value set of the whole volume for the VST slab forms (int64 NumPy, 65536 counts): `value_hist` as given,
    else the histogram of this rank's `owned` planes summed over the ranks with merge_histograms.  ValueError when
    world > 1 and no process group is initialised: the local histogram alone would silently give another map."""
    if value_hist is not None:
        return value_hist
    if world > 1 and not _process_group_ready():
        raise ValueError("world > 1 needs an initialised process group, or the whole volume's value_hist")
    import torch

    _, hist = denoiser.tile_stats(owned, return_hist=True)
    merged = merge_histograms(torch.from_numpy(hist).to(device) if device is not None else torch.from_numpy(hist),
                              group)
    return merged.cpu().numpy()


def denoise_slab_exchange(denoiser, slab, z_begin, z_total, own_begin, own_end, sigma, rank, world, device=None,
                          out=None, group=None, quantize=None, model=None, value_hist=None, first=None):
    """One rank's part of the exchange variant: stage 1 on the slab (halo `exchange_halo`), swap
    the exact basic-estimate planes next to each interior face with the neighbours, stage 2.
    `device` = the rank's torch CUDA device (planes then travel device to device).
    quantize = (offset_sub, offset_add, step[, truncate]): uint16 output of the fused quantizer; step may be a
    StepTable of the whole z_total-plane volume (checked here, before stage 1 and the exchange).
    model (PoissonGaussian, the same on every rank): through the GAT, `sigma` is then sigma_vst; value_hist as
    vst_value_hist; first = the whole volume's voxel (0, 0, 0), taken from the slab when it starts at plane 0."""
    import torch

    from .api import _step_table_args, _table_of

    table = _table_of(quantize)
    if table is not None:
        if model is not None:
            raise NotImplementedError("a step table on the VST path is not implemented")
        _step_table_args(table, tuple(slab.shape), z_begin, z_total)
    if model is None:
        denoiser.slab_stage1(slab, z_begin, z_total, sigma)
    else:
        if first is None:
            if z_begin != 0:
                raise ValueError("the VST slab form needs `first`, the whole volume's voxel (0, 0, 0)")
            first = int(slab[0, 0, 0])
        value_hist = vst_value_hist(denoiser, slab[own_begin - z_begin : own_end - z_begin], world, value_hist,
                                    device, group)
        denoiser.slab_stage1_vst(slab, z_begin, z_total, model, value_hist, first, sigma)
    lo_h, hi_h = own_begin - z_begin, (z_begin + slab.shape[0]) - own_end
    if (rank > 0 and own_end - own_begin < lo_h) or (rank < world - 1 and own_end - own_begin < hi_h):
        raise ValueError("every rank must own at least as many planes as the halo")
    o0, o1 = own_begin - z_begin, own_end - z_begin  # owned planes, slab-local
    if device is not None and world > 1 and os.environ.get("B4D_EXCHANGE_OVERLAP", "1") != "0":
        # device path: the exchange reads and writes the handle's basic-estimate buffer in place (no staging
        # copies) and overlaps the part of the stage-2 front end that needs owned planes only
        basic = denoiser.slab_basic_tensor(device)
        denoiser.slab_stage2_begin(own_begin, own_end)
        exchange_planes(basic[o0 : o0 + lo_h] if rank > 0 else None, basic[o1 - hi_h : o1] if rank < world - 1 else None,
                        basic[0:lo_h] if rank > 0 else None, basic[o1 : o1 + hi_h] if rank < world - 1 else None,
                        rank, world, group)
        torch.cuda.current_stream(device).synchronize()  # the received planes are in place
        return denoiser.slab_stage2(own_begin, own_end, out=out, device=device if out is None else None,
                                    quantize=quantize)

    def planes(p0, n):
        t = denoiser.slab_basic(p0, n, device=device)
        return t if device is not None else torch.from_numpy(t)

    send_down = planes(o0, lo_h) if rank > 0 else None           # the neighbour's upper halo
    send_up = planes(o1 - hi_h, hi_h) if rank < world - 1 else None
    hw = tuple(slab.shape[1:])
    mk = (lambda n: torch.empty((n,) + hw, dtype=torch.float32, device=device)) if device is not None else (
        lambda n: torch.empty((n,) + hw, dtype=torch.float32))
    recv_below = mk(lo_h) if rank > 0 else None
    recv_above = mk(hi_h) if rank < world - 1 else None
    exchange_planes(send_down, send_up, recv_below, recv_above, rank, world, group)
    if recv_below is not None:
        denoiser.slab_set_basic(0, recv_below if device is not None else recv_below.numpy())
    if recv_above is not None:
        denoiser.slab_set_basic(o1, recv_above if device is not None else recv_above.numpy())
    return denoiser.slab_stage2(own_begin, own_end, out=out, device=device if out is None else None, quantize=quantize)


def denoise_volume_sharded(get_slab, z_total, sigma, denoiser, world=1, rank=0, exchange=False, device=None,
                           model=None, value_hist=None):
    """Denoise this rank's share of a (z_total, H, W) uint16 volume.

    get_slab(z_begin, z_end) -> uint16 array/tensor of those planes (host or
    device).  Returns (own_begin, own_end, float32 planes).  With `exchange`
    (needs an initialised process group when world > 1) the slabs carry half the
    halo and neighbours swap basic-estimate planes between the stages.
    model (PoissonGaussian, the same on every rank): denoise through the GAT
    (DESIGN §3.12) with `sigma` as sigma_vst; the value set is `value_hist` (the
    whole volume's 65536 counts) or, when None, the owned planes' histograms
    merged across the ranks (world > 1 then needs an initialised process group).
    """
    p = denoiser.profile
    ns1, ns2 = 2 * int(np.ravel(p.search_window_ht)[0]) + 1, 2 * int(np.ravel(p.search_window_wiener)[0]) + 1
    if model is not None and value_hist is None and world > 1 and not _process_group_ready():
        raise ValueError("world > 1 needs an initialised process group, or the whole volume's value_hist")
    first = None if model is None else int(get_slab(0, 1)[0, 0, 0])
    if exchange and denoiser._stages == 2 and world > 1:
        own_begin, own_end, z_begin, z_end = slab_plan(z_total, world, rank, exchange_halo(ns1, ns2))
        out = denoise_slab_exchange(denoiser, get_slab(z_begin, z_end), z_begin, z_total, own_begin, own_end, sigma,
                                    rank, world, device=device, model=model, value_hist=value_hist, first=first)
        return own_begin, own_end, out
    own_begin, own_end, z_begin, z_end = slab_plan(z_total, world, rank, halo_planes(ns1, ns2, denoiser._stages))
    slab = get_slab(z_begin, z_end)
    if model is None:
        out = denoiser.denoise_slab(slab, z_begin, z_total, own_begin, own_end, sigma)
    else:
        value_hist = vst_value_hist(denoiser, slab[own_begin - z_begin : own_end - z_begin], world, value_hist,
                                    device)
        out = denoiser.denoise_slab_vst(slab, z_begin, z_total, own_begin, own_end, model, value_hist, first, sigma)
    return own_begin, own_end, out


def bind_to_gpu_numa(device):
    """Pin this process (and the threads it starts later) to the CPUs next to GPU `device`, so that pinned
    host buffers and the copy threads of the library sit on the GPU's NUMA node — with one process per
    GPU on a multi-socket host, PCIe copies from the far socket are the first thing to slow down.
    Call it before allocating host buffers.  Returns the number of CPUs bound to, or None when NVML or
    the topology is unavailable (nothing is changed then)."""
    import os

    try:
        import pynvml
        import torch

        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(int(device))
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        handle = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        before = os.sched_getaffinity(0)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        after = os.sched_getaffinity(0)
        if not after:
            os.sched_setaffinity(0, before)
            return None
        return len(after)
    except Exception:
        return None


def merge_histograms(hist, group=None):
    """All-gather + sum of per-rank histograms of any length (the path's only
    collective): the 65536-bin intensity histograms of tile_stats or the 262141-bin
    |d| histograms of noise_sigma.  `hist` is an int64 torch tensor on the rank's
    device (NCCL) or on the CPU (gloo).  Without an initialised process group it is
    returned as is."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return hist
    world = dist.get_world_size(group)
    gathered = [torch.empty_like(hist) for _ in range(world)]
    dist.all_gather(gathered, hist, group=group)
    return torch.stack(gathered, 0).sum(0)


def stats_from_hist_lib(hist, percentile=1.0):
    """The same statistics through libb4d's own host routine (b4d_stats_from_hist): what the ranks call on the
    summed histogram inside the timed step (0.1 ms instead of the milliseconds of the NumPy form below)."""
    import ctypes

    from . import _lib

    h = np.ascontiguousarray(hist, dtype=np.int64)
    if h.shape != (65536,):
        raise ValueError("hist must have 65536 bins")
    st = _lib.Stats()
    _lib.check(_lib.load().b4d_stats_from_hist(h.ctypes.data, percentile, ctypes.byref(st)))
    return {k: getattr(st, k) for k, _ in _lib.Stats._fields_}


def stats_from_hist(hist, percentile=1.0):
    """Offset percentile over non-zero voxels, median, MAD, sigma from an exact
    uint16 histogram, with NumPy-2 float32 semantics (float32 virtual index and
    interpolation) — the same arithmetic libb4d's b4d_tile_stats performs."""
    f32 = np.float32
    h = np.asarray(hist, dtype=np.int64)
    n = int(h.sum())
    if n == 0:
        raise ValueError("empty histogram")

    def order_stat(hh, k):
        return int(np.searchsorted(np.cumsum(hh), k, side="right"))

    def pct(hh, first, cnt, p):
        q = f32(p) / f32(100)
        vi = f32(cnt - 1) * q
        prev = np.floor(vi)
        if vi >= f32(cnt - 1):
            pi = ni = cnt - 1
        elif vi < 0:
            pi = ni = 0
        else:
            pi = int(prev)
            ni = pi + 1
        g = f32(vi - prev)
        sub = hh.copy()
        sub[:first] = 0
        a, b = f32(order_stat(sub, pi)), f32(order_stat(sub, ni))
        d = f32(b - a)
        r = f32(a + f32(d * g))
        if g >= f32(0.5):
            r = f32(b - f32(d * f32(f32(1) - g)))
        return float(r)

    nnz = n - int(h[0])
    offset = pct(h, 1, nnz, percentile) if nnz > 0 else pct(h, 0, n, percentile)
    m_lo, m_hi = order_stat(h, (n - 1) // 2), order_stat(h, n // 2)
    med = f32((f32(m_lo) + f32(m_hi)) * f32(0.5))
    m2 = m_lo + m_hi
    t = np.abs(2 * np.arange(65536, dtype=np.int64) - m2)
    h2 = np.bincount(t, weights=None, minlength=131072) * 0
    np.add.at(h2, t, h)
    a_lo, a_hi = order_stat(h2, (n - 1) // 2), order_stat(h2, n // 2)
    mad = f32(f32((f32(a_lo) * f32(0.5) + f32(a_hi) * f32(0.5)) * f32(0.5)) + f32(1e-6))
    sigma = f32(f32(1.4826) * mad)
    nz = np.nonzero(h)[0]
    return {
        "n": n,
        "n_nonzero": nnz,
        "offset": offset,
        "median": float(med),
        "mad": float(mad),
        "sigma": float(sigma),
        "vmin": float(nz[0]),
        "vmax": float(nz[-1]),
    }
