"""BASELINE configs[4] end to end on the GPU box: one uint16 volume (default 1024 x 2048 x 2048, z,y,x)
sharded in z-slabs over the ranks -> tile statistics (histogram all-gather) -> BM4D denoise (13-plane
halos + one neighbour exchange) -> offset-subtract + quantize at step 1, at step = kappa * sigma and at
a step per 64^3 chunk (kappa * the chunk's noise_sigma, the table assembled by an all-gather of the ranks' rows) ->
64^3 chunk gather + byte shuffle + byte counts on the device -> entropy bound of the compressed size,
and real zstd (host, system libzstd) on a sample of the shuffled pieces.  numcodecs/Blosc is absent
here, so the zstd figure approximates the reference's cratio (b4d/codec.py).  Developer tool.

  torchrun --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29517 tools/config5_e2e.py
"""
import argparse, json, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "aind-exaspim-image-compression_b200")); sys.path.insert(0, ROOT)
import numpy as np
import torch
import torch.distributed as dist
import b4d
from b4d import codec, synth
from b4d.sharding import denoise_slab_exchange, exchange_halo, halo_planes, merge_histograms, slab_plan, stats_from_hist

SIGMA, SEED, NS = 24.0, 5, 11


def make_slab(shape, zb, ze, device):
    D, H, W = shape
    clean = torch.from_numpy(synth.clean_tile(SEED)).to(device)
    T = clean.shape[0]
    tile = clean.repeat(1, (H + T - 1) // T, (W + T - 1) // T)[:, :H, :W]
    out = torch.empty((ze - zb, H, W), dtype=torch.uint16, device=device)
    for c in range(zb // T, (ze - 1) // T + 1):
        a, b = max(zb, c * T), min(ze, (c + 1) * T)
        g = torch.Generator(device=device); g.manual_seed(SEED * 1000003 + c)
        for z in range(a, b, 16):  # 16 planes at a time keeps the float scratch small
            z1 = min(b, z + 16)
            noise = torch.randn((z1 - z, H, W), generator=g, device=device) * SIGMA
            v = tile[z - c * T : z1 - c * T] + noise
            out[z - zb : z1 - zb] = torch.clamp(torch.round(v), 0, 65535).to(torch.int32).to(torch.uint16)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", type=int, nargs=3, default=[1024, 2048, 2048])
    ap.add_argument("--kappa", type=float, default=0.5)
    ap.add_argument("--zstd-pieces", type=int, default=48, help="pieces per rank and variant compressed on the host")
    ap.add_argument("--steps", type=int, default=2)
    args = ap.parse_args()
    world, rank, local = (int(os.environ.get(k, d)) for k, d in (("WORLD_SIZE", "1"), ("RANK", "0"), ("LOCAL_RANK", "0")))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    D, H, W = args.shape
    exchange = world > 1
    halo = exchange_halo(NS, NS) if exchange else halo_planes(NS, NS, 2)
    own_b, own_e, zb, ze = slab_plan(D, world, rank, halo)
    dn = b4d.Denoiser(local)
    slab = make_slab((D, H, W), zb, ze, dev)
    own = slab[own_b - zb : own_e - zb]
    # the per-chunk variant: every rank measures sigma on whole 64-plane tile layers of its own planes
    if D % (64 * world):
        raise SystemExit("the step-per-chunk variant needs D divisible by 64 x ranks (owned planes = whole tile layers)")
    assert own_b % 64 == 0 and (own_e - own_b) % 64 == 0, (own_b, own_e)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(); torch.cuda.synchronize()

    def step():
        st, hist = dn.tile_stats(own, 0.1, return_hist=True)  # production percentile (transforms.py:414-438)
        if world > 1:
            st = stats_from_hist(merge_histograms(torch.from_numpy(hist).to(dev)).cpu().numpy(), 0.1)
        if exchange:
            y = denoise_slab_exchange(dn, slab, zb, D, own_b, own_e, SIGMA, rank, world, device=dev)
        else:
            y = dn.denoise_slab(slab, zb, D, own_b, own_e, SIGMA)
        step_k = b4d.noise_scaled_step(st["sigma"], args.kappa)
        rows = torch.from_numpy(dn.noise_sigma(own, tile=(64, 64, 64))["sigma"]).to(dev)
        if world > 1:
            parts = [torch.empty_like(rows) for _ in range(world)]
            dist.all_gather(parts, rows)
            rows = torch.cat(parts, 0)
        table = b4d.noise_scaled_steps(rows, args.kappa, (64, 64, 64))
        q1 = dn.quantize(y, offset_sub=float(st["offset"]), offset_add=0.0, step=1.0)
        qk = dn.quantize(y, offset_sub=float(st["offset"]), offset_add=0.0, step=step_k)
        qt = dn.quantize(y, offset_sub=float(st["offset"]), offset_add=0.0, step=table, z_begin=own_b)
        del y
        s1 = dn.chunk_shuffle(q1, (64, 64, 64))
        sk = dn.chunk_shuffle(qk, (64, 64, 64))
        stt = dn.chunk_shuffle(qt, (64, 64, 64))
        return st, step_k, table, s1, sk, stt

    step(); barrier()
    ext = torch.cuda.ExternalStream(dn.stream_ptr(), device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for _ in range(args.steps):
        st, step_k, table, s1, sk, stt = step()
    e1.record(ext); barrier()
    t = torch.tensor([e0.elapsed_time(e1) * 1e-3 / args.steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    s0 = dn.chunk_shuffle(own, (64, 64, 64))

    # entropy bound (all pieces) and real zstd level 6 (a sample of pieces) per variant; totals over ranks
    grid = codec.chunk_grid(tuple(own.shape), (64, 64, 64))
    pick = np.linspace(0, len(grid) - 1, min(args.zstd_pieces, len(grid))).astype(int)
    tot = []
    t_host = time.perf_counter()
    for by, hist in (s0, s1, sk, stt):
        h = hist.cpu().numpy()
        raw_b, ent_b = float(h.sum()), float(np.maximum(codec.entropy_bytes(h), 1.0).sum())
        zu = zc = 0.0
        if codec.zstd_available():
            for i in pick:
                _, d, pos = grid[i]
                nb = 2 * d[0] * d[1] * d[2]
                zc += codec.zstd_compress(by[pos : pos + nb].cpu().numpy(), 6).size + codec.BLOSC_HEADER + codec.BLOSC_BSTART
                zu += nb
        tot += [raw_b, ent_b, zu, zc]
    t_host = time.perf_counter() - t_host
    tt = torch.tensor(tot, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt)
    if rank == 0:
        tt = tt.cpu().numpy().reshape(4, 4)
        names = ("noisy input", "denoised, step 1", "denoised, step %.3g (kappa %.2g)" % (step_k, args.kappa),
                 "denoised, step per 64^3 chunk (kappa %.2g, steps %.3g .. %.3g)"
                 % (args.kappa, float(table.steps.min()), float(table.steps.max())))
        res = {
            "config": "BASELINE configs[4]: %dx%dx%d uint16, denoise + offset + quantize + chunk shuffle, %d x B200" % (D, H, W, world),
            "seconds_per_volume_device": float(t.item()), "voxels_per_s": D * H * W / float(t.item()),
            "stats": {k: st[k] for k in ("offset", "median", "sigma")},
            "cratio": {n: {"entropy_bound": r[0] / r[1], "zstd6_shuffled_sample": (r[2] / r[3]) if r[3] else None}
                       for n, r in zip(names, tt)},
            "zstd_pieces_per_rank": int(len(pick)), "host_codec_seconds_rank0": t_host,
            "codec_note": "numcodecs/Blosc absent: zstd level 6 over device-shuffled 64^3 pieces + Blosc's fixed framing "
                          "approximates the reference's compute_cratio (img_util.py:401-441)",
        }
        print(json.dumps(res), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
