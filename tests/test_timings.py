"""Launch accounting of b4d_last_timings: every b4d_last_* value describes the whole last public call, and the launch
count of a kernel family is the number of kernels enqueued in the intervals it books.

Every launcher enqueues through b4d_launch (csrc/b4d_common.cuh), which counts; the host pipeline books the count
since the previous stage mark.  The CPU test checks that no kernel can be enqueued around it; the GPU tests compare
the booked counts with the kernels the CUDA profiler records for each denoising path.
"""
import json
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "aind-exaspim-image-compression_b200", "csrc")


def test_every_kernel_launch_goes_through_the_counting_helper():
    """Outside b4d_launch no source file under csrc/ contains a launch (triple chevron), so no kernel is enqueued
    without being counted."""
    sites = []
    for name in sorted(os.listdir(CSRC)):
        if not name.endswith((".cu", ".cuh", ".h", ".cpp")):
            continue
        with open(os.path.join(CSRC, name)) as f:
            sites += [(name, i + 1, line.strip()) for i, line in enumerate(f) if "<<<" in line]
    assert len(sites) == 1, sites
    name, _, line = sites[0]
    assert name == "b4d_common.cuh" and re.match(r"kernel<<<grid, block, smem, s>>>\(", line), sites
    with open(os.path.join(CSRC, name)) as f:
        src = f.read()
    helper = src[src.index("inline void b4d_launch("):]
    assert helper.index("<<<") < helper.index("++b4d_kernels_enqueued") < helper.index("}")


# ---------------------------------------------------------------------------------------------------------- GPU --

def _launches(d):
    return sum(n for _, n in d.last_timings().values())


def _profiled_kernels(call, tmp_path):
    """Kernels the CUDA profiler records during `call` (memcpy and memset excluded), after one warm-up call."""
    import torch

    call()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        call()
        torch.cuda.synchronize()
    trace = os.path.join(str(tmp_path), "trace.json")
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        events = json.load(f)["traceEvents"]
    return sum(1 for e in events if e.get("cat") == "kernel")


def _vol(D, H, W, seed):
    from b4d import synth

    return synth.vol(D, H, W, seed=seed)


def _case(name):
    """(handle, call, kernels booked to no family on purpose) of one denoising path, on a fresh handle."""
    import torch

    import b4d

    dn = b4d.Denoiser(0)
    v64 = _vol(64, 64, 64, 1)
    if name == "u16_host":
        return dn, (lambda: dn.denoise(v64, 24.0)), 0
    if name == "u16_device":
        t = torch.from_numpy(v64).cuda()
        return dn, (lambda: dn.denoise(t, 24.0)), 0
    if name == "f32":
        f = v64.astype(np.float32)
        return dn, (lambda: dn.denoise(f, 24.0)), 0
    if name == "f32_dc_centred":  # a large DC level: denoised on z - c0, c0 added back unbooked
        f = v64.astype(np.float32) + 1.0e6
        return dn, (lambda: dn.denoise(f, 24.0)), 1
    if name == "q16":
        return dn, (lambda: dn.denoise_quantized(v64, 24.0, 10.0, 0.0, 2.0)), 0
    if name == "slab":
        return dn, (lambda: dn.denoise_slab(v64[8:56], 8, 64, 16, 48, 24.0)), 0
    if name == "two_call":
        def call():
            dn.slab_stage1(v64[8:56], 8, 64, 24.0)
            dn.slab_stage2(16, 48)
        return dn, call, 0
    if name == "two_call_begin":
        def call():
            dn.slab_stage1(v64[8:56], 8, 64, 24.0)
            dn.slab_stage2_begin(16, 48)
            dn.slab_stage2(16, 48)
        return dn, call, 0
    if name == "streamed_upload_chunked_sink":
        deep = _vol(208, 16, 20, 12)  # 69 reference planes: enough for 8 chunks
        dn.set_pipeline_min_voxels(0)
        return dn, (lambda: dn.denoise(deep, 24.0)), 0
    if name == "oversize":
        tall = _vol(100, 24, 28, 21)
        dn.set_pass_voxels(60 * 24 * 28)  # 13 slabs
        return dn, (lambda: dn.denoise(tall, 24.0)), 0
    if name == "vst":
        model = b4d.PoissonGaussian(2.0, 10.0, 1.0)
        return dn, (lambda: dn.denoise_vst(v64, model, 1.0)), 0
    if name == "targets_two_chunks":
        batch = np.stack([_vol(24, 24, 24, s) for s in range(4)])
        dn.set_pass_voxels(2 * 24 ** 3)
        return dn, (lambda: dn.targets(batch, np.float32(5.0), 24.0, 4000.0)), 2 * 2  # offset subtraction + clip
    if name == "match_stage1":
        return dn, (lambda: dn.match_stage1(v64, 24.0)), 1  # block energies ahead of the instrumented matcher
    raise KeyError(name)


CASES = ["u16_host", "u16_device", "f32", "f32_dc_centred", "q16", "slab", "two_call", "two_call_begin",
         "streamed_upload_chunked_sink", "oversize", "vst", "targets_two_chunks", "match_stage1"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_booked_launches_equal_the_kernels_the_profiler_records(name, tmp_path):
    dn, call, unbooked = _case(name)
    try:
        kernels = _profiled_kernels(call, tmp_path)
        booked = _launches(dn)
        print("%s: %d kernels, %d booked %s" % (name, kernels, booked, {k: v[1] for k, v in dn.last_timings().items()}))
        assert booked + unbooked == kernels
        if name == "streamed_upload_chunked_sink":  # both pipelined paths ran
            tm = dn.last_timings()
            assert tm["match1"][1] > 8 and tm["norm2"][1] > 1, tm
    finally:
        dn.close()


@pytest.mark.gpu
def test_match_stats_of_a_chunked_batch_are_the_sum_over_its_volumes():
    import b4d

    vols = [_vol(24, 28, 32, s) for s in (31, 32)]
    dn = b4d.Denoiser(0)
    try:
        want = {}
        for v in vols:
            dn.denoise(v, 24.0)
            for k, n in dn.last_match_stats().items():
                want[k] = want.get(k, 0) + n
        dn.set_pass_voxels(vols[0].size)  # one volume per pass: two chunks
        dn.denoise(np.stack(vols), 24.0)
        assert dn.last_match_stats() == want
        assert sum(want.values()) > 0
    finally:
        dn.close()
