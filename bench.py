#!/usr/bin/env python
"""bench.py -- headline benchmark: 3D D-LKA block forward at (B,C,D,H,W) = (2,96,64,128,128).

    python bench.py --gpus N --steps K --warmup W            (ours; under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W   (reference arm: CPU oracle)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (also writes the last timed step's output to DIR)

A "step" is one forward of ``LKA_Attention3d_deform`` (proj_1 -> GELU -> dw5^3 -> dw7^3 dil3 ->
conv_offset -> deformable 3^3 conv -> conv1 -> gate -> proj_2 -> +shortcut) over one batch of synthetic
tokens [2, 64*128*128, 96].  Metric: GVoxel/s with voxels = B*D*H*W per step (SURVEY.md 8d).
Multi-GPU: every rank runs the same per-rank batch (weak scaling, no data-path collective, SURVEY 8e).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)

import torch  # noqa: E402

METRIC = "3D D-LKA block fwd GVoxel/s @ (2,96,64,128,128)"
SHAPE = dict(B=2, C=96, D1=64, D2=128, D3=128)
# algorithmic work per voxel at C=96 (SURVEY.md 8d / DESIGN.md): compulsory HBM bytes and tensor-pipe FLOPs
HBM_BYTES_PER_VOXEL = 2 * 96 * 4
CONTRACTION_FLOP_PER_VOXEL = 2 * 27 * 96 * 81 + 2 * 27 * 96 * 96 + 3 * 2 * 96 * 96


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained"),
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # median over the upper half of the samples = under load
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": load[len(load) // 2] if load else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_block(C, device, seed=1234):
    """Parameters: PyTorch default init under seed 1234; the zero-initialised conv_offset is re-initialised
    N(0, 0.05^2) / U(-1, 1) so offsets are non-trivial (BASELINE.md section 3)."""
    import deformablelka_b200 as dl
    torch.manual_seed(seed)
    m = dl.LKA_Attention3d_deform(C)
    g = torch.Generator().manual_seed(seed)
    co = m.spatial_gating_unit.deform_conv.conv_offset
    with torch.no_grad():
        co.weight.copy_(torch.randn(co.weight.shape, generator=g) * 0.05)
        co.bias.copy_(torch.rand(co.bias.shape, generator=g) * 2 - 1)
    return m.to(device).eval()


C4_BLOCKS = ((32, 32, 6), (64, 16, 6), (128, 8, 6), (256, 4, 3))   # (C, cube edge, instances) of the 3D net at batch 2 (SURVEY 3.4)
C2_BLOCKS = ((384, 14), (192, 28), (96, 56))                          # (C, H = W) of the 2D net's decoder blocks at batch 24 (SURVEY 3.3)


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout: libraries that print there (NCCL's version banner on rank 0) are sent to stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, line)


DUMP_SAMPLE = 1 << 22   # elements kept of an output larger than this (16 MB in float32)


def dump_outputs(out_dir, **outputs):
    """--dump-outputs: every output as <out_dir>/<name>.npy, float32, flattened.  An output of more than DUMP_SAMPLE elements is
    written as the elements at DUMP_SAMPLE sorted positions drawn from a generator seeded with 0: the same positions in every
    run, so two builds run with the same arguments can be compared element by element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach().reshape(-1)
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def _time_call(fn, iters=20, warm=5, reps=3):
    """ms per call: CUDA events around `iters` back-to-back calls, median of `reps` such measurements (one host hiccup -- a
    garbage collection, a freed graph pool -- inside a 3 ms window otherwise shows up as a 2-3x outlier on the 0.1 ms shapes)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) / iters)
    return sorted(out)[len(out) // 2]


def other_configs(dl, dev):
    """BASELINE.json configs[1..3] (and the block shapes of configs[3] / [4]) as ms per call of the block / operator that the
    reference network runs at that shape: CUDA events, 5 warm-ups, median of 3 x 20 timed calls, inputs resident, seeded random parameters."""
    out = {}
    with torch.no_grad():
        for C, hw in C2_BLOCKS:
            torch.manual_seed(1234)
            m = dl.deformable_LKA_Attention(C).to(dev).eval()
            x = torch.randn(24, C, hw, hw, device=dev)
            out[f"c2_block2d_24x{C}x{hw}x{hw}_ms"] = _time_call(lambda: m(x))
            g = dl.GraphedCall(m, x)            # same call replayed as one CUDA graph (host launch path out of the way)
            out[f"c2_block2d_24x{C}x{hw}x{hw}_graph_ms"] = _time_call(lambda: g(x))
            del g
        torch.manual_seed(1234)
        B, C, D, H, W = 2, 64, 32, 64, 64
        x = torch.randn(B, C, D, H, W, device=dev); w = torch.randn(C, C, 3, 3, 3, device=dev) * 0.05
        b = torch.randn(C, device=dev); off = torch.randn(B, 81, D, H, W, device=dev)
        out["c3_deform_conv3d_2x64x32x64x64_ms"] = _time_call(lambda: dl.ops.deform_conv3d_forward(x, w, b, off, 3, 1, 1, 1, 1, 1, 64))
        del x, off
        for C, s, _ in C4_BLOCKS:
            m = make_block(C, dev)
            x = torch.randn(2, s * s * s, C, device=dev)
            out[f"c4_block3d_2x{C}x{s}x{s}x{s}_ms"] = _time_call(lambda: m(x, 2, C, s, s, s))
            g = dl.GraphedCall(m, x, 2, C, s, s, s)
            out[f"c4_block3d_2x{C}x{s}x{s}x{s}_graph_ms"] = _time_call(lambda: g(x, 2, C, s, s, s))
            del g
    return out


def gpu_reference_leg(dl, dev):
    """Informational: the reference's OWN CUDA extension (3D/dcn D3D, compiled unmodified apart from the two-token torch-2 patch
    by oracle/build_ref.py into oracle/_ref/) against this library's operator, same GPU, same tensors, BASELINE configs[2]
    (2,64,32,64,64), k=3: forward and backward, ms per call.  None when oracle/_ref was not built."""
    try:
        from oracle import build_ref
        d3d = build_ref.load_d3d()
    except Exception as e:   # noqa: BLE001 -- informational leg, never fails the bench
        return {"unavailable": f"{type(e).__name__}: {e}"}
    if d3d is None:
        return {"unavailable": "oracle/_ref/D3D*.so not built"}
    torch.manual_seed(1234)
    B, C, D, H, W = 2, 64, 32, 64, 64
    x = torch.randn(B, C, D, H, W, device=dev); w = torch.randn(C, C, 3, 3, 3, device=dev) * 0.05
    b = torch.randn(C, device=dev); off = torch.randn(B, 81, D, H, W, device=dev); go = torch.randn(B, C, D, H, W, device=dev)
    geo = (3, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 64)
    out = {"shape": [B, C, D, H, W], "what": "deform_conv3d k=3 s=1 p=1 g=1 dg=1 im2col_step=64"}
    with torch.no_grad():
        out["reference_d3d_forward_ms"] = _time_call(lambda: d3d.deform_conv_forward(x, w, b, off, *geo))
        out["ours_forward_ms"] = _time_call(lambda: dl.ops.deform_conv3d_forward(x, w, b, off, 3, 1, 1, 1, 1, 1, 64))
        out["reference_d3d_backward_ms"] = _time_call(lambda: d3d.deform_conv_backward(x, w, b, off, go, *geo))
        out["ours_backward_ms"] = _time_call(lambda: dl.ops.deform_conv3d_backward(x, w, b, off, go, 3, 1, 1, 1, 1, 1, 64))
    return out


def run_c4net(args, dl, dev, world, rank):
    """--config c4net: one step = the 21 D-LKA attention blocks of the 3D D-LKA Net forward (SURVEY 3.4) at per-rank batch 2
    (BASELINE configs[3]; under torchrun with 8 ranks = configs[4], global batch 16, batch-sharded, no collective)."""
    from deformablelka_b200.dist import max_over_ranks
    blocks = []
    with torch.no_grad():
        for C, s, n in C4_BLOCKS:
            m = make_block(C, dev)
            x = torch.randn(2, s * s * s, C, device=dev)
            blocks.append((m, x, C, s, n))

        def step():
            for m, x, C, s, n in blocks:
                for _ in range(n):
                    m(x, 2, C, s, s, s)

        n_a = dl.launch_count()
        for _ in range(args.warmup):
            step()
        launches_per_step = (dl.launch_count() - n_a) // max(args.warmup, 1)
        torch.cuda.synchronize()
        run = step
        if not args.no_graph:   # the 21 calls of a step recorded ONCE as a CUDA graph; every timed step replays the same kernels
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                step()
            run = graph.replay
            run()
            torch.cuda.synchronize()
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            run()
        e1.record()
        torch.cuda.synchronize()
        ms = max_over_ranks(e0.elapsed_time(e1), dev) / args.steps
        launches = launches_per_step * args.steps   # kernels executed in the timed region (replayed from the graph when graphed)
    if rank == 0:
        emit(({
            "metric": "3D D-LKA Net, D-LKA block path fwd (21 blocks), patches/s @ batch 2 per GPU", "value": 2 * world / (ms * 1e-3),
            "unit": "patches/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE configs[3]/[4]: LKA_Attention3d_deform at the 21 block shapes of the 3D net, 64x128x128 patches",
                       "blocks": [list(b) for b in C4_BLOCKS], "math": args.math, "parallelism": f"dp{world}",
                       "launch": "eager" if args.no_graph else "cuda_graph (one graph per step)"},
            "gpu_launches": int(launches)}))


def cpu_threads():
    """One software thread per PHYSICAL core, capped at 64: the torch intra-op pool and the C oracle's OpenMP team share the
    same libgomp, and with every hyper-thread in both the sample time swung 4.6x between two boxes (VERDICT r1 weak #6)."""
    n = os.cpu_count() or 1
    try:
        import psutil
        n = psutil.cpu_count(logical=False) or n
    except Exception:
        pass
    return max(1, min(n, 64))


_CPU_MODEL = {}


def cpu_reference_model(C, threads):
    if C not in _CPU_MODEL:
        os.environ["OMP_NUM_THREADS"] = str(threads)      # read by libgomp when the oracle's C library first runs
        from oracle import oracle
        torch.set_num_threads(threads)
        torch.manual_seed(1234)
        m = oracle.LKA_Attention3d_deform(C).eval()
        oracle.randomize_offsets_(m, std=0.05, bias_range=1.0, seed=1234)
        _CPU_MODEL[C] = m
    return _CPU_MODEL[C]


def cpu_reference_sample(C, threads, sample_dims=(16, 64, 64), iters=3, warm=1):
    """The reference's CPU implementation of the path = the oracle (stock nn.Conv3d/GELU + restated D3D) on a
    bounded sample of the workload: one sub-volume [1, C, 16, 64, 64] (1/32 of the step's voxels); `warm` untimed passes,
    then the MEDIAN of `iters` timed passes."""
    m = cpu_reference_model(C, threads)
    d1, d2, d3 = sample_dims
    x = torch.randn(1, d1 * d2 * d3, C, generator=torch.Generator().manual_seed(1234))
    times = []
    with torch.no_grad():
        for i in range(warm + iters):
            t0 = time.perf_counter()
            m(x, 1, C, d1, d2, d3)
            if i >= warm:
                times.append(time.perf_counter() - t0)
    vox = d1 * d2 * d3
    times.sort()
    t = times[len(times) // 2]
    return vox / t / 1e9, t, (f"1x{C}x{d1}x{d2}x{d3} sub-volume of the step ({vox} of {2 * 64 * 128 * 128} voxels), "
                              f"{warm} warm-up + median of {iters}, {threads} threads")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = cpu_threads()
    vals = []
    sample = ""
    for i in range(args.warmup + args.steps):      # each step = one pass over the bounded sample
        v, t, sample = cpu_reference_sample(SHAPE["C"], threads, iters=1, warm=0)
        if i >= args.warmup:
            vals.append((v, t))
    vals.sort(key=lambda vt: vt[1])
    v, t = vals[len(vals) // 2]                    # median step (robust against a noisy neighbour on the host)
    sample = sample.replace("0 warm-up + median of 1", f"{args.warmup} warm-up steps + median of {args.steps} steps")
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "GVoxel/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "LKA_Attention3d_deform fwd, tokens [2, 64*128*128, 96] (3D D-LKA block)", "reference_arm":
                   "oracle port of the reference CPU path (D3D is CUDA-only, 3D/dcn/src/deform_conv.h:46); each step = one bounded sample"},
        "cpu_baseline": {"value": v, "unit": "GVoxel/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "GVoxel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--math", default=os.environ.get("DLKA_MATH", "bf16x3"))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--config", default="headline", choices=["headline", "c4net"], help="c4net: BASELINE configs[3] / [4] (block path)")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="c4net: launch the 21 block calls eagerly instead of replaying one CUDA graph")
    ap.add_argument("--no-profile-pass", action="store_true", help="skip the per-kernel event pass (tools/measure_traffic.py)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output of the last timed step to DIR/y.npy (float32; a seeded "
                    f"sample of {DUMP_SAMPLE} of its elements, see dump_outputs); rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != "headline"):
        ap.error("--dump-outputs applies to the headline workload of --impl ours")
    if args.warmup < 3:
        args.warmup = 3
    quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (ours) needs a CUDA device: there is no CPU path"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    os.environ["DLKA_MATH"] = args.math
    import deformablelka_b200 as dl
    # host side of the e2e path: this rank's thread on the GPU's NUMA node, pinned buffers placed there (ops.pinned_empty)
    numa_node = dl.ops.bind_host_thread(dev) if os.environ.get("DLKA_HOST_NUMA", "local") != "off" else -1

    if args.config == "c4net":
        run_c4net(args, dl, dev, world, rank)
        if world > 1:
            dist.destroy_process_group()
        return
    B, C, D1, D2, D3 = (SHAPE[k] for k in ("B", "C", "D1", "D2", "D3"))
    N = D1 * D2 * D3
    vox = B * N
    m = make_block(C, dev)
    torch.manual_seed(1234 + rank)
    x = torch.randn(B, N, C, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step():
        return m(x, B, C, D1, D2, D3)

    with torch.no_grad():
        for _ in range(args.warmup):
            y = step()
        barrier()
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        n0 = dl.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            y = step()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = dl.launch_count() - n0
        clocks = sampler.stop() if rank == 0 else None
        from deformablelka_b200.dist import max_over_ranks
        ms_total = max_over_ranks(ms, dev)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, y=y)     # y: the block output [B, N, C] of the last timed step

        # per-kernel durations over the same K steps (CUDA events on the launch stream, inside the library)
        prof = {}
        if not args.no_profile_pass:
            dl._lib.profile_enable(True)
            for _ in range(args.steps):
                y = step()
            torch.cuda.synchronize()
            prof = dl._lib.profile_summary()
            dl._lib.profile_enable(False)

        # end-to-end through the module API with host buffers: pinned H2D of the step input, D2H of the result
        e2e = None
        if not args.no_e2e:
            wc = os.environ.get("DLKA_HOST_WC", "0") == "1"     # write-combined input buffer (the host only writes it)
            xh = dl.ops.pinned_empty((B, N, C), dev, write_combined=wc)
            yh = dl.ops.pinned_empty((B, N, C), dev)
            xh.copy_(torch.randn(B, N, C, generator=torch.Generator().manual_seed(4321 + rank)))   # writes only (a write-combined buffer must not be read)
            # streaming serving loop through the public module API: every step copies its input from pinned host memory
            # and its result back to pinned host memory; the pipeline keeps 2 steps in flight (H2D of step k+1 and D2H of
            # step k-1 overlap the compute of step k).
            pipe = m.host_pipe(depth=int(os.environ.get("DLKA_PIPE_DEPTH", "2")))
            ksteps = max(4, args.steps)
            for _ in range(3):
                m.submit_host(pipe, xh, yh, B, C, D1, D2, D3)
            pipe.wait()

            def e2e_region(k):
                """k steps from an EMPTY pipe to the last result on the host: includes the pipeline fill (H2D of the first sample,
                nothing to overlap it with) and drain (D2H of the last sample)."""
                barrier()
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                f0.record()
                for _ in range(k):
                    m.submit_host(pipe, xh, yh, B, C, D1, D2, D3)
                pipe.join()          # current stream now waits for the last D2H copy
                f1.record()
                pipe.wait()
                barrier()
                return max_over_ranks(f0.elapsed_time(f1), dev)

            e2e_ms = e2e_region(ksteps)
            e2e = {"value": world * vox * ksteps / (e2e_ms * 1e-3) / 1e9, "unit": "GVoxel/s",
                   "h2d_bytes_per_step": xh.numel() * 4, "d2h_bytes_per_step": yh.numel() * 4, "steps": ksteps}
            # informational: the same loop over 2K steps; (T(2K) - T(K)) / K is the per-step time of the running pipeline with the
            # fixed fill + drain (~14 ms at this shape: one sample each way with nothing to overlap) taken out.  `value` above keeps them.
            e2e_ms2 = e2e_region(2 * ksteps)
            steady_ms = (e2e_ms2 - e2e_ms) / ksteps
            e2e["steady_state"] = {"value": world * vox / (steady_ms * 1e-3) / 1e9, "ms_per_step": steady_ms,
                                   "fill_drain_ms": e2e_ms - ksteps * steady_ms, "method": "(T(2K) - T(K)) / K, both regions start from an empty pipe"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    others = None
    if world == 1 and not args.no_other_configs:
        del x, y
        torch.cuda.empty_cache()
        others = other_configs(dl, dev)
        others["gpu_reference"] = gpu_reference_leg(dl, dev)

    pk = peaks()
    # DRAM traffic per launch: measured by tools/measure_traffic.py (ncu) and used only if it was measured on THESE sources
    traffic, traffic_note = {}, "profiles/traffic.json absent"
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from measure_traffic import csrc_sha
        tj = json.load(open(tp))
        if tj.get("csrc_sha") == csrc_sha():
            traffic = {k: v["dram_bytes_per_launch"] for k, v in tj["kernels"].items()}
            traffic_note = f"ncu, measured on these sources (csrc {tj['csrc_sha']}, git {tj.get('git_head')})"
        else:
            traffic_note = f"stale: measured on csrc {tj.get('csrc_sha')}, running {csrc_sha()}"
    ms_step = ms_total / args.steps
    value = world * vox / (ms_step * 1e-3) / 1e9
    # dominant kernel by device time
    dom = max(prof.items(), key=lambda kv: kv[1][1]) if prof else (None, (1, float("nan")))
    dom_name, (dom_n, dom_ms) = dom
    dom_avg_ms = dom_ms / max(dom_n, 1)
    launches_per_step = {k: v[0] / args.steps for k, v in prof.items()}
    total_prof_ms = sum(v[1] for v in prof.values())
    # Roofline of the dominant kernel.  The contract's two bounds (tensor FLOP/s, HBM bytes/s) are reported for it, and -- for the
    # deformable kernel, where neither binds -- the bound that does: the SM's L1TEX data pipe (one 128-byte wavefront per cycle and
    # SM for global lines, shared-memory accesses, shuffles and UMMA operand reads alike; DESIGN.md 4).  Its algorithmic work is
    # the trilinear gather: 8 corners x 27 taps x C/32 lines of 128 bytes per voxel, every one of which must cross that pipe.
    per_launch_flop = {
        "igemm_simt_deform": 2 * 27 * C * C * vox, "igemm_simt_conv": 2 * 27 * C * 81 * vox,
        "tc_deform": 2 * 27 * C * C * vox, "tc_conv": 2 * 27 * C * 81 * vox, "tc_conv_tiled": 2 * 27 * C * 81 * vox,
        "tc_deform3d": 2 * 27 * C * C * vox, "tc_deform3d_chain": (2 * 27 * C * C + 2 * 2 * C * C) * vox,
        "tc_dense": 2 * C * C * vox,
    }
    per_launch_hbm = {   # compulsory bytes of each kernel: what it must read and write once
        "tc_deform3d_chain": (4 * C * 4 + 81 * 4) * vox,   # a (gather source), u (gate), x (residual) in, y out, offsets in
        "tc_conv_tiled": (C * 4 + 81 * 4) * vox, "tc_dense": 2 * C * 4 * vox,
        "dwconv3d_smem_k5": 2 * C * 4 * vox, "dwconv3d_smem_k7d3": 2 * C * 4 * vox,
    }
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    share = dom_ms / total_prof_ms if total_prof_ms else None
    tensor = None
    if dom_name in per_launch_flop:
        ach = per_launch_flop[dom_name] / (dom_avg_ms * 1e-3) / 1e12
        tensor = {"achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"],
                  "peak_source": pk["source"] + " bf16 burst"}
    hbm_bytes = per_launch_hbm.get(dom_name, HBM_BYTES_PER_VOXEL * vox)
    ach_hbm = hbm_bytes / (dom_avg_ms * 1e-3) / 1e9
    hbm = {"achieved": ach_hbm, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach_hbm / pk["hbm_gbs"], "peak_source": pk["source"],
           "algorithmic_bytes": hbm_bytes}
    if dom_name and dom_name.startswith("tc_deform3d"):
        lines = vox * 27 * 8 * (C // 32)
        peak_l1 = 148 * 128 * sm_mhz * 1e6 / 1e9          # GB/s: 128 bytes per clock and SM at the SM clock seen during the run
        ach_l1 = lines * 128 / (dom_avg_ms * 1e-3) / 1e9
        roof = {"bound": "l1tex_data_pipe", "kernel": dom_name, "achieved": ach_l1, "peak": peak_l1, "unit": "GB/s",
                "frac": ach_l1 / peak_l1, "traffic": traffic.get(dom_name), "avg_launch_ms": dom_avg_ms, "share_of_step": share,
                "peak_source": f"148 SMs x 128 B/clk x {sm_mhz:.0f} MHz (L1TEX data pipe, one wavefront per cycle; ncu: "
                               "l1tex__data_pipe_lsu_wavefronts + l1tex__data_pipe_tc_wavefronts ~ elapsed cycles)",
                "algorithmic_bytes": lines * 128, "gather_lines_128B": lines,
                "note": "the gather alone is 1024 of the ~2000 wavefronts of a K step (profiles/r02_deform_ps_l1tex.txt); "
                        "tensor and hbm are the contract's bounds for the same kernel and do not bind",
                "tensor": tensor, "hbm": hbm}
    elif tensor is not None and dom_name != "tc_dense":
        roof = dict(tensor, bound="tensor", kernel=dom_name, traffic=traffic.get(dom_name), avg_launch_ms=dom_avg_ms, share_of_step=share,
                    hbm=hbm)
    else:
        roof = dict(hbm, bound="hbm", kernel=dom_name, traffic=traffic.get(dom_name), avg_launch_ms=dom_avg_ms, share_of_step=share,
                    tensor=tensor)
    roof["traffic_source"] = traffic_note
    out = {
        "metric": METRIC, "value": value, "unit": "GVoxel/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "LKA_Attention3d_deform fwd, tokens [2, 64*128*128, 96] per GPU (3D D-LKA block at (2,96,64,128,128))",
                   "math": args.math, "parallelism": f"dp{world} (batch-sharded replicas, no collective in the timed region)",
                   "l2": "inputs 805 MB per tensor > 126 MB L2 (no flush needed)",
                   "params": "default init seed 1234; conv_offset ~ N(0,0.05^2), bias U(-1,1)",
                   "host": f"rank thread + pinned e2e buffers on NUMA node {numa_node} of the GPU (DLKA_HOST_NUMA="
                           f"{os.environ.get('DLKA_HOST_NUMA', 'local')})"},
        "block_hbm_frac": HBM_BYTES_PER_VOXEL * vox / (ms_step * 1e-3) / 1e9 / pk["hbm_gbs"],
        "block_contraction_tflops": CONTRACTION_FLOP_PER_VOXEL * vox / (ms_step * 1e-3) / 1e12,
        "roofline": roof,
        "kernels_ms_per_step": {k: v[1] / args.steps for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])},
        "gpu_launches": int(launches),
        "clocks": clocks,
    }
    if e2e is not None:
        out["e2e"] = e2e
    if others is not None:
        out["other_configs"] = others
    if world == 1 and not args.no_cpu_baseline:
        threads = cpu_threads()
        v, t, sample = cpu_reference_sample(C, threads)
        out["cpu_baseline"] = {"value": v, "unit": "GVoxel/s", "cores": threads, "kind": "port", "sample": sample,
                               "seconds": t}
    emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
