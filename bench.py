"""Benchmark of the Wan DiT denoise-step hot path (BASELINE.json metric: denoise-step latency & frames/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--shape A|B] [--impl b200|reference] [--no-extras] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one pass of the hot path over one batch of synthetic input = one denoise step of the DiT block stack
(30 blocks for Wan2.1-T2V-1.3B at 480p: L = 32760 video tokens, dim 1536, 12 heads x 128, ffn 8960, 512 text tokens;
SageSLA top-k 0.1, W8A8 linears, FastNorm) = the loop at rcm/networks/wan2pt1.py:697-698 with random-init weights.
value = 81 frames / (4 denoise steps x step latency)  [frames/s], higher is better; ms_per_step is the step latency.

Multi-GPU (N > 1): the video-token axis is sharded over ranks (128-row aligned); every block does one exchange step for the
attention (turbodiffusion_b200/dist.py), "strong" scaling.

The JSON line carries two roofline objects (W8A8 GEMM vs the MEASURED INT8 tensor peak of profiles/r02_hw_probes.json, and the
fused attention kernel), `cpu_baseline` (the reference's CPU-runnable dense SDPA at the full shape, BASELINE.md 3) and
`extra_configs`: short timed runs of the other BASELINE.json configs (shape B = Wan-14B 720p block stack at this N, the
literal [1,24,32760,64] SageSLA shape, LTX-2 shape C kernels), so the driver's BENCH/SCALE records carry them too.

--impl reference times the reference's own CPU path for this metric: torch SDPA dense attention
(rcm/utils/attention.py:152-166 body) on the bench's q/k/v shape, on all host cores; each step is ONE layer's attention call
(a bounded sample: 1 of `layers` blocks, linears excluded), value scales it by the layer count only.

--dump-outputs DIR writes DIR/step_output.npy after the timed steps: the output of the last timed step in float32, a fixed
sample of its rows (output_sample).  Weights and inputs are seeded, so every run with the same arguments sees the same inputs.
The output is not bit-reproducible: the fused attention sums its linear-attention moments with fp32 atomics in a run-dependent
order, and 30 blocks amplify that.  In three runs of one build at shape A on one B200 (1000 W power limit), every pair of
dumps differed by rel-L2 1.87e-2 (cos 0.99983, max |diff| <= 0.25 at max |y| 6.6; profiles/r03_dump_run_to_run.txt, which
lists the commands).  Compare dumps of two builds with a tolerance above that spread.
"""
from __future__ import annotations

import argparse
import contextlib
import datetime
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPES = {
    # name: (L, dim, heads, ffn, layers, text_len, latent T,H,W after patching)
    "A": dict(name="Wan2.1-T2V-1.3B-480p", L=32760, dim=1536, heads=12, ffn=8960, layers=30, text=512, thw=(21, 30, 52)),
    "B": dict(name="Wan2.1-T2V-14B-720p", L=75600, dim=5120, heads=40, ffn=13824, layers=40, text=512, thw=(21, 45, 80)),
}
FRAMES, DENOISE_STEPS = 81, 4
DUMP_BYTES = 48 << 20  # --dump-outputs stays below 64 MB: the full step output is 200 MB (shape A) / 1.5 GB (shape B) in float32


def peaks():
    """Roofline denominators: MEASURED_PEAKS.json (driver-written: HBM, bf16) + profiles/r02_hw_probes.json (this repo's
    measurement of the INT8 tensor peak with the same protocol: torch._int_mm 8192^3 burst / 4 s sustained)."""
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}
    try:
        p.update(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))))
        p["_source"] = "measured"
    except Exception:
        pass
    try:
        hp = json.load(open(os.path.join(ROOT, "profiles", "r02_hw_probes.json")))
        p["int8_tops_burst"] = max(hp.get("int8_tops_burst_cublaslt", 0.0), hp.get("int8_tops_burst_tdb200_rowwise", 0.0))
        p["int8_tops_sustained"] = max(hp.get("int8_tops_sustained_cublaslt", 0.0), hp.get("int8_tops_sustained_tdb200_rowwise", 0.0))
        p["_int8_source"] = "profiles/r02_hw_probes.json (torch._int_mm / tdb200 rowwise 8192^3; best of the two)"
    except Exception:
        p["int8_tops_burst"] = 2.0 * p["bf16_tflops"]
        p["int8_tops_sustained"] = 2.0 * p["bf16_tflops_sustained"]
        p["_int8_source"] = "2 x bf16 (no INT8 measurement file found)"
    return p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  The sampler process is started before the warm-up
    steps (nvidia-smi needs a few hundred ms to come up on an 8-GPU box, longer than a short timed region); every row is stamped
    on arrival and summary() uses the rows that arrived between mark_start() and mark_end(), or - if the timed region was too
    short to catch one - the rows since the sampler started (GPU under the same load: warm-up + timed), and says which."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def __exit__(self, *a):
        if self.t1 is None:
            self.t1 = time.time()
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass

    def summary(self):
        def ok(r):
            return r and r[0].replace(".", "").isdigit()
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = self.t1 if self.t1 is not None else time.time()
        rows, window = [r for t, r in self.rows if t0 <= t <= t1 + 0.05 and ok(r)], "timed region"
        if not rows:
            rows, window = [r for _, r in self.rows if ok(r)], "warm-up + timed region (timed region shorter than one sample period)"
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(float(r[0])) for r in rows)
        reasons = []
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in rows):
                reasons.append(name)
        mx = max(int(float(r[1])) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit())
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm), "window": window}


class KernelTimer:
    """CUDA-event timing of every launch of one kernel family inside the timed region (same stream as the launch)."""

    def __init__(self):
        self.records = []

    @contextlib.contextmanager
    def __call__(self, *work):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        yield
        e.record()
        self.records.append((s, e, work))

    def result(self, flops_of):
        ms = sum(s.elapsed_time(e) for s, e, _ in self.records)
        fl = sum(flops_of(*w) for _, _, w in self.records)
        return len(self.records), ms, fl


# ------------------------------------------------------------------------------------------------ CPU reference arm
def cpu_sdpa_once(shape, g=None):
    """One call of the reference's CPU-runnable attention (BASELINE.md 3): F.scaled_dot_product_attention on
    q,k,v ~ N(0,1) bf16 [1, H, L, D] (torch.manual_seed(0)), all host threads.  Returns seconds."""
    import torch.nn.functional as F
    heads, d, L = shape["heads"], shape["dim"] // shape["heads"], shape["L"]
    if "_qkv" not in shape:
        gen = torch.Generator().manual_seed(0)
        shape["_qkv"] = tuple(torch.randn(1, heads, L, d, generator=gen).bfloat16() for _ in range(3))
    q, k, v = shape["_qkv"]
    t0 = time.perf_counter()
    F.scaled_dot_product_attention(q, k, v)
    return time.perf_counter() - t0


def cpu_baseline(shape, runs=3):
    torch.set_num_threads(os.cpu_count())
    cpu_sdpa_once(shape)  # warm-up
    ts = sorted(cpu_sdpa_once(shape) for _ in range(runs))
    t = ts[len(ts) // 2]
    heads, d, L, layers = shape["heads"], shape["dim"] // shape["heads"], shape["L"], shape["layers"]
    flop = 4.0 * heads * L * L * d
    return {"value": FRAMES / (DENOISE_STEPS * layers * t), "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
            "seconds_per_call": t, "gflops": flop / t / 1e9,
            "sample": f"torch SDPA [1,{heads},{L},{d}] bf16 dense attention of ONE block (4HL^2D = {flop:.3g} FLOP), 1 warm-up + "
                      f"{runs} runs (median), x{layers} blocks; the block's linears are not included (BASELINE.md 3 protocol)"}


def run_reference(args, shape, rank, world):
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count())
    for _ in range(max(1, args.warmup)):
        cpu_sdpa_once(shape)
    ts = [cpu_sdpa_once(shape) for _ in range(args.steps)]
    t = sum(ts) / len(ts)
    layers, heads, d, L = shape["layers"], shape["heads"], shape["dim"] // shape["heads"], shape["L"]
    val = FRAMES / (DENOISE_STEPS * layers * t)
    sample = (f"each timed step = ONE block's dense self-attention (torch SDPA [1,{heads},{L},{d}] bf16, the reference's CPU-runnable "
              f"path, BASELINE.md 3); value = 81 frames / (4 steps x {layers} blocks x that time); linears excluded")
    line = {"impl": "reference", "metric": "frames_per_sec_4step_81f", "value": val, "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": max(1, args.warmup), "ms_per_step": t * 1e3, "ms_per_step_scaled_to_full_step": layers * t * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{shape['name']} DiT denoise step, reference CPU path: dense SDPA attention of one block per "
                                   f"timed step, scaled x{layers} blocks", "L": L, "dim": shape["dim"], "heads": heads,
                       "head_dim": d, "layers": layers},
            "cpu_baseline": {"value": val, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ B200 arm
def ncu_traffic(shape_key, world):
    """dram bytes of ONE ffn-down GEMM launch from the committed `ncu --set full` summary of this round (single GPU only:
    the sharded GEMM at N > 1 has a different M and was not captured)."""
    if world != 1 or shape_key != "A":
        return {"traffic": None}
    for fn in ("r02_ncu_gemm.txt", "r01_ncu_gemm_final.txt"):
        path = os.path.join(ROOT, "profiles", fn)
        try:
            tot = 0.0
            for ln in open(path):
                for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    if ln.strip().startswith(key + " ="):
                        val, unit = ln.split("=")[1].split()[:2]
                        tot += float(val) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[unit]
            if tot:
                return {"traffic": tot, "traffic_algorithmic": 407.9e6,
                        "traffic_source": f"profiles/{fn} (ffn-down GEMM 32760x1536x8960, one launch)"}
        except OSError:
            continue
    return {"traffic": None}


def output_sample(y, L, row0, world):
    """The rows of the step output [L, dim] that --dump-outputs writes, as float32 on the host: a fixed sample (randperm of
    torch.Generator().manual_seed(0)) of at most DUMP_BYTES, in ascending row order.  Under sequence parallelism every rank
    contributes the sampled rows of its shard [row0, row0 + local rows) and every rank returns the whole sample."""
    import torch.distributed as dist
    n = min(L, DUMP_BYTES // (4 * y.shape[1]))
    rows = torch.randperm(L, generator=torch.Generator().manual_seed(0))[:n].sort().values
    mine = rows[(rows >= row0) & (rows < row0 + y.shape[0])] - row0
    part = y[mine.to(y.device)].float().cpu()
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, part)   # shards are contiguous and in rank order
        part = torch.cat(parts)
    return part


def run_b200(shape_key, shape, args, dev, rank, world, local_rank, steps, warmup, want_e2e, sp_mode_req, dump=False):
    """Build the block stack of `shape`, time `steps` denoise steps (eager pass with per-kernel events, then CUDA-graph
    replay), optionally the end-to-end variant with host buffers.  Returns a dict of measurements; with `dump`, also
    res["dump"]: output_sample() of what the timed path computed in its last step."""
    import torch.distributed as dist
    from turbodiffusion_b200 import _lib
    from turbodiffusion_b200 import turbo_diffusion_ops as tdo
    from turbodiffusion_b200.SLA import core as sla_core
    from turbodiffusion_b200.block import WanHotPath
    from turbodiffusion_b200.ops import wan_rope_angles

    L, dim, heads, ffn, layers, text = (shape[k] for k in ("L", "dim", "heads", "ffn", "layers", "text"))
    d = dim // heads
    model = WanHotPath(dim, ffn, heads, layers, dev, topk=args.topk, seed=1234)
    sp_mode = "single"
    if world > 1:
        from turbodiffusion_b200.dist import SequenceParallel
        sp = SequenceParallel(L, world, rank)
        sp_mode = sp.install(model, sp_mode_req)
        rows, row0 = sp.local_rows, sp.row_begin
    else:
        rows, row0 = L, 0

    g = torch.Generator().manual_seed(7)
    x_host = torch.randn(L, dim, generator=g).bfloat16()[row0:row0 + rows].contiguous().pin_memory()
    e0_host = (torch.randn(6, dim, generator=g) * 0.1).pin_memory()
    ctx_host = torch.randn(text, dim, generator=g).bfloat16().pin_memory()
    angles = wan_rope_angles(*shape["thw"], d)[row0:row0 + rows].contiguous().to(dev)
    out_host = torch.empty(rows, dim, dtype=torch.bfloat16).pin_memory()
    x, e0, ctx = x_host.to(dev), e0_host.to(dev), ctx_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # (1) eager pass: every kernel launched from Python through the C ABI; GEMM and attention launches bracketed by events
    for _ in range(warmup):
        model.step(x, e0, angles, ctx)
    barrier()
    gt, at = KernelTimer(), KernelTimer()
    tdo.GEMM_TIMER, sla_core.ATTN_TIMER = gt, at
    launches0 = _lib.LAUNCHES
    with ClockSampler(local_rank) as clk:
        barrier()
        clk.mark_start()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            y = model.step(x, e0, angles, ctx)
        e.record()
        barrier()
        clk.mark_end()
    tdo.GEMM_TIMER, sla_core.ATTN_TIMER = None, None
    launches = _lib.LAUNCHES - launches0
    eager_total = s.elapsed_time(e)
    ms_eager = max_over_ranks(eager_total / steps)
    n_gemm, gemm_ms, gemm_flops = gt.result(lambda m, n, k: 2.0 * m * n * k)
    n_attn, attn_ms, attn_flops = at.result(lambda h_, mblk, topk, dd: float(h_) * mblk * topk * 4 * 128 * 64 * dd)

    # (2) the same step captured once into a CUDA graph (kernels + NCCL collectives) and replayed
    graph, graph_note = None, "disabled"
    xs, es, cs = x.clone(), e0.clone(), ctx.clone()
    ys = None
    if not args.no_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                model.step(xs, es, angles, cs)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                ys = model.step(xs, es, angles, cs)
            graph_note = "cuda graph replay"
        except Exception as ex:  # noqa: BLE001
            graph, graph_note = None, f"capture failed ({type(ex).__name__}), eager timing reported"
    if graph is not None:
        with ClockSampler(local_rank) as clk:      # started before the warm-up replays so that it is streaming by the timed region
            for _ in range(warmup):
                graph.replay()
            barrier()
            clk.mark_start()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(steps):
                graph.replay()
            e.record()
            barrier()
            clk.mark_end()
        ms_step = max_over_ranks(s.elapsed_time(e) / steps)
    else:
        ms_step = ms_eager

    res = {"ms_step": ms_step, "ms_eager": ms_eager, "launches": launches, "graph_note": graph_note, "clocks": clk.summary(),
           "sp_mode": sp_mode, "n_gemm": n_gemm, "gemm_ms": gemm_ms, "gemm_flops": gemm_flops, "gemm_share": gemm_ms / eager_total,
           "n_attn": n_attn, "attn_ms": attn_ms, "attn_flops": attn_flops, "attn_share": attn_ms / eager_total,
           "rows": rows}
    if dump:
        res["dump"] = output_sample(ys if graph is not None else y, L, row0, world)

    # (3) end to end through the public call with HOST buffers (H2D of the inputs + D2H of the result per step)
    if want_e2e:
        def step_host():
            if graph is not None:  # static graph inputs are refilled from pinned host memory, result read back
                xs.copy_(x_host, non_blocking=True)
                es.copy_(e0_host, non_blocking=True)
                cs.copy_(ctx_host, non_blocking=True)
                graph.replay()
                out_host.copy_(ys, non_blocking=True)
                return
            xd = x_host.to(dev, non_blocking=True)
            ed = e0_host.to(dev, non_blocking=True)
            cd = ctx_host.to(dev, non_blocking=True)
            out_host.copy_(model.step(xd, ed, angles, cd), non_blocking=True)

        step_host()
        barrier()
        s2, e2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s2.record()
        for _ in range(steps):
            step_host()
        e2.record()
        barrier()
        res["ms_e2e"] = max_over_ranks(s2.elapsed_time(e2) / steps)
        res["h2d"] = x_host.numel() * 2 + e0_host.numel() * 4 + ctx_host.numel() * 2
        res["d2h"] = out_host.numel() * 2
    graph = None
    del model, xs, es, cs, ys, x, e0, ctx, y
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return res


def rooflines(res, pk, shape_key, world):
    gemm_ach = res["gemm_flops"] / res["gemm_ms"] / 1e9 if res["gemm_ms"] > 0 else 0.0
    attn_ach = res["attn_flops"] / res["attn_ms"] / 1e9 if res["attn_ms"] > 0 else 0.0
    i8 = pk["int8_tops_sustained"]
    # the fused attention kernel does half of its MACs in INT8 (Q.K^T) and half in bf16 (P.V): at equal MAC counts the
    # time-weighted peak is the harmonic mean of the two rates
    mixed = 2.0 / (1.0 / i8 + 1.0 / pk["bf16_tflops_sustained"])
    gemm = {"bound": "tensor", "kernel": "gemm_w8a8_kernel (tcgen05 kind::i8, per-128-K dequant)", "achieved": gemm_ach, "peak": i8,
            "unit": "TFLOP/s", "frac": gemm_ach / i8 if i8 else None,
            "frac_of_bf16_sustained_peak": gemm_ach / pk["bf16_tflops_sustained"],
            "peak_source": f"INT8 sustained, {pk['_int8_source']}; bf16 from MEASURED_PEAKS.json ({pk['_source']})",
            "launches": res["n_gemm"], "share_of_step": res["gemm_share"], **ncu_traffic(shape_key, world),
            "timed_in": "eager pass of the same K steps (CUDA events around each GEMM launch on the launch stream)"}
    attn = {"bound": "tensor", "kernel": "sla_attn kernel (tcgen05 kind::i8 Q.K^T + kind::f16 P.V, fused softmax/linear branch)",
            "achieved": attn_ach, "peak": mixed, "unit": "TFLOP/s", "frac": attn_ach / mixed if mixed else None,
            "flops_split": {"int8_qk": 0.5, "bf16_pv": 0.5},
            "peak_source": "harmonic mean of the measured INT8 and bf16 sustained peaks (equal MAC counts in each)",
            "launches": res["n_attn"], "share_of_step": res["attn_share"], "traffic": None,
            "timed_in": "eager pass (CUDA events around each fused-attention launch); FLOPs = H*Mblk*topk*4*128*64*D"}
    return gemm, attn


def extra_kernels(dev, args):
    """BASELINE.json configs 2 and 5 as short kernel timings: SageSLA at the literal [1,24,32760,64] shape, and the LTX-2
    shape C (28672 tokens, 32x128 heads, dim 4096): SageSLA top-k 0.3, per-row W8A8 GEMMs, FastNorm ada kernels."""
    from turbodiffusion_b200 import ltx
    from turbodiffusion_b200.SLA import SageSparseLinearAttention
    pk = peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timeit(fn, iters=5, warmup=3):
        for _ in range(warmup):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        ts.sort()
        return ts[len(ts) // 2]

    out = {}
    g = torch.Generator(device=dev).manual_seed(3)
    for tag, (L, H, D, ratio) in {"sage_sla_24x64": (32760, 24, 64, 0.1), "ltx_C_sage_sla_32x128": (28672, 32, 128, 0.3)}.items():
        q = torch.randn(1, L, H, D, device=dev, generator=g).bfloat16()
        k = (torch.randn(1, L, H, D, device=dev, generator=g) + 2 * torch.randn(1, 1, H, D, device=dev, generator=g)).bfloat16()
        v = torch.randn(1, L, H, D, device=dev, generator=g).bfloat16()
        mod = SageSparseLinearAttention(D, ratio).to(dev)
        with torch.no_grad():
            mod.proj_l.weight.normal_(0, 0.05)
        ms = timeit(lambda: mod(q, k, v))
        mblk, nblk = (L + 127) // 128, (L + 63) // 64
        fl = float(H) * mblk * int(ratio * nblk) * 4 * 128 * 64 * D
        out[tag] = {"workload": f"SageSparseLinearAttention.forward q,k,v [1,{L},{H},{D}] bf16 top-k {ratio} (module: prep + block map "
                                f"+ moments + fused attention)", "ms": ms, "tflops_sparse_attention": fl / ms / 1e9, "l2": "flushed"}
        del q, k, v, mod
    m = 28672
    for name, n, kk in (("ltx_C_gemm_proj_4096x4096", 4096, 4096), ("ltx_C_gemm_ffn_up_16384x4096", 16384, 4096),
                        ("ltx_C_gemm_ffn_down_4096x16384", 4096, 16384)):
        a = torch.randint(-128, 128, (m, kk), device=dev, dtype=torch.int8)
        b = torch.randint(-128, 128, (n, kk), device=dev, dtype=torch.int8)
        a_s, b_s = torch.rand(m, device=dev) * 0.01, torch.rand(n, device=dev) * 0.01
        bias = torch.randn(n, device=dev).bfloat16()
        ms = timeit(lambda: ltx.gemm_int8_post_scale_bias(a, a_s, b, b_s, bias))
        tf = 2.0 * m * n * kk / ms / 1e9
        out[name] = {"workload": f"per-row post-scale W8A8 GEMM {m}x{n}x{kk} (tilelang_w8a8.py:78-117 semantics)", "ms": ms,
                     "tflops": tf, "frac_int8_peak": tf / pk["int8_tops_sustained"], "l2": "flushed"}
        del a, b
    return out


def _leave(exit_group):
    """End of a multi-rank run: every rank has finished its GPU work and rank 0 has printed the line.  Leave without tearing the
    NCCL communicators down (destroy_process_group() can block after graph-captured collectives): drain the GPU, meet the other
    ranks over the gloo group so that no process unmaps peer buffers a neighbour's last collective still reads, then _exit.  A
    watchdog bounds the whole path: once the results are out, a rank that cannot rendezvous within 60 s leaves anyway."""
    import threading
    import torch
    import torch.distributed as dist
    sys.stdout.flush()
    threading.Timer(60.0, lambda: os._exit(0)).start()
    try:
        torch.cuda.synchronize()
        dist.barrier(group=exit_group) if exit_group is not None else dist.barrier()
    except Exception:  # noqa: BLE001
        pass
    sys.stdout.flush()
    os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shape", default="A", choices=list(SHAPES))
    ap.add_argument("--layers", type=int, default=None, help="override the number of blocks (diagnostics only)")
    ap.add_argument("--topk", type=float, default=0.1)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sp-mode", default="auto", choices=["auto", "allgather", "ulysses"],
                    help="N>1 attention exchange: K/V all-gather + moment all-reduce, or head<->sequence all-to-all "
                         "(needs heads %% N == 0); auto = the mode that measured faster (dist.py pick_mode)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra_configs runs (shape B, 24x64, LTX shape C)")
    ap.add_argument("--profile", action="store_true", help="device-resident region only (for runs under ncu)")
    ap.add_argument("--no-graph", action="store_true", help="time the eager (Python-launched) step instead of the CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output of the last timed step as DIR/step_output.npy (float32, a "
                         "fixed sample of its rows, see output_sample) so that two builds can be compared on identical inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the output of the b200 step; --impl reference times a CPU attention call with nothing to compare")
    if args.profile:
        args.no_graph = True
        args.no_extras = True
    args.warmup = max(3, args.warmup) if args.impl == "b200" and not args.profile else args.warmup
    shape = dict(SHAPES[args.shape])
    if args.layers:
        shape["layers"] = args.layers

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return run_reference(args, shape, rank, world)

    import torch.distributed as dist
    from turbodiffusion_b200 import _lib
    _lib.lib()  # fail loudly when the CUDA library is missing
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    exit_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        # host-side rendezvous for the very end of the run (see _leave): the NCCL communicators are captured into CUDA graphs and
        # a last NCCL collective or their teardown has been seen to block, so the ranks meet over gloo instead
        try:
            os.environ.setdefault("GLOO_SOCKET_IFNAME", "lo")   # one node: no hostname lookup (the box's name may not resolve)
            exit_group = dist.new_group(backend="gloo", timeout=datetime.timedelta(seconds=120))
        except Exception as ex:  # noqa: BLE001  -- fall back to the NCCL barrier at exit (still under _leave's watchdog)
            print(f"[bench] gloo exit group unavailable ({type(ex).__name__}: {ex}); using the NCCL barrier", file=sys.stderr)
            exit_group = None

    res = run_b200(args.shape, shape, args, dev, rank, world, local_rank, args.steps, args.warmup, not args.profile, args.sp_mode,
                   dump=args.dump_outputs is not None)
    if args.dump_outputs is not None and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "step_output.npy"), res.pop("dump").numpy())
    if args.profile:
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step": res["ms_step"], "gpu_launches": res["launches"]}), flush=True)
        if world > 1:
            _leave(exit_group)
        return

    extras = {}
    if not args.no_extras:
        # BASELINE.json configs 3/4: the Wan-14B 720p block stack at this N (2 timed steps after 3 warm-ups)
        other = "B" if args.shape == "A" else "A"
        try:
            sh = dict(SHAPES[other])
            r2 = run_b200(other, sh, args, dev, rank, world, local_rank, 2, 3, False, args.sp_mode)
            g2, a2 = rooflines(r2, peaks(), other, world)
            extras[f"shape_{other}"] = {
                "workload": f"{sh['name']} DiT denoise step: {sh['layers']} blocks, L={sh['L']}, dim {sh['dim']}, {sh['heads']} heads",
                "n_gpus": world, "parallelism": f"sp{world}-{r2['sp_mode']}" if world > 1 else "single", "steps": 2, "warmup": 3,
                "ms_per_step": r2["ms_step"], "ms_per_step_eager": r2["ms_eager"],
                "frames_per_sec": FRAMES / (DENOISE_STEPS * r2["ms_step"] * 1e-3), "gpu_launches": r2["launches"],
                "gemm_tflops": g2["achieved"], "gemm_frac_int8_peak": g2["frac"], "attn_tflops": a2["achieved"],
                "attn_frac_mixed_peak": a2["frac"], "clocks": r2["clocks"]}
        except Exception as ex:  # noqa: BLE001
            extras[f"shape_{other}"] = {"error": f"{type(ex).__name__}: {ex}"}
        if rank == 0:
            try:
                extras.update(extra_kernels(dev, args))
            except Exception as ex:  # noqa: BLE001
                extras["kernels_error"] = f"{type(ex).__name__}: {ex}"
        if world > 1:
            dist.barrier()

    if rank == 0:
        pk = peaks()
        gemm, attn = rooflines(res, pk, args.shape, world)
        L, dim, heads, ffn, layers, text = (shape[k] for k in ("L", "dim", "heads", "ffn", "layers", "text"))
        ms_step = res["ms_step"]
        line = {
            "metric": "frames_per_sec_4step_81f", "value": FRAMES / (DENOISE_STEPS * ms_step * 1e-3), "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int8 (W8A8 GEMM, QK^T) / bf16 (PV, io) / fp32 (accumulate)",
            "data": "synthetic",
            "config": {"workload": f"{shape['name']} DiT denoise step: {layers} blocks (SageSLA top-k {args.topk} + W8A8 + FastNorm)",
                       "L": L, "dim": dim, "heads": heads, "head_dim": dim // heads, "ffn": ffn, "text_len": text,
                       "parallelism": f"sp{world}-{res['sp_mode']}" if world > 1 else "single",
                       "l2": "activations per block exceed L2 (>=100 MB tensors, 30+ distinct weight sets)"},
            "e2e": {"value": FRAMES / (DENOISE_STEPS * res["ms_e2e"] * 1e-3), "unit": "frames/s", "ms_per_step": res["ms_e2e"],
                    "h2d_bytes_per_step": res["h2d"], "d2h_bytes_per_step": res["d2h"]},
            "gpu_launches": res["launches"],
            "roofline": gemm, "roofline_attention": attn,
            "ms_per_step_eager": res["ms_eager"], "launch_mode": res["graph_note"],
            "clocks": res["clocks"],
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(shape)
        if extras:
            line["extra_configs"] = extras
        print(json.dumps(line), flush=True)
    if world > 1:
        _leave(exit_group)


if __name__ == "__main__":
    main()
