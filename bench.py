#!/usr/bin/env python
"""bench.py - Llama-3-8B W4A16 decode (default) / prefill throughput of the AWQ linear path on B200.

A "step" is one pass of the hot path over one batch of synthetic input: every quantised linear of
Llama-3-8B (32 layers x [qkv 4096->6144, o 4096->4096, gate|up 4096->28672, down 14336->4096], GEMM
layout, group 128, random-init AWQ-packed weights, 3.63 GB per replica >> the 126 MB L2, so every step
streams the weights from HBM) plus the RMSNorm / SiLU*mul glue kernels that keep the activations O(1).
Attention, KV cache, embeddings and lm_head are not on the path (BASELINE.json north_star:
"awq/modules/fused/* sits unchanged on top", "synthetic Llama-shape activations").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--mode decode|prefill] [--impl reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  value = whole-job tokens/s with inputs resident in HBM (CUDA-graph
replay of the plugin calls); e2e = the same step driven from pinned HOST buffers through the
awq_ext-facing operator calls (H2D of the token's hidden state and D2H of the result inside the timed
region); roofline = the GEMV (decode) or tcgen05 GEMM (prefill) kernels alone against MEASURED_PEAKS.json;
cpu_baseline / --impl reference = the reference's CPU path (dequantize_gemm + torch.matmul,
awq/modules/linear/gemm.py:71-77) restated in oracle/ref_cpu_path.py, timed on the host cores on a
bounded sample (whole layers), extrapolated to the 32-layer step.
N > 1: Llama-3-8B fits one GPU, so ranks are independent replicas (no data-path collective, weak
scaling); the tensor-parallel column/row sharding for models that exceed one GPU is autoawq_b200/shard.py.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HIDDEN, INTER, LAYERS, QKV_N, GROUP = 4096, 14336, 32, 6144, 128
LINEARS = [("qkv", HIDDEN, QKV_N), ("o", HIDDEN, HIDDEN), ("gate_up", HIDDEN, 2 * INTER), ("down", INTER, HIDDEN)]


def linear_bytes(K, N, M, G=GROUP):
    """Algorithmic bytes of one W4A16 linear (SURVEY.md 8d): packed weights + scales + zeros + x + y."""
    return K * N // 2 + (K // G) * N * 2 + (K // G) * N // 2 + 2 * M * K + 2 * M * N


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.nv_rows, self.nv_stop, self.nv_thread, self.nv_max = None, [], False, None, None

    # NVML (pynvml / nvidia-ml-py) polled every ~2 ms from a thread: a decode run's timed region is ~40 ms, shorter than
    # nvidia-smi's first sample (its -lms loop delivered 0-2 rows there); nvidia-smi stays as the fallback.
    def _nvml_start(self):
        import pynvml as nv

        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        idx = self.index
        if vis and all(t.strip().isdigit() for t in vis.split(",")):
            idx = int(vis.split(",")[self.index])
        h = nv.nvmlDeviceGetHandleByIndex(idx)
        self.nv_max = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

        def loop():
            while not self.nv_stop:
                try:
                    mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    r = int(get_reasons(h))
                    self.nv_rows.append((time.time(), mhz, [n for n, b in bits.items() if r & b]))
                except Exception:  # noqa: BLE001
                    pass
                time.sleep(0.002)

        self.nvml = nv
        self.nv_thread = threading.Thread(target=loop, daemon=True)
        self.nv_thread.start()

    def start(self):
        try:
            self._nvml_start()
            return
        except Exception:  # noqa: BLE001
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def count(self, t0, t1):
        """NVML samples taken inside [t0, t1] so far (the sampler keeps running)."""
        return sum(1 for ts, _, _ in list(self.nv_rows) if t0 <= ts <= t1) if self.nvml is not None else -1

    def stop(self, t0, t1, t_ext=None):
        """Clocks over the timed region [t0, t1]; t_ext > t1: the region was followed by untimed replays of the SAME step
        until t_ext because too few samples fell inside it (reported separately, never mixed silently)."""
        if self.nvml is not None:
            self.nv_stop = True
            self.nv_thread.join(timeout=1.0)
            hi = t_ext if t_ext is not None else t1
            sm_in = [m for ts, m, _ in self.nv_rows if t0 <= ts <= t1]
            sm = sorted(m for ts, m, _ in self.nv_rows if t0 <= ts <= hi)
            reasons = sorted({n for ts, _, rs in self.nv_rows if t0 <= ts <= hi for n in rs})
            out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.nv_max, "reasons": reasons,
                   "samples": len(sm), "samples_in_timed_region": len(sm_in), "source": "nvml, 2 ms period"}
            if t_ext is not None:
                out["note"] = ("fewer than 3 samples fell inside the timed region: the same step kept replaying (untimed) for "
                               f"{(t_ext - t1) * 1e3:.0f} ms more and those samples are included")
            return out
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                mx = float(f[1])
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(f[0]))
                    for nm, v in zip(names, f[3:7]):
                        if v.lower().startswith("active"):
                            reasons.add(nm)
            except ValueError:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------- GPU arm
class Replica:
    """Random-init AWQ-packed Llama-3-8B linears on one GPU + the step that chains them."""

    def __init__(self, dev, M, layers=LAYERS, seed=0):
        import torch

        from autoawq_b200 import ext

        self.torch, self.ext, self.dev, self.M, self.layers = torch, ext, dev, M, layers
        g = torch.Generator(device=dev).manual_seed(seed)
        self.w = []
        for _ in range(layers):
            lw = {}
            for name, K, N in LINEARS:
                qw = torch.randint(-2**31, 2**31 - 1, (K, N // 8), dtype=torch.int32, device=dev, generator=g)
                qz = torch.randint(-2**31, 2**31 - 1, (K // GROUP, N // 8), dtype=torch.int32, device=dev, generator=g)
                # (q - z) has std ~6.1: keep std(W) * sqrt(K) ~ 1 so activations stay O(1) down the chain
                s = (torch.rand((K // GROUP, N), device=dev, generator=g) * 0.5 + 0.75) / (6.1 * K**0.5)
                lw[name] = (qw, s.half(), qz)
            self.w.append(lw)
        self.norm_w = torch.ones(HIDDEN, dtype=torch.float16, device=dev)
        self.xn = torch.empty((M, HIDDEN), dtype=torch.float16, device=dev)
        self.act = torch.empty((M, INTER), dtype=torch.float16, device=dev)
        self.h = torch.randn((M, HIDDEN), generator=g, device=dev, dtype=torch.float16)
        self.out = torch.empty((M, HIDDEN), dtype=torch.float16, device=dev)
        self.launches_per_step = layers * 7

    def lin(self, x, w, api=None):
        # the awq_ext-facing operator (awq_ext.gemm_forward_cuda semantics; autoawq_b200/ext.py)
        return (api or self.ext).gemm_forward_cuda(x, w[0], w[1], w[2], 8)

    def step(self, h, api=None):
        """The operator-call sequence of one step.  `api` = the awq_ext surface (default) or a DecodeProgram
        recorder with the same call names (autoawq_b200/program.py)."""
        e = api or self.ext
        for lw in self.w:
            e.layernorm_forward_cuda(h, self.norm_w, self.xn, 1e-5)
            qkv = self.lin(self.xn, lw["qkv"], e)
            o = self.lin(qkv[:, :HIDDEN], lw["o"], e)
            e.layernorm_forward_cuda(o, self.norm_w, self.xn, 1e-5)
            gu = self.lin(self.xn, lw["gate_up"], e)
            e.silu_and_mul(self.act, gu)
            h = self.lin(self.act, lw["down"], e)
        return h

    def gemm_only(self, h):
        """The quantised linears alone (roofline leg): same weights, fixed inputs, no glue kernels."""
        for lw in self.w:
            self.lin(self.xn, lw["qkv"])
            self.lin(self.xn, lw["o"])
            self.lin(self.xn, lw["gate_up"])
            self.lin(self.act, lw["down"])


def capture(torch, fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        res = fn()
    return g, res


def timed(torch, fn, steps, warmup, dist=None):
    """W untimed + K timed calls of fn, CUDA events on the launching stream, barrier + sync both sides,
    max over ranks.  Returns seconds for the K steps."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    sec = e0.elapsed_time(e1) / 1e3
    if dist is not None:
        t = torch.tensor([sec], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    return sec


def pick_cpu_threads(M):
    """The reference runs torch with its default thread count (= all cores), which on a many-core host is slower
    than a moderate count for these bandwidth-bound elementwise + GEMV ops.  Give the CPU arm its best case:
    try a few counts once and keep the fastest."""
    cores = os.cpu_count() or 1
    best = None
    for th in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        t, _ = cpu_reference_sample(M, 1, 1, threads=th)
        if best is None or t < best[0]:
            best = (t, th)
    return best[1]


def cpu_reference_sample(M, layers_sample, reps, threads=None):
    """Reference CPU path on a bounded sample: `layers_sample` whole layers of the step, fp16,
    all host threads.  Returns (seconds per sampled layer, cores)."""
    import torch

    from oracle import ref_cpu_path as R

    cores = threads or os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(0)
    ws = []
    for name, K, N in LINEARS:
        qw = torch.randint(-2**31, 2**31 - 1, (K, N // 8), dtype=torch.int32, generator=g)
        qz = torch.randint(-2**31, 2**31 - 1, (K // GROUP, N // 8), dtype=torch.int32, generator=g)
        s = ((torch.rand((K // GROUP, N), generator=g) * 0.5 + 0.75) / (6.1 * K**0.5)).half()
        ws.append((K, N, qw, qz, s))
    xs = {K: torch.randn((M, K), generator=g, dtype=torch.float16) for K in (HIDDEN, INTER)}
    ts = []
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            for _l in range(layers_sample):
                for K, N, qw, qz, s in ws:
                    R.wqlinear_forward(xs[K], qw, qz, s, GROUP)
            ts.append((time.perf_counter() - t0) / layers_sample)
    return min(ts), cores


def dump_outputs(directory, y, max_elems=4096 * 1024):
    """The output of the last timed step, [M, 4096], as DIR/output.npy in float32.  The inputs and weights come from
    seeded generators, so two builds run with the same arguments can be compared file for file.  A prefill output
    (M = 4096) is larger than 64 MB in float32: then a fixed, seeded sample of rows is written, with their indices in
    DIR/output_rows.npy."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    y = y.float().cpu().numpy().reshape(-1, y.shape[-1])
    rows = np.arange(y.shape[0])
    if y.size > max_elems:
        rows = np.sort(np.random.default_rng(0).choice(y.shape[0], max_elems // y.shape[1], replace=False))
    np.save(os.path.join(directory, "output.npy"), np.ascontiguousarray(y[rows]))
    np.save(os.path.join(directory, "output_rows.npy"), rows.astype(np.float64))


def gemv_4096_leg(torch, ext, dev, steps, peaks):
    """The metric's own shape: ONE 4096 x 4096 g128 GEMV (M = 1), stand-alone launches rotating over a pool of
    distinct weights larger than L2 (48 x 8.7 MB = 419 MB), CUDA graph of the pool, CUDA events."""
    K = N = HIDDEN
    pool = 48
    g = torch.Generator(device=dev).manual_seed(123)
    ws = []
    for _ in range(pool):
        qw = torch.randint(-2**31, 2**31 - 1, (K, N // 8), dtype=torch.int32, device=dev, generator=g)
        qz = torch.randint(-2**31, 2**31 - 1, (K // GROUP, N // 8), dtype=torch.int32, device=dev, generator=g)
        s = ((torch.rand((K // GROUP, N), device=dev, generator=g) * 0.5 + 0.75) / (6.1 * K**0.5)).half()
        ws.append((qw, s, qz))
    x = torch.randn((1, K), device=dev, dtype=torch.float16, generator=g)

    def sweep():
        for w in ws:
            ext.gemm_forward_cuda(x, w[0], w[1], w[2], 8)

    gr, _ = capture(torch, sweep)
    n = max(5, steps)
    sec = timed(torch, gr.replay, n, 3)
    us = sec / n / pool * 1e6
    b = linear_bytes(K, N, 1)
    return {"shape": "4096x4096 g128 M=1", "us_per_launch": round(us, 3), "gbs": round(b / us / 1e3, 1),
            "frac": round(b / us / 1e3 / peaks["hbm_gbs"], 4), "alg_bytes": b,
            "pool": f"{pool} distinct weight sets ({pool * b / 1e6:.0f} MB > L2), one CUDA graph of {pool} launches"}


def small_batch_leg(torch, ext, dev, steps, peaks):
    """Batched decode (BASELINE config 3's small-M end, VERDICT r1 item 4): one linear at M = 8 / 16 / 64 tokens on
    4096 x 4096 and 4096 x 28672 (gate|up), stand-alone launches rotating over > L2 of distinct weights, CUDA graph, CUDA
    events.  HBM-bound up to M ~ 73: the figure of merit is the fraction of the HBM peak."""
    out = {}
    g = torch.Generator(device=dev).manual_seed(321)
    for (K, N) in ((HIDDEN, HIDDEN), (HIDDEN, 2 * INTER)):
        wb = K * N // 2
        pool = max(3, int(400e6 // wb) + 1)
        ws = []
        for _ in range(pool):
            qw = torch.randint(-2**31, 2**31 - 1, (K, N // 8), dtype=torch.int32, device=dev, generator=g)
            qz = torch.randint(-2**31, 2**31 - 1, (K // GROUP, N // 8), dtype=torch.int32, device=dev, generator=g)
            s = ((torch.rand((K // GROUP, N), device=dev, generator=g) * 0.5 + 0.75) / (6.1 * K**0.5)).half()
            ws.append((qw, s, qz))
        for M in (8, 16, 64):
            x = torch.randn((M, K), device=dev, dtype=torch.float16, generator=g)

            def sweep():
                for w in ws:
                    ext.gemm_forward_cuda(x, w[0], w[1], w[2], 8)

            gr, _ = capture(torch, sweep)
            n = max(5, steps)
            sec = timed(torch, gr.replay, n, 3)
            us = sec / n / pool * 1e6
            bts = linear_bytes(K, N, M)
            out[f"{K}x{N} M={M}"] = {"us": round(us, 2), "gbs": round(bts / us / 1e3, 1),
                                     "frac_hbm": round(bts / us / 1e3 / peaks["hbm_gbs"], 4),
                                     "tflops": round(2.0 * M * K * N / us / 1e6, 1)}
        del ws
    out["kernel"] = "gemm_tcq_kernel (tcgen05, TMA-staged packed weights), 5 <= M <= 128"
    return out


def prefill_leg(torch, rep_weights, dev, steps, peaks):
    """BASELINE config 3 as a secondary leg of the default run: bs=1, seq=4096 through every quantised linear
    (tcgen05 kernel), same weights; tok/s, TFLOP/s, fraction of the sustained bf16 peak."""
    M = 4096
    from autoawq_b200 import ext

    xn = torch.randn((M, HIDDEN), device=dev, dtype=torch.float16) * 0.5
    act = torch.randn((M, INTER), device=dev, dtype=torch.float16) * 0.5
    xk = {HIDDEN: xn, INTER: act}

    def step():
        for lw in rep_weights:
            for name, K, _N in LINEARS:
                w = lw[name]
                ext.gemm_forward_cuda(xk[K], w[0], w[1], w[2], 8)

    gr, _ = capture(torch, step)
    n = max(3, min(steps, 6))
    sec = timed(torch, gr.replay, n, 3)
    flops = sum(2.0 * M * K * N for _, K, N in LINEARS) * len(rep_weights)
    tf = flops / (sec / n) / 1e12
    return {"workload": "Llama-3-8B prefill bs=1 seq=4096, quantised linears (128 launches)", "tok_s": round(M * n / sec, 1),
            "ms_per_step": round(sec / n * 1e3, 3), "tflops": round(tf, 1),
            "frac_of_sustained_bf16_peak": round(tf / peaks["bf16_tflops_sustained"], 4),
            "frac_of_burst_bf16_peak": round(tf / peaks["bf16_tflops"], 4), "kernel": "gemm_tc_kernel (tcgen05)"}


# ------------------------------------------------------------- tensor-parallel leg (BASELINE config 5), N > 1 only
L70 = {"hidden": 8192, "inter": 28672, "layers": 80, "heads": 64, "kv_heads": 8, "head_dim": 128}


def tp70b_leg(torch, dist, rank, world, dev, steps, layers=None):
    """Llama-3-70B-shaped decode step (bs = 1), tensor-parallel over the `world` GPUs of the box through
    autoawq_b200/shard.py: fused q|k|v split by head group and gate|up split by column (no collective), o / down split
    by row, ONE NCCL all-reduce of the fp16 [1, 8192] partial output after each of them (SURVEY 8e) - 160 all-reduces
    of 16 KB per token, captured with the kernels in one CUDA graph.  Every rank builds the same full packed tensors
    layer by layer (same seed), keeps its shard and drops the rest.  Attention / KV cache are not on the path: the
    rank's q columns stand in for its attention output, as in the single-GPU step."""
    from autoawq_b200 import ext, shard as S

    c = dict(L70)
    if layers:
        c["layers"] = layers
    H, I, G = c["hidden"], c["inter"], GROUP
    qkv_n = (c["heads"] + 2 * c["kv_heads"]) * c["head_dim"]
    if c["kv_heads"] % world or c["heads"] % world:
        return {"unavailable": f"heads do not divide by {world}"}

    def packed(K, N, gen):
        qw = torch.randint(-2**31, 2**31 - 1, (K, N // 8), dtype=torch.int32, device=dev, generator=gen)
        qz = torch.randint(-2**31, 2**31 - 1, (K // G, N // 8), dtype=torch.int32, device=dev, generator=gen)
        sc = ((torch.rand((K // G, N), device=dev, generator=gen) * 0.5 + 0.75) / (6.1 * K**0.5)).half()
        return S.PackedGemm(qw, qz, sc)

    ws, alg = [], 0
    for l in range(c["layers"]):
        gen = torch.Generator(device=dev).manual_seed(1000 + l)       # same full tensors on every rank
        qkv = S.shard_qkv(packed(H, qkv_n, gen), c["heads"], c["kv_heads"], c["head_dim"], rank, world)
        o = S.shard_rows(packed(H, H, gen), rank, world)
        mlp = S.TensorParallelMLP(packed(H, I, gen), packed(H, I, gen), packed(I, H, gen), rank, world)
        ws.append((qkv, o, mlp.gu, mlp.down))
        if l == 0:
            alg = sum(linear_bytes(p.in_features, p.out_features, 1) for p in ws[0])
    torch.cuda.empty_cache()
    q_local = c["heads"] // world * c["head_dim"]
    nw = torch.ones(H, dtype=torch.float16, device=dev)
    h0 = torch.randn((1, H), device=dev, dtype=torch.float16, generator=torch.Generator(device=dev).manual_seed(7))
    xn = torch.empty((1, H), dtype=torch.float16, device=dev)
    act = torch.empty((1, ws[0][3].in_features), dtype=torch.float16, device=dev)

    def lin(x, p):
        return ext.linear_forward("gemm", x, p.qweight, p.scales, p.qzeros, G)

    from autoawq_b200.comm import OneShotAllReduce

    oneshot = OneShotAllReduce(max_elems=H)          # symmetric buffers + IPC handle exchange, once

    def step(collective="nccl"):
        ar = {"nccl": dist.all_reduce, "oneshot": oneshot, "none": lambda t: t}[collective]
        h = h0
        for qkv, o, gu, down in ws:
            ext.layernorm_forward_cuda(h, nw, xn, 1e-5)
            a = lin(xn, qkv)[:, :q_local]
            y = lin(a, o)
            ar(y)
            ext.layernorm_forward_cuda(y, nw, xn, 1e-5)
            g = lin(xn, gu)
            ext.silu_and_mul(act, g)
            h = lin(act, down)
            ar(h)
        return h

    # the same step with every collective-free segment as ONE persistent kernel (decode program, DESIGN 3.5): per layer
    # [RMSNorm -> qkv -> o] | all-reduce | [RMSNorm -> gate|up -> SiLU*mul -> down] | all-reduce = 4 launches, not 10
    from autoawq_b200.program import DecodeProgram

    progs, prog_err = [], None
    try:
        h_in = h0
        for qkv, o, gu, down in ws:
            pa = DecodeProgram()
            pa.layernorm_forward_cuda(h_in, nw, xn, 1e-5)
            q = pa.gemm_forward_cuda(xn, qkv.qweight, qkv.scales, qkv.qzeros, 8)
            y = pa.gemm_forward_cuda(q[:, :q_local], o.qweight, o.scales, o.qzeros, 8)
            pa.build()
            pb = DecodeProgram()
            pb.layernorm_forward_cuda(y, nw, xn, 1e-5)
            g = pb.gemm_forward_cuda(xn, gu.qweight, gu.scales, gu.qzeros, 8)
            pb.silu_and_mul(act, g)
            d = pb.gemm_forward_cuda(act, down.qweight, down.scales, down.qzeros, 8)
            pb.build()
            progs.append((pa, y, pb, d))
            h_in = d
        if not all(pa.fused and pb.fused for pa, _, pb, _ in progs):
            prog_err = "a segment did not fit the fused kernels"
    except Exception as ex:  # noqa: BLE001
        prog_err = f"{type(ex).__name__}: {str(ex)[:160]}"

    def step_programs():
        for pa, y, pb, d in progs:
            pa.run()
            oneshot(y)
            pb.run()
            oneshot(d)
        return progs[-1][3]

    def ar_only(collective="nccl"):
        ar = dist.all_reduce if collective == "nccl" else oneshot
        for _ in range(2 * c["layers"]):
            ar(xn)

    dist.all_reduce(xn)            # communicator warm-up outside any capture
    torch.cuda.synchronize()
    out = {"workload": f"Llama-3-70B W4A16 g128 decode bs=1, tp={world}: {c['layers']} layers x [qkv {H}x{qkv_n // world}, "
                       f"o {H // world}x{H} + all-reduce, gate|up {H}x{2 * I // world}, down {I // world}x{H} + all-reduce]",
           "weights_gb_per_gpu": round(alg * c["layers"] / 1e9, 2)}
    res = {}
    variants = [("step", lambda: step("oneshot")), ("step_nccl", lambda: step("nccl")),
                ("no_collective", lambda: step("none")), ("allreduce_only", lambda: ar_only("oneshot")),
                ("allreduce_only_nccl", lambda: ar_only("nccl"))]
    if prog_err is None:
        variants.append(("step_programs", step_programs))
    for name, fn in variants:
        try:
            g, _ = capture(torch, fn)
            f = g.replay
            graphed = True
        except Exception as ex:  # noqa: BLE001
            torch.cuda.synchronize()
            f, graphed = fn, False
            out.setdefault("notes", []).append(f"{name}: not captured ({type(ex).__name__}), timed eagerly")
        sec = timed(torch, f, steps, 3, dist)
        res[name] = (sec / steps, graphed)
    oneshot.check()
    # both collectives give the same sums up to the fp16 rounding of NCCL's own reduction order
    # (the per-op GEMV adds split-K partials with fp32 atomics: two runs of the SAME step differ in the last bit, and
    # 160 chained random linears amplify that - the nccl-vs-nccl figure is the noise floor of this comparison)
    y1, y2, y3 = step("oneshot").float().clone(), step("nccl").float().clone(), step("nccl").float().clone()
    torch.cuda.synchronize()
    t = res["step"][0]
    out["per_op_launches"] = {"tok_s": round(1.0 / t, 2), "ms_per_step": round(t * 1e3, 4),
                              "launches_per_step": 10 * c["layers"]}
    if "step_programs" in res and res["step_programs"][0] < t:
        t = res["step_programs"][0]
        out["path"] = (f"decode programs: {2 * c['layers']} persistent kernels ({progs[0][0].kind} / {progs[0][2].kind}) + "
                       f"{2 * c['layers']} one-shot all-reduces per token")
    else:
        out["path"] = "per-op launches + one-shot all-reduces"
    if "step_programs" in res:
        out["decode_programs"] = {"tok_s": round(1.0 / res["step_programs"][0], 2),
                                  "ms_per_step": round(res["step_programs"][0] * 1e3, 4), "launches_per_step": 4 * c["layers"]}
    elif prog_err:
        out["decode_programs"] = {"unavailable": prog_err}
    out.update({"tok_s": round(1.0 / t, 2), "ms_per_step": round(t * 1e3, 4), "cuda_graph": res["step"][1],
                "collective": f"one-shot all-reduce over NVLink peer memory (csrc/comm.cu), fp16 [1, {H}] (16 KB) x "
                              f"{2 * c['layers']} per token, one kernel each, inside the CUDA graph",
                "nccl": {"tok_s": round(1.0 / res["step_nccl"][0], 2), "ms_per_step": round(res["step_nccl"][0] * 1e3, 4),
                         "allreduce_us_each": round(res["allreduce_only_nccl"][0] / (2 * c["layers"]) * 1e6, 2)},
                "max_abs_diff_vs_nccl": float((y1 - y2).abs().max()),
                "max_abs_diff_nccl_vs_nccl": float((y2 - y3).abs().max()),
                "ms_per_step_without_collectives": round(res["no_collective"][0] * 1e3, 4),
                "allreduce_us_each": round(res["allreduce_only"][0] / (2 * c["layers"]) * 1e6, 2),
                "allreduce_ms_per_step": round(res["allreduce_only"][0] * 1e3, 4),
                "per_gpu_gbs": round(alg * c["layers"] / t / 1e9, 1),
                "per_gpu_frac_of_hbm_peak": round(alg * c["layers"] / t / 1e9 / measured_peaks()["hbm_gbs"], 4),
                "limiter": "all-reduce latency" if res["allreduce_only"][0] > 0.5 * t else "weight streaming + launches"})
    return out


# ------------------------------------------------------------------- Mixtral leg (BASELINE config 4), N = 1
def mixtral_leg(torch, dev, steps, layers=32):
    """Mixtral-8x7B-shaped decode step (bs = 1): per layer RMSNorm -> fused qkv 4096x6144 -> o 4096x4096 -> RMSNorm ->
    router (fp16 4096 -> 8, torch.matmul: not quantised, awq/models/mixtral.py:129-158 keeps `gate` a plain nn.Linear)
    -> the reference's FusedSparseMoeBlock call sequence over OUR awq_ext (awq/modules/fused/moe.py:45-89: topk_softmax,
    moe_alig_block_size, grouped_gemm_forward gate|up, silu_and_mul, grouped_gemm_forward down x routing weight, sum).
    46.7 B parameters = 24 GB packed: it fits ONE B200 (the reference needed 2 x RTX 4090 for capacity, README.md:246),
    so per north_star ("shard only where the model exceeds one GPU") N GPUs = N replicas; this leg reports one."""
    import awq_ext

    E, H, I, topk, QKV = 8, HIDDEN, INTER, 2, 6144
    g = torch.Generator(device=dev).manual_seed(4242)

    def lin(K, N):
        return (torch.randint(-2**31, 2**31 - 1, (K, N // 8), dtype=torch.int32, device=dev, generator=g),
                ((torch.rand((K // GROUP, N), device=dev, generator=g) * 0.5 + 0.75) / (6.1 * K**0.5)).half(),
                torch.randint(-2**31, 2**31 - 1, (K // GROUP, N // 8), dtype=torch.int32, device=dev, generator=g))

    def stacked(K, N):
        return (torch.randint(-2**31, 2**31 - 1, (E, K, N // 8), dtype=torch.int32, device=dev, generator=g),
                ((torch.rand((E, K // GROUP, N), device=dev, generator=g) * 0.5 + 0.75) / (6.1 * K**0.5)).half(),
                torch.randint(-2**31, 2**31 - 1, (E, K // GROUP, N // 8), dtype=torch.int32, device=dev, generator=g))

    ws = [dict(qkv=lin(H, QKV), o=lin(H, H), w13=stacked(H, 2 * I), w2=stacked(I, H),
               router=(torch.randn((H, E), device=dev, generator=g) * 0.05).half()) for _ in range(layers)]
    nw = torch.ones(H, dtype=torch.float16, device=dev)
    h0 = torch.randn((1, H), device=dev, dtype=torch.float16, generator=g)
    xn = torch.empty((1, H), dtype=torch.float16, device=dev)
    tw = torch.empty((1, topk), dtype=torch.float32, device=dev)
    tid = torch.empty((1, topk), dtype=torch.int32, device=dev)
    src = torch.empty((1, topk), dtype=torch.int32, device=dev)
    s_ids = torch.empty((topk + E * 15,), dtype=torch.int32, device=dev)
    e_ids = torch.empty((topk + E,), dtype=torch.int32, device=dev)
    npost = torch.empty((1,), dtype=torch.int32, device=dev)
    act = torch.empty((1, topk, I), dtype=torch.float16, device=dev)

    def step():
        h = h0
        for w in ws:
            awq_ext.layernorm_forward_cuda(h, nw, xn, 1e-5)
            qkv = awq_ext.gemm_forward_cuda(xn, *w["qkv"], 8)
            a = awq_ext.gemm_forward_cuda(qkv[:, :H], *w["o"], 8)
            awq_ext.layernorm_forward_cuda(a, nw, xn, 1e-5)
            logits = torch.matmul(xn, w["router"]).float()
            awq_ext.topk_softmax(tw, tid, src, logits)
            s_ids.fill_(topk)
            awq_ext.moe_alig_block_size(tid, E, 16, s_ids, e_ids, npost)
            gu = awq_ext.grouped_gemm_forward(xn.view(1, 1, H), *w["w13"], tw, s_ids, e_ids, npost, False, 8)
            awq_ext.silu_and_mul(act, gu)
            out = awq_ext.grouped_gemm_forward(act, *w["w2"], tw, s_ids, e_ids, npost, True, 8)
            h = torch.sum(out, dim=1)
        return h

    from autoawq_b200 import ext as _ext

    gr, h_graph = capture(torch, step)
    n = max(5, steps // 2)
    sec = timed(torch, gr.replay, n, 3)
    torch.cuda.synchronize()
    # Validity of the TIMED configuration (graph, PDL as set).  The routing is data-dependent and the step is chaotic in
    # its rounding noise (fp32 split-K order can flip a near-tie in some layer), so two runs cannot be compared end to
    # end; but every layer must be consistent with ITS OWN inputs.  The last layer's state is still in the static buffers
    # after a replay: recompute its routing and its MoE output from them with plain torch on OUR dequantised weights.
    # (A launch-overlap race - a grouped GEMV reading the routing tables before its predecessor finished - made this
    # leg run "too fast" once: that is what this catches.)
    wl = ws[-1]
    logits_l = torch.matmul(xn, wl["router"]).float()
    probs = torch.softmax(logits_l, dim=-1)
    want_e = sorted(int(v) for v in torch.topk(probs, topk, dim=-1).indices.flatten().tolist())
    got_e = [int(v) for v in tid.flatten().tolist()]
    tw_ok = bool(torch.allclose(tw.flatten(), probs[0, got_e] if all(0 <= v < E for v in got_e) else tw.flatten() + 1,
                                atol=2e-3))
    h_ref = torch.zeros((1, H), dtype=torch.float32, device=dev)
    if sorted(got_e) == want_e:
        for k, ex in enumerate(got_e):
            w13 = awq_ext.dequantize_weights_cuda(wl["w13"][0][ex], wl["w13"][1][ex], wl["w13"][2][ex], 0, 0, 0, False)
            w2 = awq_ext.dequantize_weights_cuda(wl["w2"][0][ex], wl["w2"][1][ex], wl["w2"][2][ex], 0, 0, 0, False)
            gu_k = torch.matmul(xn.float(), w13.float())
            a_k = (torch.nn.functional.silu(gu_k[:, :I]) * gu_k[:, I:]).half().float()
            h_ref += tw[0, k] * torch.matmul(a_k, w2.float()).half().float()
            del w13, w2
    finite = bool(torch.isfinite(h_graph).all().item())
    rms = float(h_graph.float().pow(2).mean().sqrt().item()) if finite else float("nan")
    max_diff = float((h_graph.float() - h_ref).abs().max().item()) if finite else float("inf")
    if not finite or sorted(got_e) != want_e or not tw_ok or max_diff > 0.03 * max(rms, 1e-3) + 0.02:
        raise RuntimeError(f"mixtral leg: the timed step is not consistent with its own inputs (finite={finite}, last "
                           f"layer routed {got_e}, its logits say {want_e}, routing weights ok={tw_ok}, MoE output max "
                           f"|diff| vs torch {max_diff:.4f}, rms {rms:.4f})")
    # the same step without programmatic dependent launch, for the record (PDL hides the launch gaps of 416 small launches)
    pdl_was = _ext.get_knob(4)
    _ext.set_knob(4, 0)
    gr0, _ = capture(torch, step)
    sec0 = timed(torch, gr0.replay, n, 3)
    _ext.set_knob(4, pdl_was)
    experts_last = sorted(got_e)
    wb = lambda K, N: K * N // 2 + (K // GROUP) * N * 2 + (K // GROUP) * N // 2  # noqa: E731
    active = layers * (wb(H, QKV) + wb(H, H) + topk * (wb(H, 2 * I) + wb(I, H)))
    total = layers * (wb(H, QKV) + wb(H, H) + E * (wb(H, 2 * I) + wb(I, H)))
    t = sec / n
    return {"workload": f"Mixtral-8x7B W4A16 g128 decode bs=1, {layers} layers x [rmsnorm, qkv, o, rmsnorm, router, "
                        "topk_softmax, moe_align, grouped gate|up (2 of 8 experts), silu*mul, grouped down x weight, sum]",
            "tok_s": round(1.0 / t, 2), "ms_per_step": round(t * 1e3, 4), "active_gb_per_token": round(active / 1e9, 3),
            "weights_gb": round(total / 1e9, 2), "gbs_over_active_bytes": round(active / t / 1e9, 1),
            "frac_of_hbm_peak": round(active / t / 1e9 / measured_peaks()["hbm_gbs"], 4),
            "launches_per_step": layers * 13, "cuda_graph": True,
            "ms_per_step_without_pdl": round(sec0 / n * 1e3, 4),
            "checked": {"output_finite": finite, "output_rms": round(rms, 4), "experts_last_layer": experts_last,
                        "last_layer_routing_matches_its_logits": True,
                        "last_layer_moe_max_abs_diff_vs_torch": round(max_diff, 5)},
            "multi_gpu": "fits one B200 (24 GB): 2 GPUs = 2 replicas, as for Llama-3-8B"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--mode", choices=["decode", "prefill"], default="decode")
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--pdl", type=int, default=1, help="1: launch kernels with programmatic dependent launch")
    ap.add_argument("--nextw", type=int, default=0, help="1: learned next-weight L2 prefetch (knob 6)")
    ap.add_argument("--knob", action="append", default=[], help="debug: KEY=VALUE library knob (repeatable)")
    ap.add_argument("--program", type=int, default=1,
                    help="decode: 1 = record the step once and run it as ONE persistent kernel (b200awq_program_*); "
                         "0 = one kernel launch per operator call")
    ap.add_argument("--layers", type=int, default=LAYERS, help="debug only: fewer layers => INVALID as a bench value")
    ap.add_argument("--tp-layers", type=int, default=0, help="debug: layers of the tensor-parallel leg (0 = all 80)")
    ap.add_argument("--legs", type=int, default=1,
                    help="1: also run the secondary legs at N=1 (4096x4096 GEMV, small batch, prefill, Mixtral); "
                         "0: headline only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step to DIR/output.npy (float32) for comparing builds")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    M = 1 if a.mode == "decode" else 4096
    tokens_per_step = M
    metric = f"{a.mode} tok/s Llama-3-8B W4A16 (quantised linears, bs=1" + (", seq=1)" if M == 1 else ", seq=4096)")
    config = {"workload": f"Llama-3-8B W4A16 GEMM-layout g128, {a.mode} bs=1 seq={M}: 32 layers x "
                          "[rmsnorm, qkv 4096x6144, o 4096x4096, rmsnorm, gate|up 4096x28672, silu*mul, down 14336x4096]",
              "weights": "random-init AWQ-packed, distinct per layer (3.63 GB/replica)",
              "l2": "inputs larger than L2: 3.63 GB of weights streamed per step vs 126 MB L2",
              "parallelism": f"replicas x{a.gpus}" if a.gpus > 1 else "single GPU", "layers": a.layers}

    # ------------------------------------------------------------------ reference arm (CPU)
    if a.impl == "reference":
        if rank != 0:
            return
        layers_sample = 1
        per_layer = []
        threads = pick_cpu_threads(M if M == 1 else 64)
        cores = threads
        for i in range(a.warmup + a.steps):
            t, cores = cpu_reference_sample(M if M == 1 else 64, layers_sample, 1, threads=threads)
            if i >= a.warmup:
                per_layer.append(t)
            if M == 1 and sum(per_layer) > 150:
                break
        mean_layer = sum(per_layer) / len(per_layer)
        m_eff = M if M == 1 else 64
        val = m_eff / (mean_layer * LAYERS)
        line = {"impl": "reference", "metric": metric, "value": val, "unit": "tok/s", "n_gpus": a.gpus,
                "steps": len(per_layer), "warmup": a.warmup, "ms_per_step": mean_layer * LAYERS * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": val, "unit": "tok/s", "cores": cores, "kind": "port",
                                 "sample": f"{layers_sample} of 32 layers per step (4 linears, dequantize_gemm + "
                                           f"torch.matmul fp16, M={m_eff}), x32 extrapolated; thread count "
                                           f"auto-picked from a sweep (fastest)"},
                "e2e": {"value": val, "unit": "tok/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0,
                # the CPU path takes ~15 s per sampled layer at M = 1: the run stops after 150 s of samples and says so
                "steps_requested": a.steps, "steps_truncated": len(per_layer) < a.steps}
        print(json.dumps(line), flush=True)
        return

    # ------------------------------------------------------------------------- B200 arm
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the product path)")
    dist = None
    nccl_log = None
    if world > 1:
        # NCCL's INFO log (communicator ranks, NVLS / ring choice) goes to STDERR: stdout carries exactly one JSON line
        if os.environ.get("NCCL_DEBUG", "").upper() not in ("INFO", "TRACE"):
            os.environ["NCCL_DEBUG"] = "INFO"
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT,GRAPH")
        if "NCCL_DEBUG_FILE" not in os.environ:      # (a caller's own NCCL log file wins)
            logdir = tempfile.gettempdir()
            os.environ["NCCL_DEBUG_FILE"] = os.path.join(logdir, "nccl_bench.%h.%p.log")
            nccl_log = os.path.join(logdir, f"nccl_bench.{os.uname().nodename}.{os.getpid()}.log")
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
        if rank == 0 and nccl_log and os.path.exists(nccl_log):      # the communicator's own words, on stderr
            for ln in open(nccl_log, errors="replace"):
                if "nranks" in ln or "NVLS" in ln or "Connected" in ln:
                    print(ln.rstrip(), file=sys.stderr)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    rep = Replica(dev, M, layers=a.layers, seed=rank)
    rep.ext.set_knob(4, 1 if a.pdl else 0)
    rep.ext.set_knob(6, 1 if a.nextw else 0)
    for kv in a.knob:
        k, v = kv.split("=")
        rep.ext.set_knob(int(k), int(v))
        config.setdefault("knobs", {})[k] = int(v)
    config["pdl"] = bool(a.pdl)
    config["next_weight_l2_prefetch"] = bool(a.nextw)
    peaks = measured_peaks()

    # the step as ONE persistent kernel (decode): same operator calls, recorded once through the recorder that
    # mirrors the awq_ext call names, replayed by b200awq_program_run
    prog = None
    if a.mode == "decode" and a.program:
        from autoawq_b200.program import DecodeProgram

        prog = DecodeProgram()
        prog_out = rep.step(rep.h, api=prog)
        prog.build()
        if not prog.fused:
            prog = None
        else:
            config["program_kind"] = prog.kind
            config["program_calibration"] = prog.calibration

    # per-op path: the step replayed as one CUDA graph of 224 kernel launches
    g_ops, out_ops = capture(torch, lambda: rep.step(rep.h))
    per_op = None
    if prog is not None:
        sec_ops = timed(torch, g_ops.replay, a.steps, a.warmup, dist)
        per_op = {"tok_s": round(world * tokens_per_step * a.steps / sec_ops, 2),
                  "ms_per_step": round(sec_ops / a.steps * 1e3, 4), "launches_per_step": rep.launches_per_step}
        g_step, _ = capture(torch, prog.run)
        out_static = prog_out
        launches_per_step = 1
    else:
        g_step, out_static = g_ops, out_ops
        launches_per_step = rep.launches_per_step

    # value leg: inputs resident in HBM, the step replayed as one CUDA graph
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t_wall0 = time.time()
    sec = timed(torch, g_step.replay, a.steps, a.warmup, dist)
    t_wall1 = time.time()
    if rank == 0 and a.dump_outputs:
        dump_outputs(a.dump_outputs, out_static)
    clocks = None
    if rank == 0:
        t_ext = None
        if 0 <= sampler.count(t_wall0, t_wall1) < 3:
            # the timed region of a decode run is ~40 ms: keep the identical load up (untimed) until the sampler has seen it
            t_end = time.time() + 0.25
            while time.time() < t_end and sampler.count(t_wall0, time.time()) < 5:
                g_step.replay()
                torch.cuda.synchronize()
            t_ext = time.time()
        clocks = sampler.stop(t_wall0, t_wall1, t_ext)
    if dist is not None:
        dist.barrier()
    value = world * tokens_per_step * a.steps / sec

    # What did the timed region compute?  (1) The per-op path is deterministic: its graph under PDL must reproduce the
    # eager run in plain stream order bit for bit.  (2) The decode program rounds differently from the per-op kernels
    # (fixed-point packed sums) and this chain of 32 random-init layers without residuals amplifies one-ulp differences
    # to O(1) by the last layer (measured: max |diff| 4.0 at rms 0.76), so the two paths cannot be compared end to end;
    # instead the LAST layer of the timed run is checked against its own inputs, which are still in the static buffers
    # after a replay: act = silu(gate) * up of xn, and y = act . W_down, recomputed with torch on our dequantised weights.
    if rank == 0 and a.mode == "decode":
        try:
            torch.cuda.synchronize()
            y_timed = out_static.float().clone()
            xn_l, act_l = rep.xn.float().clone(), rep.act.float().clone()
            lw_last = rep.w[-1]
            w_gu = rep.ext.dequantize_weights_cuda(*lw_last["gate_up"]).float()
            gu = torch.matmul(xn_l, w_gu)
            act_ref = torch.nn.functional.silu(gu[:, :INTER]) * gu[:, INTER:]
            del w_gu, gu
            w_dn = rep.ext.dequantize_weights_cuda(*lw_last["down"]).float()
            y_ref_last = torch.matmul(act_l, w_dn)
            del w_dn
            d_act = float((act_l - act_ref).abs().max().item())
            d_y = float((y_timed - y_ref_last).abs().max().item())
            rms_act = float(act_ref.pow(2).mean().sqrt().item())
            rms_y = float(y_ref_last.pow(2).mean().sqrt().item())
            chk = {"finite": bool(torch.isfinite(y_timed).all().item()), "output_rms": round(rms_y, 4),
                   "last_layer_act_max_abs_diff_vs_torch": round(d_act, 6),
                   "last_layer_output_max_abs_diff_vs_torch": round(d_y, 6),
                   # fp16 rounding of gate|up (2^-11 relative, |gate|, |up| up to ~5) propagates to ~0.01 on the largest
                   # activations; work that was skipped or raced would be off by O(1)
                   "last_layer_consistent": bool(d_act <= 0.03 * rms_act + 0.03 and d_y <= 0.03 * rms_y + 0.03),
                   "how": "after the last timed replay: silu(gate) * up of the stored xn vs the stored act, act . W_down vs "
                          "the step's output, torch fp32 on dequantize_weights_cuda of the last layer's tensors"}
            pdl_was = rep.ext.get_knob(4)
            rep.ext.set_knob(4, 0)
            try:
                y_eager = rep.step(rep.h).float().clone()
                torch.cuda.synchronize()
            finally:
                rep.ext.set_knob(4, pdl_was)
            g_ops.replay()
            torch.cuda.synchronize()
            chk["per_op_graph_with_pdl_vs_eager_max_abs_diff"] = round(float((out_ops.float() - y_eager).abs().max().item()), 6)
            config["output_check"] = chk
        except Exception as ex:  # noqa: BLE001  (a check must never take the bench line down)
            config["output_check"] = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}

    # roofline leg: the quantised-linear kernels alone, same weights
    g_lin, _ = capture(torch, lambda: rep.gemm_only(rep.h))
    sec_lin = timed(torch, g_lin.replay, a.steps, a.warmup, dist)
    n_lin = 4 * a.layers
    alg_bytes = sum(linear_bytes(K, N, M) for _, K, N in LINEARS) * a.layers
    alg_flops = sum(2.0 * M * K * N for _, K, N in LINEARS) * a.layers
    avg_launch_s = sec_lin / a.steps / n_lin
    if prog is not None:
        # the dominant (only) kernel is the program kernel: one launch streams every linear of the step
        step_s = sec / a.steps
        ach = alg_bytes / step_s / 1e9
        lin_ach = alg_bytes / n_lin / avg_launch_s / 1e9
        per_op["linear_avg_us"] = round(avg_launch_s * 1e6, 2)
        per_op["linear_gbs"] = round(lin_ach, 1)
        per_op["linear_frac"] = round(lin_ach / peaks["hbm_gbs"], 4)
        roof = {"bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(ach / peaks["hbm_gbs"], 4),
                # dram__bytes_read + write per program_kernel launch, one ncu --set full capture of this command:
                # profiles/r02_ncu_program_kernel.md (3,629.7 MB read + 30.5 MB written; algorithmic 3,626 MB).
                # Captured for the split-K kernel; the stream kernel reads the same bytes by construction (no ncu).
                "traffic": (3629674000 + 30530560) if (a.layers == LAYERS and prog.kind != "stream") else None,
                "kernel": ("stream_program_kernel" if prog.kind == "stream" else "program_kernel") +
                          " (persistent decode program: 128 linears + glue per launch)",
                "peak_src": peaks["src"] + " (hbm_gbs)",
                "per_launch": {"avg_us": round(step_s * 1e6, 2), "alg_bytes": alg_bytes,
                               "launches_timed": a.steps,
                               "how": "CUDA events around graph replays of b200awq_program_run (memset + kernel); "
                                      "algorithmic bytes = packed weights + scales + zeros + activations of all "
                                      "128 linears"}}
    elif a.mode == "decode":
        ach = alg_bytes / n_lin / avg_launch_s / 1e9
        roof = {"bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(ach / peaks["hbm_gbs"], 4),
                # dram__bytes_read + write per launch, averaged over one layer's four GEMV launches, from the committed
                # ncu --set full capture profiles/r01_gemv_v3_one_layer_M1.md (113.69 MB / 4; algorithmic 113.31 MB / 4)
                "traffic": 28422000 if a.layers == LAYERS else None,
                "kernel": "gemv_v3_kernel<1> (persistent TMA-ring GEMV)", "peak_src": peaks["src"] + " (hbm_gbs)",
                "per_launch": {"avg_us": round(avg_launch_s * 1e6, 2), "alg_bytes": alg_bytes // n_lin,
                               "launches_timed": n_lin * a.steps,
                               "how": "CUDA events around a graph of the 128 linear launches of one step"}}
    else:
        ach = alg_flops / n_lin / avg_launch_s / 1e12
        pk = peaks["bf16_tflops_sustained"]
        roof = {"bound": "tensor", "achieved": round(ach, 1), "peak": pk, "unit": "TFLOP/s",
                "frac": round(ach / pk, 4), "traffic": None, "kernel": "gemm_tc_kernel<256,0>",
                "peak_src": peaks["src"] + " (bf16_tflops_sustained: kernel timed inside a long step)",
                "per_launch": {"avg_us": round(avg_launch_s * 1e6, 2), "alg_flops": alg_flops / n_lin,
                               "launches_timed": n_lin * a.steps}}

    # e2e leg: host buffers, H2D + plugin calls + D2H inside the timed region
    h_host = torch.randn((M, HIDDEN), dtype=torch.float16).pin_memory()
    y_host = torch.empty((M, HIDDEN), dtype=torch.float16).pin_memory()

    def e2e_step():
        rep.h.copy_(h_host, non_blocking=True)
        g_step.replay()
        y_host.copy_(out_static, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    sec_e2e = timed(torch, e2e_step, a.steps, a.warmup, dist)
    e2e_val = world * tokens_per_step * a.steps / sec_e2e

    # eager plugin calls (no graph): what a Python caller that does not capture graphs sees
    def eager_step():
        rep.h.copy_(h_host, non_blocking=True)
        if prog is not None:
            prog.run()
            y = prog_out
        else:
            y = rep.step(rep.h)
        y_host.copy_(y, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    n_eager = max(3, a.steps // 5)
    sec_eager = timed(torch, eager_step, n_eager, 2, dist)

    # secondary legs (N = 1 only; the headline metric is unchanged): the metric's own 4096 x 4096 GEMV, small batches,
    # config 3 (prefill) and Mixtral - all CUDA-event timed like the value leg
    if world == 1 and a.legs:
        if a.mode == "decode":
            config["gemv_4096"] = gemv_4096_leg(torch, rep.ext, dev, a.steps, peaks)
            config["small_batch"] = small_batch_leg(torch, rep.ext, dev, a.steps, peaks)
            eager_ops = timed(torch, lambda: rep.step(rep.h), max(3, a.steps // 5), 2)
            config["per_op_eager_tok_s"] = round(max(3, a.steps // 5) / eager_ops, 1)
            config["prefill"] = prefill_leg(torch, rep.w, dev, a.steps, peaks)
            try:
                config["mixtral"] = mixtral_leg(torch, dev, a.steps)
            except Exception as ex:  # noqa: BLE001
                config["mixtral"] = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}
    # N > 1: the tensor-parallel leg (config 5); 35.6 GB / N of packed weights per GPU next to the replica's 7 GB
    if world > 1 and a.legs and a.mode == "decode":
        try:
            config["tp70b"] = tp70b_leg(torch, dist, rank, world, dev, max(5, a.steps // 2), a.tp_layers)
        except Exception as ex:  # noqa: BLE001
            config["tp70b"] = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    # CPU baseline on rank 0, N = 1 only (bounded sample)
    cpu = None
    if world == 1:
        t_layer, cores = cpu_reference_sample(M if M == 1 else 64, 1, 2, threads=pick_cpu_threads(M if M == 1 else 64))
        m_eff = M if M == 1 else 64
        cpu = {"value": m_eff / (t_layer * LAYERS), "unit": "tok/s", "cores": cores, "kind": "port",
               "sample": f"1 of 32 layers (4 linears, dequantize_gemm + torch.matmul fp16, M={m_eff}), best of 2, x32"}
    config["e2e_eager_tok_s"] = round(world * tokens_per_step * n_eager / sec_eager, 1)
    if prog is not None:
        config["value_leg"] = ("CUDA-graph replay of b200awq_program_run: the step's awq_ext-facing operator calls "
                               "recorded once, executed as one persistent kernel; inputs resident in HBM")
        config["per_op_path"] = per_op
    else:
        config["value_leg"] = "CUDA-graph replay of the awq_ext-facing operator calls, inputs resident in HBM"
    line = {"metric": metric, "value": round(value, 2), "unit": "tok/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": round(sec / a.steps * 1e3, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": config,
            "clocks": clocks,
            "e2e": {"value": round(e2e_val, 2), "unit": "tok/s", "h2d_bytes_per_step": M * HIDDEN * 2,
                    "d2h_bytes_per_step": M * HIDDEN * 2},
            "gpu_launches": launches_per_step * a.steps,
            "roofline": roof, "cpu_baseline": cpu}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
