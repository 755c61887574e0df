"""First-contact GPU diagnostics + micro-benchmarks (run under gpurun; writes gpurun_out/probe.json).

1. which UMMA A-descriptor variant (knob 3) reproduces the oracle on the tensor-core path;
2. correctness spot-checks of every kernel family;
3. kernel timings (CUDA events, rotating weight pool > L2) for the Llama-3-8B linear shapes.
"""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from autoawq_b200 import ext  # noqa: E402
from oracle import awq_oracle as O  # noqa: E402

dev = torch.device("cuda:0")
out = {"device": torch.cuda.get_device_name(0)}


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def relerr(y, ref):
    return float(np.abs(y.astype(np.float64) - ref).max() / (np.abs(ref).max() + 1e-12))


def check_paths():
    res = {}
    K, N, G = 512, 256, 128
    c = O.make_case(K, N, G, seed=0)
    w = O.dequantize_gemm(c["qweight"], c["qzeros"], c["scales"], G)
    wd = ext.dequantize_weights_cuda(t(c["qweight"]), t(c["scales"]), t(c["qzeros"]))
    res["dequant_bit_exact"] = bool(np.array_equal(wd.cpu().numpy().view(np.uint16), w.view(np.uint16)))
    rng = np.random.default_rng(0)
    for M in (1, 4, 8):
        x = rng.standard_normal((M, K)).astype(np.float16)
        y = ext.linear_forward("gemm", t(x), t(c["qweight"]), t(c["scales"]), t(c["qzeros"]), G).cpu().numpy()
        res[f"gemv_M{M}_relerr"] = relerr(y, O.gemm_f64(x, w))
    for variant in (0,):
        ext.set_knob(3, variant)
        for M in (16, 100, 256):
            x = rng.standard_normal((M, K)).astype(np.float16)
            try:
                y = ext.linear_forward("gemm", t(x), t(c["qweight"]), t(c["scales"]), t(c["qzeros"]), G).cpu().numpy()
                torch.cuda.synchronize()
                res[f"tc_variant{variant}_M{M}_relerr"] = relerr(y, O.gemm_f64(x, w))
            except Exception as e:  # noqa: BLE001
                res[f"tc_variant{variant}_M{M}_relerr"] = f"ERR {e}"
    ext.set_knob(3, 0)
    vw, vz, vs = O.pack_gemv(c["intweight"], c["zeros"], c["scales"], G)
    fw, fs, fz = O.pack_gemv_fast(c["intweight"], c["zeros"], c["scales"], G)
    wf = O.dequantize_gemv_fast_f64(fw, fs, fz, G)
    for M in (1, 8, 64):
        x = rng.standard_normal((M, K)).astype(np.float16)
        yv = ext.linear_forward("gemv", t(x), t(vw), t(vs), t(vz), G).cpu().numpy()
        yf = ext.linear_forward("fast", t(x), t(fw), t(fs), t(fz), G).cpu().numpy()
        res[f"gemvlayout_M{M}_relerr"] = relerr(yv, O.gemm_f64(x, w))
        res[f"fastlayout_M{M}_relerr"] = relerr(yf, O.gemm_f64(x, wf))
    return res


def time_kernel(fn, nbuf, iters=200, warm=20):
    """Device time per call: the nbuf calls (rotating weight buffers, pool > L2) are captured into ONE CUDA
    graph so that Python / ctypes launch overhead (~15 us per call) is not what gets measured."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(min(nbuf, 3)):
            fn(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for i in range(nbuf):
            fn(i)
    reps = max(1, iters // nbuf)
    for _ in range(max(1, warm // nbuf)):
        g.replay()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(reps):
        g.replay()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / (reps * nbuf) * 1e3  # us


def bench_shapes():
    res = {}
    G = 128
    shapes = [(4096, 4096), (4096, 6144), (4096, 14336), (14336, 4096), (4096, 28672)]
    for (K, N) in shapes:
        wbytes = K * N // 2 + (K // G) * N * 2 + (K // G) * N // 2
        nbuf = max(3, int(400e6 // wbytes) + 1)
        qw = [torch.randint(-2**31, 2**31 - 1, (K, N // 8), dtype=torch.int32, device=dev) for _ in range(nbuf)]
        qz = [torch.randint(-2**31, 2**31 - 1, (K // G, N // 8), dtype=torch.int32, device=dev) for _ in range(nbuf)]
        sc = [(torch.rand((K // G, N), device=dev) * 0.01 + 0.001).half() for _ in range(nbuf)]
        for M in (1, 8, 16, 64, 256, 4096):
            if M > 8 and N == 28672 and M > 256:
                continue
            x = torch.randn((M, K), device=dev, dtype=torch.float16)
            try:
                us = time_kernel(lambda i: ext.linear_forward("gemm", x, qw[i], sc[i], qz[i], G), nbuf,
                                 iters=100 if M <= 256 else 20, warm=5)
                byts = wbytes + 2 * M * K + 2 * M * N
                res[f"gemm_K{K}_N{N}_M{M}"] = {"us": round(us, 2), "GBps": round(byts / us / 1e3, 1),
                                                "TFLOPs": round(2.0 * M * K * N / us / 1e6, 1)}
            except Exception as e:  # noqa: BLE001
                res[f"gemm_K{K}_N{N}_M{M}"] = f"ERR {e}"
        # dequant kernel
        us = time_kernel(lambda i: ext.dequantize_weights_cuda(qw[i], sc[i], qz[i]), nbuf, iters=50, warm=5)
        res[f"dequant_K{K}_N{N}"] = {"us": round(us, 2), "GBps": round((wbytes + 2 * K * N) / us / 1e3, 1)}
        del qw, qz, sc
        torch.cuda.empty_cache()
    # python/ctypes call overhead: tiny problem
    x = torch.randn((1, 128), device=dev, dtype=torch.float16)
    qw = torch.zeros((128, 16), dtype=torch.int32, device=dev)
    qz = torch.zeros((1, 16), dtype=torch.int32, device=dev)
    sc = torch.ones((1, 128), dtype=torch.float16, device=dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(2000):
        ext.linear_forward("gemm", x, qw, sc, qz, 128)
    torch.cuda.synchronize()
    res["host_call_us"] = round((time.perf_counter() - t0) / 2000 * 1e6, 2)
    return res


def bench_gemv_knobs():
    """M = 1 decode GEMV: rows-per-warp (knob 0) x PDL (knob 4) sweep on the four Llama-3-8B shapes."""
    res = {}
    G = 128
    for (K, N) in [(4096, 4096), (4096, 6144), (4096, 28672), (14336, 4096)]:
        wbytes = K * N // 2 + (K // G) * N * 2 + (K // G) * N // 2
        nbuf = max(3, int(400e6 // wbytes) + 1)
        qw = [torch.randint(-2**31, 2**31 - 1, (K, N // 8), dtype=torch.int32, device=dev) for _ in range(nbuf)]
        qz = [torch.randint(-2**31, 2**31 - 1, (K // G, N // 8), dtype=torch.int32, device=dev) for _ in range(nbuf)]
        sc = [(torch.rand((K // G, N), device=dev) * 0.01 + 0.001).half() for _ in range(nbuf)]
        x = torch.randn((1, K), device=dev, dtype=torch.float16)
        for name, k5, rw in (("v3", 0, 0), ("v2rw64", 1, 64)):
            for pdl in (0, 1):
                for M in (1, 8):
                    xm = torch.randn((M, K), device=dev, dtype=torch.float16)
                    ext.set_knob(5, k5)
                    ext.set_knob(0, rw)
                    ext.set_knob(4, pdl)
                    try:
                        us = time_kernel(lambda i: ext.linear_forward("gemm", xm, qw[i], sc[i], qz[i], G), nbuf, iters=200, warm=10)
                        res[f"K{K}_N{N}_{name}_pdl{pdl}_M{M}"] = {"us": round(us, 2), "GBps": round((wbytes + 2 * M * K + 2 * M * N) / us / 1e3, 1)}
                    except Exception as e:  # noqa: BLE001
                        res[f"K{K}_N{N}_{name}_pdl{pdl}_M{M}"] = f"ERR {e}"
        ext.set_knob(0, 0)
        ext.set_knob(4, 0)
        ext.set_knob(5, 0)
        del qw, qz, sc
        torch.cuda.empty_cache()
    return res


if __name__ == "__main__":
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    out["checks"] = check_paths()
    print(json.dumps(out["checks"], indent=1), flush=True)
    if "--knobs" in sys.argv:
        out["gemv_knobs"] = bench_gemv_knobs()
        print(json.dumps(out["gemv_knobs"], indent=1), flush=True)
    if "--no-bench" not in sys.argv:
        out["bench"] = bench_shapes()
        print(json.dumps(out["bench"], indent=1), flush=True)
    json.dump(out, open(os.path.join(ROOT, "gpurun_out", "probe.json"), "w"), indent=1)
