"""The drop-in, exercised as the reference package (casper-hansen/AutoAWQ @ 88e4c76) calls it: tests/golden/
dropin_calls.json holds every `awq_ext` / `awq_v2_ext` call that the reference's own module classes make - WQLinear_GEMM
forward in every dispatch arm and backward (awq/modules/linear/gemm.py:24-298), WQLinear_GEMV / GEMVFast (gemv.py:27-197,
gemv_fast.py:68-208), FasterTransformerRMSNorm (fused/norm.py:19-38), fuse_qkv (utils/fused_utils.py:45-142),
apply_moe_weights, fused_topk and moe_align_block_size (fused/moe.py:45-170) - recorded by tests/golden/
make_dropin_calls.py: function, argument order, scalars, tensor shapes / dtypes and where each tensor comes from.
These tests rebuild the same seeded inputs, replay the calls on this repository's extension modules and compare the
results with the CPU oracle (fp64 contraction of the bit-exact dequantised weights), not with this repo's mirrors.
"""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from oracle import awq_oracle as O

pytestmark = pytest.mark.gpu

RTOL, WR_GEMV, WR_TC = 2.0**-10, 2.0**-11, 2.0**-16
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_DT = {"float16": torch.float16, "bfloat16": torch.bfloat16, "float32": torch.float32, "int16": torch.int16,
       "int32": torch.int32}


def _dev():
    return torch.device("cuda:0")


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(_dev())


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint16)


def _budget(x, w):
    return np.abs(np.asarray(x, dtype=np.float64)) @ np.abs(np.asarray(w, dtype=np.float64))


def _close(y, ref64, budget, wr, what=""):
    y = np.asarray(y, dtype=np.float64)
    tol = RTOL * np.abs(ref64) + wr * budget + 1e-6
    bad = np.abs(y - ref64) > tol
    assert not bad.any(), f"{what}: {bad.sum()} / {bad.size} outside tolerance, max err {np.abs(y - ref64).max():.3e}"


@pytest.fixture(scope="module")
def calls():
    with open(os.path.join(GOLDEN, "dropin_calls.json")) as f:
        return json.load(f)


def _segments(calls, scenario):
    return {s["label"]: s for s in calls["segments"][scenario]}


def _replay(segment, inputs):
    """Makes the recorded calls of one segment on this repository's awq_ext / awq_v2_ext, with the tensors built from
    `inputs` (name -> tensor), from earlier calls' results, or as the reference allocated them.  Returns one
    (args, result) pair per call."""
    import awq_ext
    import awq_v2_ext

    mods = {"awq_ext": awq_ext, "awq_v2_ext": awq_v2_ext}
    done = []
    for c in segment["calls"]:
        args = []
        for a in c["args"]:
            if "v" in a:
                args.append(a["v"])
                continue
            shape, dt = tuple(a["shape"]), _DT[a["dtype"]]
            if "in" in a:
                t = inputs[a["in"]].to(dt).reshape(shape)
            elif "call" in a:
                prev_args, prev_ret = done[a["call"]]
                t = prev_ret if a["arg"] == "ret" else prev_args[a["arg"]]
                assert tuple(t.shape) == shape and t.dtype == dt, (c["fn"], a)
            elif "values" in a:
                t = torch.tensor(a["values"], dtype=dt, device=_dev()).reshape(shape)
            elif "fill" in a:
                t = torch.full(shape, a["fill"], dtype=dt, device=_dev())
            else:
                t = torch.empty(shape, dtype=dt, device=_dev())
            args.append(t)
        ret = getattr(mods[c["mod"]], c["fn"])(*args)
        if c["ret"] is None:
            assert ret is None, c["fn"]
        else:
            assert tuple(ret.shape) == tuple(c["ret"]["shape"]) and ret.dtype == _DT[c["ret"]["dtype"]], c["fn"]
        done.append((args, ret))
    torch.cuda.synchronize()
    return done


def _gemm_inputs(c):
    return {"qweight": _t(c["qweight"]), "scales": _t(c["scales"]), "qzeros": _t(c["qzeros"])}


# ------------------------------------------------------------------ WQLinear_GEMM (gemm.py:116-298), all dispatch arms
@pytest.mark.parametrize("K,N,G", [(512, 256, 128), (1024, 1792, 128), (4096, 4096, 128), (256, 64, 64)])
def test_reference_wqlinear_gemm_forward(calls, K, N, G):
    segs = _segments(calls, f"gemm_forward_{K}_{N}_{G}")
    c = O.make_case(K, N, G, seed=K + N)
    w = O.dequantize_gemm(c["qweight"], c["qzeros"], c["scales"], G)
    inputs = _gemm_inputs(c)
    rng = np.random.default_rng(3)
    # [1,1,K] / [1,8,K]: gemm_forward_cuda (gemm.py:56-58); [1,40,K]: same entry, tensor-core kernel;
    # [2,600,K]: B*S >= 1024 -> dequantize_weights_cuda + torch.matmul (gemm.py:50-54); 2-D: M*K >= 1024 -> same
    cases = [((1, 1, K), np.float16), ((1, 8, K), np.float16), ((1, 40, K), np.float16), ((2, 600, K), np.float16),
             ((3, K), np.float16), ((2, 3, K), None)]
    for shape, dt in cases:
        label = str(shape) if dt is not None else "bf16 (2, 3, K)"
        if dt is None:   # a bf16 input: the module casts it to fp16 before the call (gemm.py:43)
            xt = torch.randn(shape, device=_dev(), dtype=torch.bfloat16)
            x = xt.half().cpu().numpy()
        else:
            x = (rng.standard_normal(shape) * 0.5).astype(np.float16)
            xt = _t(x)
        [(args, y)] = _replay(segs[label], dict(inputs, x=xt))
        x2 = x.reshape(-1, K)
        if segs[label]["calls"][0]["fn"] == "dequantize_weights_cuda":
            # the reference multiplies by the dequantised weight itself: the extension's part is that weight, bit for bit
            assert np.array_equal(_bits(y.cpu().numpy()), _bits(w)), f"dequantize_weights_cuda {shape}"
        else:
            wr = WR_GEMV if x2.shape[0] <= 8 else WR_TC
            _close(y.cpu().numpy().reshape(x2.shape[0], N), O.gemm_f64(x2, w), _budget(x2, w), wr,
                   f"ref WQLinear_GEMM {shape}")
    # an empty batch returns before any extension call (gemm.py:44-45)
    assert segs["empty batch"]["calls"] == []


def test_reference_from_linear_then_forward(calls):
    """The reference packer (gemm.py:171-251) gave exactly the oracle's packed buffers; its forward on our kernels."""
    K, N, G = 256, 128, 64
    rng = np.random.default_rng(0)
    iw, iz, s = O.quantize_rtn((rng.standard_normal((N, K)) * 0.05).astype(np.float32), G)
    qw, qz = O.pack_gemm(iw, iz)
    packed = {"qweight": qw, "scales": s.astype(np.float16), "qzeros": qz}
    for name, a in packed.items():
        assert hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest() == calls["from_linear_sha256"][name], name
    wq = O.dequantize_gemm(qw, qz, s, G)
    x = (rng.standard_normal((1, 5, K))).astype(np.float16)
    [(_, y)] = _replay(calls["segments"]["from_linear"][0], dict({k: _t(v) for k, v in packed.items()}, x=_t(x)))
    _close(y.cpu().numpy().reshape(5, N), O.gemm_f64(x[0], wq), _budget(x[0], wq), WR_GEMV, "from_linear fwd")


def test_reference_backward(calls):
    """WQLinearMMFunction.backward (gemm.py:88-114): dX = dY . W^T through awq_ext.dequantize_weights_cuda(…,1,0,0,False);
    no weight gradient.  Replayed as the reference module calls it in training mode, and through this repo's mirror."""
    from autoawq_b200.linear import WQLinear_GEMM as Mirror

    K, N, G = 512, 256, 128
    c = O.make_case(K, N, G, seed=9)
    w16 = O.dequantize_gemm(c["qweight"], c["qzeros"], c["scales"], G)
    w = w16.astype(np.float64)
    rng = np.random.default_rng(4)
    x = (rng.standard_normal((2, 6, K)) * 0.5).astype(np.float16)
    gy = (rng.standard_normal((2, 6, N)) * 0.5).astype(np.float16)
    ref_gx = gy.astype(np.float64) @ w.T
    (_, y), (_, wd) = _replay(calls["segments"]["backward"][0], dict(_gemm_inputs(c), x=_t(x)))
    x2 = x.reshape(-1, K)
    _close(y.cpu().numpy(), O.gemm_f64(x2, w16), _budget(x2, w16), WR_TC, "training forward")
    assert np.array_equal(_bits(wd.cpu().numpy()), _bits(w16)), "backward's dequantised weight"
    m = Mirror(4, G, K, N, False, _dev())
    m.training = True
    m.qweight.copy_(_t(c["qweight"]))
    m.qzeros.copy_(_t(c["qzeros"]))
    m.scales.copy_(_t(c["scales"]))
    xt = _t(x).requires_grad_(True)
    y = m(xt)
    assert y.requires_grad
    y.backward(_t(gy))
    gx = xt.grad.float().cpu().numpy()
    assert gx.shape == x.shape
    tol = 2.0**-9 * np.abs(ref_gx) + 2.0**-10 * (np.abs(gy.astype(np.float64)) @ np.abs(w.T)) + 1e-4
    assert np.all(np.abs(gx - ref_gx) <= tol), f"mirror: max err {np.abs(gx - ref_gx).max():.3e}"


# ----------------------------------------------------------- WQLinear_GEMV / GEMVFast (gemv.py:27-197, gemv_fast.py:68-208)
@pytest.mark.parametrize("K,N,G", [(512, 128, 128), (4096, 512, 128), (1024, 256, 64)])
def test_reference_wqlinear_gemv_and_fast_forward(calls, K, N, G):
    segs = _segments(calls, f"gemv_{K}_{N}_{G}")
    c = O.make_case(K, N, G, seed=K)
    w = O.dequantize_gemm(c["qweight"], c["qzeros"], c["scales"], G)
    vw, vz, vs = O.pack_gemv(c["intweight"], c["zeros"], c["scales"], G)
    fw, fs, fz = O.pack_gemv_fast(c["intweight"], c["zeros"], c["scales"], G)
    wfast = O.dequantize_gemv_fast_f64(fw, fs, fz, G)
    rng = np.random.default_rng(1)
    # GEMV module: M <= 8 -> gemv_forward_cuda, M > 8 -> gemmv2_forward_cuda (gemv.py:168-180)
    for shape in [(1, 1, K), (2, 4, K), (1, 24, K)]:
        x = (rng.standard_normal(shape) * 0.5).astype(np.float16)
        x2 = x.reshape(-1, K)
        [(_, y)] = _replay(segs[f"gemv {shape}"], {"qweight": _t(vw), "qzeros": _t(vz), "scales": _t(vs), "x": _t(x)})
        _close(y.cpu().numpy().reshape(-1, N), O.gemm_f64(x2, w), _budget(x2, w),
               WR_GEMV if x2.shape[0] <= 8 else WR_TC, f"ref WQLinear_GEMV {shape}")
    # GEMVFast module: batch < 8 and one token -> decode kernel, else prefill (gemv_fast.py:185-208)
    for shape in [(1, 1, K), (4, 1, K), (1, 20, K), (9, 1, K)]:
        x = (rng.standard_normal(shape) * 0.5).astype(np.float16)
        x2 = x.reshape(-1, K)
        [(_, y)] = _replay(segs[f"fast {shape}"], {"qweight": _t(fw), "qzeros": _t(fz), "scales": _t(fs), "x": _t(x)})
        assert tuple(y.shape) == shape[:-1] + (N,)
        _close(y.cpu().numpy().reshape(-1, N), O.gemm_f64(x2, wfast), _budget(x2, wfast), WR_GEMV,
               f"ref WQLinear_GEMVFast {shape}")


# ----------------------------------------------------------------------------- fused modules that call awq_ext bare
def test_reference_fastertransformer_rmsnorm(calls):
    segs = _segments(calls, "rmsnorm")
    rng = np.random.default_rng(2)
    for shape in [(1, 1, 4096), (2, 7, 512)]:
        x = rng.standard_normal(shape).astype(np.float16)
        wgt = (1 + 0.1 * rng.standard_normal(shape[-1])).astype(np.float16)
        [(args, _)] = _replay(segs[str(shape)], {"x": _t(x), "weight": _t(wgt)})
        np.testing.assert_allclose(args[2].cpu().numpy(),
                                   O.rmsnorm_f64(x.reshape(-1, shape[-1]), wgt, 1e-5).reshape(shape), rtol=2e-3, atol=2e-3)


@pytest.mark.parametrize("version", ["gemm", "gemv", "gemv_fast"])
def test_reference_fuse_qkv(calls, version):
    """fuse_qkv (fused_utils.py:45-142) concatenates the packed buffers (along the axes it used, as recorded); the fused
    module on our kernels must give [q | k | v] of the separate projections' oracle outputs."""
    K, G = 512, 128
    widths = (512, 128, 128)
    parts, ws = {"qweight": [], "scales": [], "qzeros": []}, []
    for i, N in enumerate(widths):
        c = O.make_case(K, N, G, seed=40 + i)
        if version == "gemm":
            bufs = (c["qweight"], c["scales"], c["qzeros"])
            ws.append(O.dequantize_gemm(c["qweight"], c["qzeros"], c["scales"], G))
        elif version == "gemv":
            vw, vz, vs = O.pack_gemv(c["intweight"], c["zeros"], c["scales"], G)
            bufs = (vw, vs, vz)
            ws.append(O.dequantize_gemm(c["qweight"], c["qzeros"], c["scales"], G))
        else:
            fw, fs, fz = O.pack_gemv_fast(c["intweight"], c["zeros"], c["scales"], G)
            bufs = (fw, fs, fz)
            ws.append(O.dequantize_gemv_fast_f64(fw, fs, fz, G))
        for name, b in zip(("qweight", "scales", "qzeros"), bufs):
            parts[name].append(b)
    axes = calls["fuse_qkv_axes"][version]
    inputs = {name: _t(np.concatenate(ps, axis=axes[name])) for name, ps in parts.items()}
    w = np.concatenate(ws, axis=1)
    x = (np.random.default_rng(5).standard_normal((1, 1, K)) * 0.5).astype(np.float16)
    [(_, y)] = _replay(calls["segments"][f"fuse_qkv_{version}"][0], dict(inputs, x=_t(x)))
    assert y.shape[-1] == sum(widths)
    _close(y.cpu().numpy().reshape(1, -1), O.gemm_f64(x.reshape(1, K), w), _budget(x.reshape(1, K), w), WR_GEMV,
           f"fuse_qkv {version}")


def test_reference_apply_moe_weights(calls):
    """apply_moe_weights (fused/moe.py:45-89): fused_topk -> moe_align_block_size -> grouped_gemm_forward ->
    silu_and_mul -> grouped_gemm_forward(mul_weights) -> sum, all through our awq_ext."""
    E, K, I, G, T, topk = 4, 512, 1024, 128, 3, 2
    rng = np.random.default_rng(6)
    inputs, W1, W2 = {}, [], []
    for tag, cs, store in (("w1", [O.make_case(K, 2 * I, G, seed=60 + e) for e in range(E)], W1),
                           ("w2", [O.make_case(I, K, G, seed=70 + e) for e in range(E)], W2)):
        for b in ("qweight", "qzeros", "scales"):
            inputs[f"{tag}.{b}"] = _t(np.stack([c[b] for c in cs]))
        for c in cs:
            store.append(O.dequantize_gemm(c["qweight"], c["qzeros"], c["scales"], G).astype(np.float64))
    x = (rng.standard_normal((T, K)) * 0.5).astype(np.float16)
    logits = rng.standard_normal((T, E)).astype(np.float32)
    done = _replay(calls["segments"]["moe"][0], dict(inputs, x=_t(x), logits=_t(logits)))
    # our topk_softmax, renormalised as fused_topk does (moe.py:169-170), gives the weights the reference passed on
    tw = done[0][0][0]
    assert torch.allclose(tw / tw.sum(dim=-1, keepdim=True), done[2][0][4], rtol=1e-5, atol=1e-6)
    y = torch.sum(done[-1][1], dim=1).float().cpu().numpy()      # the reference's final reduction (moe.py:89)
    p = np.exp(logits - logits.max(-1, keepdims=True))
    p /= p.sum(-1, keepdims=True)
    ref_y = np.zeros((T, K))
    for t in range(T):
        idx = np.argsort(-p[t], kind="stable")[:topk]
        wts = p[t, idx] / p[t, idx].sum()
        for e, wt in zip(idx, wts):
            gu = (x[t].astype(np.float64) @ W1[e]).astype(np.float16).astype(np.float64)
            act = (gu[:I] / (1 + np.exp(-gu[:I])) * gu[I:]).astype(np.float16).astype(np.float64)
            ref_y[t] += (wt * (act @ W2[e])).astype(np.float16).astype(np.float64)
    tol = 6e-3 * np.abs(ref_y) + 3e-3 * np.sqrt(np.mean(ref_y**2)) + 1e-4
    assert np.all(np.abs(y - ref_y) <= tol), np.abs(y - ref_y).max()


def test_reference_fused_topk_both_branches_agree(calls):
    """The reference itself holds a second definition of `topk_softmax`: on ROCm `fused_topk` computes
    `torch.softmax` + `torch.topk` instead of calling the extension (awq/modules/fused/moe.py:150-153).  That branch's
    routing, recorded from the reference's own function, must equal the extension branch run on OUR
    awq_ext.topk_softmax - which pins the operator to reference code rather than to this repository's reading of it.
    Same for the renormalisation."""
    segs = calls["segments"]["fused_topk"]
    rng = np.random.default_rng(12)
    for seg, want, (T, E, topk) in zip(segs, calls["fused_topk_torch_branch"], [(1, 8, 2), (7, 8, 2), (33, 64, 6),
                                                                              (5, 60, 4)]):
        logits = rng.standard_normal((T, E)).astype(np.float32)
        [(args, _)] = _replay(seg, {"logits": _t(logits)})
        w_ext = args[0] / args[0].sum(dim=-1, keepdim=True)          # renormalize=True (moe.py:169-170)
        w_ref = torch.tensor(want["weights"], dtype=torch.float32, device=_dev())
        id_ref = torch.tensor(want["ids"], dtype=torch.int64, device=_dev())
        assert torch.equal(args[1].long(), id_ref), (T, E, topk)
        assert torch.allclose(w_ext, w_ref, rtol=1e-5, atol=1e-7)


def test_reference_moe_align_block_size_invariants(calls):
    """moe_align_block_size through the reference's wrapper (moe.py:92-134), at sizes beyond its docstring example:
    every expert's run is a multiple of the block, holds exactly that expert's slots in ascending order, padding slots
    carry `numel`, expert_ids name the run's expert."""
    segs = calls["segments"]["moe_align"]
    rng = np.random.default_rng(13)
    for seg, (T, E, topk, block) in zip(segs, [(4, 4, 3, 4), (1, 8, 2, 16), (37, 8, 2, 16), (100, 60, 4, 16)]):
        ids = np.stack([rng.permutation(E)[:topk] for _ in range(T)]).astype(np.int32)
        [(args, _)] = _replay(seg, {"ids": _t(ids)})
        assert args[1:3] == [E, block]
        n = int(args[5].item())
        s_ids, e_ids = args[3].cpu().numpy()[:n], args[4].cpu().numpy()[: n // block]
        assert n % block == 0
        flat = ids.reshape(-1)
        pos = 0
        for e in range(E):
            mine = np.where(flat == e)[0]
            run = (len(mine) + block - 1) // block * block
            assert np.array_equal(s_ids[pos:pos + len(mine)], mine), (T, E, e)
            assert np.all(s_ids[pos + len(mine):pos + run] == flat.size)
            assert np.all(e_ids[pos // block:(pos + run) // block] == e)
            pos += run
        assert pos == n
