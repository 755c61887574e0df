"""Record how the reference package (casper-hansen/AutoAWQ @ 88e4c76) calls the `awq_ext` / `awq_v2_ext` extension
modules, into dropin_calls.json.

    python tests/golden/make_dropin_calls.py <path to an AutoAWQ checkout>

It imports the unmodified reference with recording stand-ins for both extension modules and drives the reference's own
module classes on the CPU: WQLinear_GEMM forward (every dispatch arm) and backward, WQLinear_GEMV, WQLinear_GEMVFast,
FasterTransformerRMSNorm, fuse_qkv, apply_moe_weights, fused_topk and moe_align_block_size.  Each extension call is
stored with its function, its argument order, its scalar arguments, and for every tensor argument its shape, dtype and
origin: a named test input, the result (or an argument written in place) of an earlier call, or a buffer the reference
allocated itself (stored by fill value or, when small, by value).  fused_topk's own torch branch (the one the reference
takes on ROCm) is stored as the expected routing.

tests/test_gpu_reference_dropin.py rebuilds the same seeded inputs, replays the calls on this repository's extension
modules and checks the results against the oracle, so the reference itself is needed only to regenerate this file.
"""
import contextlib
import hashlib
import importlib.machinery
import json
import os
import sys
import types
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import awq_oracle as O  # noqa: E402

warnings.filterwarnings("ignore")


def _dt(t):
    return str(t.dtype).replace("torch.", "")


class Recorder:
    """Stands in for both extension modules: records each call and returns an output of the right shape (values are
    irrelevant to the reference's control flow, except topk_softmax's, which apply_moe_weights renormalises)."""

    def __init__(self):
        self.segments = {}
        self.calls = None

    def begin(self, scenario, label, inputs):
        self.calls, self.inputs, self.outs = [], dict(inputs), []
        self.segments.setdefault(scenario, []).append({"label": label, "calls": self.calls})

    def _origin(self, t):
        ptr = t.untyped_storage().data_ptr()
        for i, j, o in reversed(self.outs):
            if o.untyped_storage().data_ptr() == ptr:
                assert t.storage_offset() == 0 and t.is_contiguous(), "view of an earlier output"
                return {"call": i, "arg": j}
        for name, ref in self.inputs.items():
            if ref.untyped_storage().data_ptr() == ptr:
                assert t.storage_offset() == 0 and t.is_contiguous() and t.numel() == ref.numel(), name
                return {"in": name}
        for name, ref in self.inputs.items():   # a cast of an input (x.to(torch.float16) of a bf16 x)
            if ref.numel() == t.numel() and ref.dtype != t.dtype and torch.equal(ref.reshape(t.shape).to(t.dtype), t):
                return {"in": name}
        flat = t.reshape(-1)
        if t.numel() and bool((flat == flat[0]).all()):
            return {"fill": flat[0].item()}
        if t.numel() <= 4096 and bool(torch.isfinite(t.float()).all()):
            return {"values": flat.tolist()}
        return {"empty": True}

    def record(self, mod, fn, args, ret_shape=None, ret=None):
        desc = []
        for a in args:
            if isinstance(a, torch.Tensor):
                desc.append(dict(self._origin(a), shape=list(a.shape), dtype=_dt(a)))
            else:
                desc.append({"v": a})
        i = len(self.calls)
        for j, a in enumerate(args):
            if isinstance(a, torch.Tensor):
                self.outs.append((i, j, a))
        if ret_shape is not None:
            ret = torch.zeros(ret_shape, dtype=torch.float16)
        if ret is not None:
            self.outs.append((i, "ret", ret))
        self.calls.append({"mod": mod, "fn": fn, "args": desc,
                           "ret": None if ret is None else {"shape": list(ret.shape), "dtype": _dt(ret)}})
        return ret

    def modules(self):
        r = self
        ext, v2 = types.ModuleType("awq_ext"), types.ModuleType("awq_v2_ext")
        ext.gemm_forward_cuda = lambda x, qw, sc, qz, sk: r.record(
            "awq_ext", "gemm_forward_cuda", [x, qw, sc, qz, sk], x.shape[:-1] + (qw.shape[1] * 8,))
        ext.dequantize_weights_cuda = lambda qw, sc, qz, a, b, c, d: r.record(
            "awq_ext", "dequantize_weights_cuda", [qw, sc, qz, a, b, c, d], (qw.shape[0], qw.shape[1] * 8))
        ext.gemv_forward_cuda = lambda x, qw, sc, qz, g: r.record(
            "awq_ext", "gemv_forward_cuda", [x, qw, sc, qz, g], x.shape[:-1] + (qw.shape[0],))
        ext.gemmv2_forward_cuda = lambda x, qw, sc, qz, g, sk: r.record(
            "awq_ext", "gemmv2_forward_cuda", [x, qw, sc, qz, g, sk], x.shape[:-1] + (qw.shape[0],))
        ext.layernorm_forward_cuda = lambda x, w, out, eps: r.record(
            "awq_ext", "layernorm_forward_cuda", [x, w, out, eps])
        ext.silu_and_mul = lambda out, gu: r.record("awq_ext", "silu_and_mul", [out, gu])
        ext.moe_alig_block_size = lambda ids, e, b, s, ei, n: r.record(
            "awq_ext", "moe_alig_block_size", [ids, e, b, s, ei, n])
        ext.grouped_gemm_forward = lambda x, qw, sc, qz, tw, s, e, n, mw, sk: r.record(
            "awq_ext", "grouped_gemm_forward", [x, qw, sc, qz, tw, s, e, n, mw, sk],
            (tw.shape[0], tw.shape[1], qw.shape[2] * 8))

        def topk_softmax(tw, tid, src, logits):
            r.record("awq_ext", "topk_softmax", [tw, tid, src, logits])
            w, i, s = O.topk_softmax(logits.numpy(), tw.shape[1])
            tw.copy_(torch.from_numpy(np.asarray(w, dtype=np.float32)))
            tid.copy_(torch.from_numpy(np.asarray(i, dtype=np.int32)))
            src.copy_(torch.from_numpy(np.asarray(s, dtype=np.int32)))

        ext.topk_softmax = topk_softmax
        v2.gemv_forward_cuda_decode = lambda x, qw, sc, qz, m, n, k, g: r.record(
            "awq_v2_ext", "gemv_forward_cuda_decode", [x, qw, sc, qz, m, n, k, g], x.shape[:-1] + (qw.shape[0] * 4,))
        v2.gemm_forward_cuda_prefill = lambda x, qw, sc, qz: r.record(
            "awq_v2_ext", "gemm_forward_cuda_prefill", [x, qw, sc, qz], x.shape[:-1] + (qw.shape[0] * 4,))
        return ext, v2


def _import_reference(ref_dir, rec):
    import transformers  # noqa: F401  (its availability probes must run before the accelerate stand-in exists)

    def stub(name, **kw):
        m = types.ModuleType(name)
        m.__spec__ = importlib.machinery.ModuleSpec(name, None)
        m.__path__ = []
        m.__dict__.update(kw)
        sys.modules[name] = m
        return m

    # the reference imports accelerate at package import; it is not on any path recorded here
    stub("accelerate", big_modeling=stub("accelerate.big_modeling", init_empty_weights=contextlib.nullcontext,
                                         load_checkpoint_and_dispatch=lambda *a, **k: None))
    stub("accelerate.utils", get_balanced_memory=lambda *a, **k: None)
    sys.modules["awq_ext"], sys.modules["awq_v2_ext"] = rec.modules()
    sys.path.insert(0, ref_dir)
    import awq

    return awq


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def _gemm_module(cls, c, K, N, G, bias=False, **kw):
    m = cls(4, G, K, N, bias, "cpu", **kw)
    m.qweight.copy_(_t(c["qweight"]))
    m.qzeros.copy_(_t(c["qzeros"]))
    m.scales.copy_(_t(c["scales"]))
    return m


def _weights(m):
    return {"qweight": m.qweight, "scales": m.scales, "qzeros": m.qzeros}


def main(ref_dir):
    rec = Recorder()
    _import_reference(ref_dir, rec)
    from awq.modules.fused.moe import apply_moe_weights, fused_topk, moe_align_block_size
    from awq.modules.fused.norm import FasterTransformerRMSNorm
    from awq.modules.linear.gemm import WQLinear_GEMM
    from awq.modules.linear.gemv import WQLinear_GEMV
    from awq.modules.linear.gemv_fast import WQLinear_GEMVFast
    from awq.utils.fused_utils import fuse_qkv

    # WQLinear_GEMM.forward, every dispatch arm (gemm.py:44-84); the inputs are the test's own seeded tensors
    for K, N, G in [(512, 256, 128), (1024, 1792, 128), (4096, 4096, 128), (256, 64, 64)]:
        scen = f"gemm_forward_{K}_{N}_{G}"
        m = _gemm_module(WQLinear_GEMM, O.make_case(K, N, G, seed=K + N), K, N, G, bias=True)
        for shape in [(1, 1, K), (1, 8, K), (1, 40, K), (2, 600, K), (3, K)]:
            x = torch.zeros(shape, dtype=torch.float16)
            rec.begin(scen, str(shape), dict(_weights(m), x=x))
            m(x)
        x = torch.randn(2, 3, K, dtype=torch.bfloat16)
        rec.begin(scen, "bf16 (2, 3, K)", dict(_weights(m), x=x))
        m(x)
        rec.begin(scen, "empty batch", dict(_weights(m), x=torch.zeros(0, 2, K, dtype=torch.float16)))
        m(torch.zeros(0, 2, K, dtype=torch.float16))

    # forward and backward in training mode (WQLinearMMFunction, gemm.py:24-114)
    K, N, G = 512, 256, 128
    m = _gemm_module(WQLinear_GEMM, O.make_case(K, N, G, seed=9), K, N, G, training=True)
    m.training = True
    x = torch.zeros((2, 6, K), dtype=torch.float16, requires_grad=True)
    rec.begin("backward", "forward + backward (2, 6, K)", dict(_weights(m), x=x))
    m(x).backward(torch.zeros((2, 6, N), dtype=torch.float16))

    # the reference packer (gemm.py:171-251), then its forward; the digests pin the packed buffers the test rebuilds
    K, N, G = 256, 128, 64
    rng = np.random.default_rng(0)
    iw, iz, s = O.quantize_rtn((rng.standard_normal((N, K)) * 0.05).astype(np.float32), G)
    lin = torch.nn.Linear(K, N, bias=False).half()
    lin.weight.data = _t(O.dequantize_gemm(*O.pack_gemm(iw, iz), s, G).T)
    m = WQLinear_GEMM.from_linear(lin, 4, G, False, _t(s.astype(np.float16)), _t(iz.astype(np.float16)))
    packed_sha = {b: hashlib.sha256(getattr(m, b).numpy().tobytes()).hexdigest() for b in ("qweight", "scales", "qzeros")}
    x = torch.zeros((1, 5, K), dtype=torch.float16)
    rec.begin("from_linear", "forward (1, 5, K)", dict(_weights(m), x=x))
    m(x)

    # WQLinear_GEMV (gemv.py:160-190) and WQLinear_GEMVFast (gemv_fast.py:185-208)
    for K, N, G in [(512, 128, 128), (4096, 512, 128), (1024, 256, 64)]:
        scen = f"gemv_{K}_{N}_{G}"
        c = O.make_case(K, N, G, seed=K)
        mv = WQLinear_GEMV(4, G, K, N, False, "cpu")
        for buf, a in zip(("qweight", "qzeros", "scales"), O.pack_gemv(c["intweight"], c["zeros"], c["scales"], G)):
            getattr(mv, buf).copy_(_t(a))
        mf = WQLinear_GEMVFast(4, G, K, N, False, "cpu")
        for buf, a in zip(("qweight", "scales", "qzeros"), O.pack_gemv_fast(c["intweight"], c["zeros"], c["scales"], G)):
            getattr(mf, buf).copy_(_t(a))
        for shape in [(1, 1, K), (2, 4, K), (1, 24, K)]:
            x = torch.zeros(shape, dtype=torch.float16)
            rec.begin(scen, f"gemv {shape}", dict(_weights(mv), x=x))
            mv(x)
        for shape in [(1, 1, K), (4, 1, K), (1, 20, K), (9, 1, K)]:
            x = torch.zeros(shape, dtype=torch.float16)
            rec.begin(scen, f"fast {shape}", dict(_weights(mf), x=x))
            mf(x)

    # FasterTransformerRMSNorm (fused/norm.py:19-38)
    for shape in [(1, 1, 4096), (2, 7, 512)]:
        x, w = torch.zeros(shape, dtype=torch.float16), torch.ones(shape[-1], dtype=torch.float16)
        rec.begin("rmsnorm", str(shape), dict(x=x, weight=w))
        FasterTransformerRMSNorm(w, eps=1e-5)(x)

    # fuse_qkv (fused_utils.py:45-142): the fused buffers are concatenations of the three projections' buffers
    fused_axes = {}
    K, G, widths = 512, 128, (512, 128, 128)
    for version in ("gemm", "gemv", "gemv_fast"):
        projs = []
        for i, N in enumerate(widths):
            c = O.make_case(K, N, G, seed=40 + i)
            if version == "gemm":
                m = _gemm_module(WQLinear_GEMM, c, K, N, G)
            elif version == "gemv":
                m = WQLinear_GEMV(4, G, K, N, False, "cpu")
                for buf, a in zip(("qweight", "qzeros", "scales"), O.pack_gemv(c["intweight"], c["zeros"], c["scales"], G)):
                    getattr(m, buf).copy_(_t(a))
            else:
                m = WQLinear_GEMVFast(4, G, K, N, False, "cpu")
                for buf, a in zip(("qweight", "scales", "qzeros"),
                                  O.pack_gemv_fast(c["intweight"], c["zeros"], c["scales"], G)):
                    getattr(m, buf).copy_(_t(a))
            projs.append(m)
        parts = {b: [getattr(p, b).clone() for p in projs] for b in ("qweight", "scales", "qzeros")}
        holder = torch.nn.Module()
        holder.q_proj, holder.k_proj, holder.v_proj = projs
        qkv = fuse_qkv(holder, *projs)
        axes = {}
        for b, ps in parts.items():
            fused = getattr(qkv, b)
            axes[b] = next(ax for ax in (0, 1) if all(p.shape[1 - ax] == fused.shape[1 - ax] for p in ps)
                           and torch.equal(torch.cat(ps, dim=ax), fused))
        fused_axes[version] = axes
        x = torch.zeros((1, 1, K), dtype=torch.float16)
        rec.begin(f"fuse_qkv_{version}", "forward (1, 1, K)", dict(_weights(qkv), x=x))
        qkv(x)

    # apply_moe_weights (fused/moe.py:45-89)
    E, K, I, G, T, topk = 4, 512, 1024, 128, 3, 2

    class W:
        pass

    rng = np.random.default_rng(6)
    w1, w2 = W(), W()
    for dst, cs in ((w1, [O.make_case(K, 2 * I, G, seed=60 + e) for e in range(E)]),
                    (w2, [O.make_case(I, K, G, seed=70 + e) for e in range(E)])):
        for b in ("qweight", "qzeros", "scales"):
            setattr(dst, b, _t(np.stack([c[b] for c in cs])))
    x = _t((rng.standard_normal((T, K)) * 0.5).astype(np.float16))
    logits = _t(rng.standard_normal((T, E)).astype(np.float32))
    rec.begin("moe", "apply_moe_weights", {"x": x, "logits": logits, "w1.qweight": w1.qweight, "w1.scales": w1.scales,
                                           "w1.qzeros": w1.qzeros, "w2.qweight": w2.qweight, "w2.scales": w2.scales,
                                           "w2.qzeros": w2.qzeros})
    apply_moe_weights(w1, w2, x, logits, topk, renormalize=True)

    # fused_topk: the extension branch is recorded; the reference's torch branch (taken on ROCm) is the expectation
    topk_expect = []
    rng = np.random.default_rng(12)
    for (T, E, k) in [(1, 8, 2), (7, 8, 2), (33, 64, 6), (5, 60, 4)]:
        lg = _t(rng.standard_normal((T, E)).astype(np.float32))
        rec.begin("fused_topk", f"T={T} E={E} topk={k}", {"logits": lg})
        fused_topk(lg, k, renormalize=True)
        hip, torch.version.hip = torch.version.hip, "reference-rocm-branch"
        try:
            w_ref, id_ref = fused_topk(lg, k, renormalize=True)
        finally:
            torch.version.hip = hip
        topk_expect.append({"weights": w_ref.tolist(), "ids": id_ref.tolist()})

    # moe_align_block_size (fused/moe.py:92-134)
    rng = np.random.default_rng(13)
    for (T, E, k, block) in [(4, 4, 3, 4), (1, 8, 2, 16), (37, 8, 2, 16), (100, 60, 4, 16)]:
        ids = _t(np.stack([rng.permutation(E)[:k] for _ in range(T)]).astype(np.int32))
        rec.begin("moe_align", f"T={T} E={E} topk={k} block={block}", {"ids": ids})
        moe_align_block_size(ids, block, E)

    out = {"source": "casper-hansen/AutoAWQ @ 88e4c76, awq/ module classes driven on the CPU",
           "segments": rec.segments, "from_linear_sha256": packed_sha, "fuse_qkv_axes": fused_axes, "fused_topk_torch_branch": topk_expect}
    with open(os.path.join(HERE, "dropin_calls.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print("wrote", os.path.join(HERE, "dropin_calls.json"), sum(len(s) for s in rec.segments.values()), "segments")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(os.path.abspath(sys.argv[1]))
