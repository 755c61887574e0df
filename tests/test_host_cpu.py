"""CPU-only checks of the host side: packed-format producers vs the reference's outputs, the C oracle vs
the numpy oracle, the torch timing port, and that libb200awq.so loads and exports the whole C ABI."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import awq_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint16)


@pytest.fixture(scope="module")
def built():
    import __graft_entry__ as g

    g.build()
    return True


# ------------------------------------------------------------------------------------ packers
@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_packers_match_reference_from_linear(golden_dir, tag, built):
    from autoawq_b200 import packing as P

    g = np.load(os.path.join(golden_dir, "packers.npz"))
    K, N, G = (int(v) for v in g[f"{tag}_meta"])
    w = torch.from_numpy(g[f"{tag}_weight"])
    s = torch.from_numpy(g[f"{tag}_scales_ng"]).float()
    z = torch.from_numpy(g[f"{tag}_zeros_ng"]).float()
    iw = P.quantize_to_int(w, s, z, G)
    assert int(iw.min()) >= 0 and int(iw.max()) <= 15
    qw, qz, sc = P.pack_gemm(iw, z, s)
    assert np.array_equal(qw.numpy(), g[f"{tag}_gemm_qweight"])
    assert np.array_equal(qz.numpy(), g[f"{tag}_gemm_qzeros"])
    assert np.array_equal(_bits(sc.numpy()), _bits(g[f"{tag}_gemm_scales"]))
    vw, vz, vs = P.pack_gemv(iw, z, s, G)
    assert np.array_equal(vw.numpy(), g[f"{tag}_gemv_qweight"])
    assert np.array_equal(vz.numpy(), g[f"{tag}_gemv_qzeros"])
    assert np.array_equal(_bits(vs.numpy()), _bits(g[f"{tag}_gemv_scales"]))
    if f"{tag}_fast_qweight" in g:
        fw, fs, fz = P.pack_gemv_fast(iw, z, s, G)
        assert np.array_equal(fw.numpy(), g[f"{tag}_fast_qweight"])
        assert np.array_equal(_bits(fs.numpy()), _bits(g[f"{tag}_fast_scales"]))
        assert np.array_equal(_bits(fz.numpy()), _bits(g[f"{tag}_fast_qzeros"]))
    assert np.array_equal(P.unpack_gemm_words(qw).numpy(), iw.t().numpy().astype(np.uint8))


def test_zeros_width(golden_dir, built):
    from autoawq_b200.packing import calculate_zeros_width

    g = np.load(os.path.join(golden_dir, "packers.npz"))
    for (k, gs), zw in zip(g["zw_in"], g["zw_out"]):
        assert calculate_zeros_width(int(k), int(gs)) == int(zw)


def test_module_mirrors_have_reference_buffers(built):
    """Buffer names / shapes / dtypes are the checkpoint contract (gemm.py:135-169, gemv.py:45-74,
    gemv_fast.py:86-125)."""
    from autoawq_b200.linear import WQLinear_GEMM, WQLinear_GEMV, WQLinear_GEMVFast

    m = WQLinear_GEMM(4, 128, 4096, 1792, True, "cpu")
    assert m.qweight.shape == (4096, 224) and m.qweight.dtype == torch.int32
    assert m.qzeros.shape == (32, 224) and m.scales.shape == (32, 1792) and m.bias.shape == (1792,)
    assert set(dict(m.named_buffers())) == {"qweight", "qzeros", "scales", "bias"}
    v = WQLinear_GEMV(4, 128, 14336, 4096, False, "cpu")
    assert v.qweight.shape == (4096, 1792) and v.qzeros.shape == (4096, 14) and v.scales.shape == (4096, 112)
    assert v.split_k_iters == 8 and v.bias is None
    f = WQLinear_GEMVFast(4, 128, 4096, 4096, False, "cpu")
    assert f.qweight.shape == (1024, 4096) and f.qweight.dtype == torch.int16
    assert f.scales.shape == (32, 4096) and f.qzeros.dtype == torch.float16
    with pytest.raises(NotImplementedError):
        WQLinear_GEMM(8, 128, 256, 256, False, "cpu")
    with pytest.raises(AssertionError):
        WQLinear_GEMM(4, 128, 200, 256, False, "cpu")
    m2 = WQLinear_GEMM(4, -1, 256, 64, False, "cpu")
    assert m2.group_size == 256 and m2.qzeros.shape == (1, 8)


def test_no_cpu_fallback(built):
    """The product path refuses CPU tensors instead of silently computing on the host."""
    from autoawq_b200 import ext
    from autoawq_b200.linear import WQLinear_GEMM

    m = WQLinear_GEMM(4, 128, 256, 64, False, "cpu")
    with pytest.raises(ext.B200AwqError):
        m(torch.zeros(1, 1, 256, dtype=torch.float16))
    with pytest.raises(ext.B200AwqError):
        ext.dequantize_weights_cuda(m.qweight, m.scales, m.qzeros, 0, 0, 0, False)


def test_product_does_not_import_oracle():
    for pkg in ("autoawq_b200", "awq_ext", "awq_v2_ext"):
        for dp, _, files in os.walk(os.path.join(ROOT, pkg)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    src = open(os.path.join(dp, f)).read()
                    assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{pkg}/{f} imports the oracle"
                    if f != "build.py":  # build.py compiles the checker (building it is not using it)
                        assert "awq_oracle" not in src and "libawqoracle" not in src, f"{pkg}/{f} uses the oracle"


# ---------------------------------------------------------------------------------- C ABI
def test_cabi_exports_every_declared_symbol(built):
    from autoawq_b200 import _cabi

    header = open(os.path.join(ROOT, "include", "b200awq.h")).read()
    declared = set(re.findall(r"\b(b200awq_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    lib = ctypes.CDLL(_cabi.lib_path())
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/b200awq.h but not exported"
    assert declared == set(_cabi.SIGNATURES), "ctypes table and header disagree"
    assert _cabi.lib.b200awq_abi_version() == 1
    assert _cabi.lib.b200awq_error_string(3).decode().startswith("workspace")
    assert _cabi.lib.b200awq_workspace_bytes(1, 4096, 4096) == 16384 + 4096 * 8   # tickets + one 64-bit word per element
    assert _cabi.lib.b200awq_workspace_bytes(4096, 4096, 4096) == 16384 + 128 * 4096 * 8


def test_cabi_argument_validation_without_gpu(built):
    """Shape / pointer validation happens before any CUDA call, so it is checkable on the CPU box."""
    from autoawq_b200._cabi import lib

    assert lib.b200awq_gemm_forward(None, 4096, None, None, None, None, None, 1, 4096, 4096, 128, None, 0, None) == 1
    assert lib.b200awq_gemm_forward(None, 4096, None, None, None, None, None, 1, 4096, 4095, 128, None, 0, None) == 1
    assert lib.b200awq_gemm_forward(None, 4096, None, None, None, None, None, 1, 4096, 4096, 100, None, 0, None) == 1
    assert lib.b200awq_gemm_forward(None, 4096, None, None, None, None, None, 0, 4096, 4096, 128, None, 0, None) == 0
    assert lib.b200awq_dequantize_gemm(None, None, None, None, 128, 64, 128, None) == 1
    assert lib.b200awq_set_knob(99, 1) == 1 and lib.b200awq_get_knob(2) == 8
    for retired in (7, 8, 9, 10, 11, 13, 17, 18, 20, 22):   # variants removed: a stale setting must fail loudly
        assert lib.b200awq_set_knob(retired, 1) == 1 and lib.b200awq_get_knob(retired) == 0, retired
    assert lib.b200awq_set_knob(12, 2) == 0 and lib.b200awq_get_knob(12) == 2
    assert lib.b200awq_set_knob(12, 0) == 0


# ------------------------------------------------------------------------------- C oracle
def test_c_oracle_matches_numpy_oracle(built):
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_build", "libawqoracle.so"))
    for (K, N, G, raw) in [(256, 64, 128, False), (128, 40, 32, True), (384, 72, 128, True)]:
        c = O.make_case(K, N, G, seed=9, raw=raw)
        out = np.empty((K, N), dtype=np.uint16)
        lib.oracle_dequantize_gemm(
            c["qweight"].ctypes.data_as(ctypes.c_void_p), c["qzeros"].ctypes.data_as(ctypes.c_void_p),
            c["scales"].ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p), K, N, G)
        w = O.dequantize_gemm(c["qweight"], c["qzeros"], c["scales"], G)
        assert np.array_equal(out, _bits(w))
        x = np.random.default_rng(0).standard_normal((3, K)).astype(np.float16)
        y = np.empty((3, N), dtype=np.float64)
        lib.oracle_gemm_f64(x.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p),
                            y.ctypes.data_as(ctypes.c_void_p), 3, K, N)
        np.testing.assert_allclose(y, O.gemm_f64(x, w), rtol=1e-12, atol=1e-12)


def test_torch_port_matches_oracle():
    from oracle import ref_cpu_path as R

    c = O.make_case(256, 64, 64, seed=4, raw=True)
    w = R.dequantize(torch.from_numpy(c["qweight"]), torch.from_numpy(c["qzeros"]), torch.from_numpy(c["scales"]), 64)
    assert w.dtype == torch.float16
    assert np.array_equal(_bits(w.numpy()), _bits(O.dequantize_gemm(c["qweight"], c["qzeros"], c["scales"], 64)))


def test_program_op_struct_matches_header(built, tmp_path):
    """ctypes mirror of b200awq_op_t vs the C compiler's view of include/b200awq.h (size + every offset)."""
    import subprocess

    from autoawq_b200 import _cabi

    fields = [f[0] for f in _cabi.Op._fields_]
    src = tmp_path / "layout.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "b200awq.h"\nint main(void) {\n'
        '  printf("%zu", sizeof(b200awq_op_t));\n'
        + "".join(f'  printf(" %zu", offsetof(b200awq_op_t, {f}));\n' for f in fields)
        + "  return 0;\n}\n"
    )
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).decode().split()]
    assert got[0] == ctypes.sizeof(_cabi.Op)
    assert got[1:] == [getattr(_cabi.Op, f).offset for f in fields]
    header = open(os.path.join(ROOT, "include", "b200awq.h")).read()
    assert (_cabi.OP_RMSNORM, _cabi.OP_LINEAR_GEMM, _cabi.OP_SILU_AND_MUL) == tuple(
        int(re.search(rf"{n}\s*=\s*(\d+)", header).group(1))
        for n in ("B200AWQ_OP_RMSNORM", "B200AWQ_OP_LINEAR_GEMM", "B200AWQ_OP_SILU_AND_MUL"))


def test_program_argument_validation_without_gpu(built):
    from autoawq_b200 import _cabi

    h = ctypes.c_void_p()
    assert _cabi.lib.b200awq_program_create(None, 0, ctypes.byref(h)) == 1
    assert _cabi.lib.b200awq_program_create(None, 3, None) == 1
    assert _cabi.lib.b200awq_program_run(None, None, 0, None) == 1
    assert _cabi.lib.b200awq_program_num_ops(None) == 0
    assert _cabi.lib.b200awq_program_destroy(None) == 0
    ops = (_cabi.Op * 1)()
    ops[0].kind = 77
    assert _cabi.lib.b200awq_program_create(ops, 1, ctypes.byref(h)) == 1 and not h.value


def test_moe_argument_validation_without_gpu(built):
    from autoawq_b200._cabi import lib

    assert lib.b200awq_topk_softmax(None, None, None, None, 4, 8, 9, None) == 1       # topk > E
    assert lib.b200awq_topk_softmax(None, None, None, None, 0, 8, 2, None) == 0       # nothing to do
    assert lib.b200awq_topk_softmax(None, None, None, None, 4, 8, 2, None) == 1       # null pointers
    assert lib.b200awq_moe_align_block_size(None, 8, 8, 16, None, None, None, None) == 1
    p8 = (None,) * 8   # qweight, scales, qzeros, topk_weights, sorted_ids, expert_ids, num_post_pad, y
    tail = (None, 0, None)   # workspace, workspace_bytes, stream
    assert lib.b200awq_grouped_gemm_forward(None, 1, *p8, 0, 2, 0, 8, 4096, 4096, 128, 0, 16, *tail) == 0   # T == 0
    assert lib.b200awq_grouped_gemm_forward(None, 1, *p8, 1, 2, 32, 8, 4096, 4095, 128, 0, 16, *tail) == 1  # N % 8 != 0
    assert lib.b200awq_grouped_gemm_forward(None, 3, *p8, 1, 2, 32, 8, 4096, 4096, 128, 0, 16, *tail) == 1  # rows/token
    assert lib.b200awq_grouped_gemm_forward(None, 1, *p8, 1, 2, 32, 8, 4096, 4096, 128, 0, 16, *tail) == 1  # null pointers


def test_c_oracle_moe_routing_matches_numpy_oracle(built):
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_build", "libawqoracle.so"))
    rng = np.random.default_rng(3)
    for T, topk, E, block in [(4, 3, 5, 4), (1, 2, 8, 16), (50, 2, 8, 16), (9, 4, 16, 8)]:
        ids = np.stack([rng.permutation(E)[:topk] for _ in range(T)]).astype(np.int32)
        numel = ids.size
        s = np.empty(numel + E * (block - 1), dtype=np.int32)
        e = np.empty(numel + E, dtype=np.int32)
        n = lib.oracle_moe_align_block_size(ids.ctypes.data_as(ctypes.c_void_p), numel, E, block,
                                            s.ctypes.data_as(ctypes.c_void_p), e.ctypes.data_as(ctypes.c_void_p))
        rs, re_, rn = O.moe_align_block_size(ids, block, E)
        assert n == rn and np.array_equal(s, rs) and np.array_equal(e, re_)
        g = (rng.standard_normal((T, E)) * 2).astype(np.float32)
        w = np.empty((T, topk), dtype=np.float32)
        i = np.empty((T, topk), dtype=np.int32)
        lib.oracle_topk_softmax(g.ctypes.data_as(ctypes.c_void_p), T, E, topk, w.ctypes.data_as(ctypes.c_void_p),
                                i.ctypes.data_as(ctypes.c_void_p))
        rw, ri, _ = O.topk_softmax(g, topk)
        assert np.array_equal(i, ri)
        np.testing.assert_allclose(w, rw, rtol=1e-6, atol=1e-8)


def test_decode_program_recorder_refuses_cpu_tensors(built):
    """No CPU path anywhere: the recorder raises on CPU tensors like the operators do."""
    import torch

    from autoawq_b200.program import DecodeProgram
    from autoawq_b200.ext import B200AwqError

    p = DecodeProgram()
    x = torch.zeros((1, 64), dtype=torch.float16)
    with pytest.raises(B200AwqError):
        p.layernorm_forward_cuda(x, torch.ones(64, dtype=torch.float16), torch.empty_like(x), 1e-5)
    with pytest.raises(B200AwqError):
        p.gemm_forward_cuda(x, torch.zeros((64, 8), dtype=torch.int32), torch.zeros((1, 64), dtype=torch.float16),
                            torch.zeros((1, 8), dtype=torch.int32), 8)
    with pytest.raises(B200AwqError):
        p.build()          # empty program
    with pytest.raises(B200AwqError):
        p.run()            # not built


def test_python_workspace_size_restates_the_abi(built):
    """ext.linear_forward sizes the split-K workspace without an extra ABI call; the restated formula must agree
    with b200awq_workspace_bytes for every M."""
    from autoawq_b200 import ext
    from autoawq_b200._cabi import lib

    for M in (1, 8, 63, 64, 65, 127, 128, 129, 256, 4096):
        for N in (8, 4096, 28672):
            assert lib.b200awq_workspace_bytes(M, 4096, N) == ext._WS_TICKETS + min(M, 128) * N * 8


def test_comm_and_stream_argument_validation_without_gpu(built):
    """The round-2 entry points reject bad arguments before touching a device."""
    import ctypes

    from autoawq_b200._cabi import lib

    h = ctypes.c_void_p()
    assert lib.b200awq_comm_create(0, 9, 8192, ctypes.byref(h)) == 1       # world > 8
    assert lib.b200awq_comm_create(2, 2, 8192, ctypes.byref(h)) == 1       # rank out of range
    assert lib.b200awq_comm_create(0, 2, 100, ctypes.byref(h)) == 1        # max_elems % 8
    assert lib.b200awq_comm_all_reduce(None, None, 8, None) == 1
    assert lib.b200awq_stream_bytes(4096, 4096, 128) == (4096 // 16) * (4096 // 128) * 1072
    assert lib.b200awq_stream_bytes(4096, 4100, 128) == 0                  # N % 16
    assert lib.b200awq_stream_bytes(4000, 4096, 32) == 0                   # K % 128
    assert lib.b200awq_stream_pack(None, None, None, None, 4096, 4096, 128, 0, None) == 1
    assert lib.b200awq_program_kind(None) == 0
