"""GPU tests of the fp16 pair-table mode (sqllm_set_lut_mode / quant_cuda.set_lut_mode("fp16")) - north_star's "per-channel fp16 LUT".

What the mode changes, and therefore what is checked:
  (1) the kernel must compute EXACTLY what it claims: the same sum with every centroid rounded to fp16 (round-to-nearest-even) and
      fp32 accumulation.  Checked against the fp64 oracle run on the fp16-rounded codebook, with the strict per-element metric of
      tests/util.py (TIGHT_TOL = 5e-5) - through the C ABI with fp16 x and fp32 y, so that no output rounding blurs it.
  (2) against the exact (fp32 codebook) result the only difference is that rounding: <= 2^-11 relative per weight.  In the max norm,
      max_i |y_i - y_ref_i| / max_i |y_ref_i| <= 1e-3 (north_star's tolerance; measured ~2.5e-4 on 4096-wide layers).  The strict
      per-element metric with its 1 % floor reads ~1.5e-2 on outputs that cancel to ~0 - 16-bit table entries cannot do better -
      which is why the exact table stays the default and this mode is opt-in.  Both numbers are asserted here.
"""
import ctypes

import numpy as np
import pytest
import torch

from util import Args, REL_TOL, TIGHT_TOL, load_lib, orc, rel_err, to_torch

pytestmark = pytest.mark.gpu

SHAPES = [  # (bits, K, N, sparsity, topX, nonzero_full_rows, skew)
    (4, 128, 128, 0.0, 0, False, False),
    (3, 128, 128, 0.0, 0, False, False),
    (4, 512, 132, 0.01, 10, True, False),       # ragged last strip
    (3, 192, 68, 0.01, 3, True, True),
    (4, 4096, 4096, 0.0, 0, False, False),
    (4, 4096, 4096, 0.0045, 10, True, False),
    (3, 4096, 4096, 0.0045, 10, True, True),
    (4, 4096, 11008, 0.0045, 10, False, False),
    (4, 11008, 4096, 0.0045, 10, False, False),
    (3, 11008, 4096, 0.0045, 0, False, True),
    (4, 4096, 22016, 0.0045, 10, False, False),
    (4, 5120, 13824, 0.0005, 10, False, False),
    (3, 8192, 22016, 0.0045, 10, False, False),
    (3, 22016, 8192, 0.0045, 10, False, False),
    (3, 8192, 2752, 0.0045, 10, False, False),
    (4, 4096, 4096, 0.0045, 64, True, False),   # > 32 dense rows: the finisher's general dense-row path
    (3, 512, 132, 0.01, 128, True, False),      # MAX_TOPX_FUSED dense rows on a ragged 3-strip layer
]
IDS = [f"w{b}-{k}x{n}-s{int(s*1e4)}-t{t}" for b, k, n, s, t, z, sk in SHAPES]
NORM_TOL = REL_TOL       # max-norm relative error against the exact-codebook result
STRICT_CEIL = 5e-2       # per-element metric (1 % floor) against the exact-codebook result: documented ceiling, see module docstring


def max_norm_err(a, b):
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


@pytest.fixture(scope="module")
def lib():
    lib = load_lib()
    yield lib
    lib.sqllm_set_lut_mode(0)


def _fused_abi(lib, T, x_half, N, y_half=False, bias=None):
    a = Args(bits=T["bits"], in_features=T["infeatures"], out_features=T["outfeatures"], batch=1,
             qweight=T["qweight"].data_ptr(), lookup_table=T["lookup_table"].data_ptr())
    if T["rows"] is not None:
        a.rows, a.cols, a.vals = T["rows"].data_ptr(), T["cols"].data_ptr(), T["vals"].data_ptr()
    if T["full_rows"] is not None:
        a.full_rows, a.full_row_indices, a.topX = T["full_rows"].data_ptr(), T["full_row_indices"].data_ptr(), T["full_rows"].shape[1]
    nbytes = lib.sqllm_workspace_bytes(T["bits"], T["infeatures"], T["outfeatures"], a.topX)
    assert nbytes > 0
    ws = torch.zeros(nbytes, dtype=torch.uint8, device="cuda")
    y = torch.empty(N, dtype=torch.float16 if y_half else torch.float32, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.sqllm_lutgemv_fused(ctypes.byref(a), ctypes.c_void_p(x_half.data_ptr()), 1, ctypes.c_void_p(y.data_ptr()), int(y_half),
                                 ctypes.c_void_p(bias.data_ptr() if bias is not None else 0), ctypes.c_void_p(ws.data_ptr()),
                                 ctypes.c_size_t(nbytes), st)
    assert rc == 0, lib.sqllm_last_error()
    torch.cuda.synchronize()
    assert lib.sqllm_workspace_error(ctypes.c_void_p(ws.data_ptr()), st) == 0
    return y


@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_fp16_pair_mode_is_the_fp16_rounded_codebook_exactly(lib, shape):
    bits, K, N, sp, topx, nz, skew = shape
    L = orc.make_layer(bits, K, N, sparsity=sp, topX=topx, seed=K + 3 * N + bits, skew=skew, nonzero_full_rows=nz, bias=True)
    if topx and sp == 0:
        L["full_rows"] = L["full_row_indices"] = None
    x = orc.make_vec(K, seed=11)  # fp16-representable
    T = to_torch(L)
    xh = torch.from_numpy(x).cuda().reshape(-1).half()
    lib.sqllm_set_lut_mode(1)
    try:
        assert lib.sqllm_get_lut_mode() == 1
        y = _fused_abi(lib, T, xh, N, bias=T["bias"]).cpu().numpy()
    finally:
        lib.sqllm_set_lut_mode(0)
    y_exact_mode = _fused_abi(lib, T, xh, N, bias=T["bias"]).cpu().numpy()
    L16 = dict(L)
    L16["lookup_table"] = L["lookup_table"].astype(np.float16).astype(np.float32)
    want16 = orc.forward_f64(L16, x, mul_init=L["bias"][None, :])
    want = orc.forward_f64(L, x, mul_init=L["bias"][None, :])
    assert rel_err(y, want16) < TIGHT_TOL, "the fp16 mode must equal the fp16-rounded codebook result up to fp32 summation order"
    assert rel_err(y_exact_mode, want) < TIGHT_TOL, "switching back restores the exact table"
    assert max_norm_err(y, want) < NORM_TOL
    assert rel_err(y, want) < STRICT_CEIL


def test_fp16_mode_through_the_module_and_fp32_x_keeps_exact(lib):
    from squeezellm_b200.quant import quant_cuda as qc
    K, N = 4096, 4096
    L = orc.make_layer(4, K, N, sparsity=0.0045, topX=10, seed=5, nonzero_full_rows=True)
    T = to_torch(L)
    x = orc.make_vec(K, seed=6)
    args = (T["qweight"], T["lookup_table"], 4, None, T["rows"], T["cols"], T["vals"], T["full_rows"], T["full_row_indices"])
    want = orc.forward_f64(L, x)
    qc.set_lut_mode("fp16")
    try:
        assert qc.get_lut_mode() == "fp16"
        yh = qc.lutgemv_fused(torch.from_numpy(x).cuda().reshape(-1).half(), *args)
        yf = qc.lutgemv_fused(torch.from_numpy(x).cuda().reshape(-1), *args)   # fp32 x: exact table, whatever the mode
        torch.cuda.synchronize()
    finally:
        qc.set_lut_mode("exact")
    assert qc.get_lut_mode() == "exact"
    assert yh.dtype == torch.float16 and max_norm_err(yh.float().cpu().numpy(), want) < NORM_TOL
    assert rel_err(yf.cpu().numpy(), want) < TIGHT_TOL
    assert not qc.workspace_error()
    with pytest.raises(RuntimeError):
        qc.set_lut_mode("bf16")
