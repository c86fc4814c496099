"""Shared helpers for the test-suite (oracle access, tolerances, ctypes view of the C ABI)."""
import ctypes
import glob
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import oracle as orc  # noqa: E402  (tests are allowed to use the oracle)

GOLDEN = os.path.join(ROOT, "tests", "golden")
LIB = os.path.join(ROOT, "squeezellm_b200", "libsqllm_b200.so")
HEADER = os.path.join(ROOT, "include", "sqllm_b200.h")

# north_star: outputs match the reference to <= 1e-3 max relative error.  Relative error needs an absolute
# floor for outputs that cancel to ~0 (SURVEY.md 8(c)); defined once, here:
#     err = max_i |a_i - b_i| / max(|b_i|, FLOOR * max_j |b_j|)
REL_TOL = 1e-3
FLOOR = 1e-2
# our kernels accumulate in fp32 with a fixed order; against the fp64 truth they must be far inside REL_TOL
TIGHT_TOL = 5e-5


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64).ravel()
    b = np.asarray(b, dtype=np.float64).ravel()
    assert a.shape == b.shape
    den = np.maximum(np.abs(b), FLOOR * max(np.abs(b).max(), 1e-30))
    return float((np.abs(a - b) / den).max())


def golden_files(prefix):
    return sorted(glob.glob(os.path.join(GOLDEN, prefix + "*.npz")))


def buffer_signature(t):
    """'int32[16, 128]': dtype and shape of a state_dict tensor, as tests/golden/reference_quant_api.json records them."""
    return f"{str(t.dtype).replace('torch.', '')}{list(t.shape)}"


def header_symbols():
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(sqllm_\w+)\s*\(", txt)))


def load_lib():
    lib = ctypes.CDLL(LIB)
    lib.sqllm_last_error.restype = ctypes.c_char_p
    lib.sqllm_workspace_bytes.restype = ctypes.c_size_t
    return lib


class Args(ctypes.Structure):  # mirrors sqllm_lutgemv_args
    _fields_ = [("bits", ctypes.c_int), ("in_features", ctypes.c_int), ("out_features", ctypes.c_int),
                ("batch", ctypes.c_int), ("qweight", ctypes.c_void_p), ("lookup_table", ctypes.c_void_p),
                ("vec", ctypes.c_void_p), ("mul", ctypes.c_void_p), ("rows", ctypes.c_void_p),
                ("cols", ctypes.c_void_p), ("vals", ctypes.c_void_p), ("full_rows", ctypes.c_void_p),
                ("full_row_indices", ctypes.c_void_p), ("topX", ctypes.c_int)]


def to_torch(layer, device="cuda"):
    """numpy layer dict (oracle.make_layer) -> dict of torch tensors on `device`."""
    import torch
    out = {}
    for k, v in layer.items():
        out[k] = torch.from_numpy(v).to(device) if isinstance(v, np.ndarray) else v
    return out


def abi_call(lib, T, x, mul, batch=1):
    """sqllm_lutgemv (accumulate into mul) on the current stream for the torch layer T (to_torch)."""
    import torch
    a = Args(bits=T["bits"], in_features=T["infeatures"], out_features=T["outfeatures"], batch=batch,
             qweight=T["qweight"].data_ptr(), lookup_table=T["lookup_table"].data_ptr(), vec=x.data_ptr(), mul=mul.data_ptr())
    if T["rows"] is not None:
        a.rows, a.cols, a.vals = T["rows"].data_ptr(), T["cols"].data_ptr(), T["vals"].data_ptr()
    if T["full_rows"] is not None:
        a.full_rows, a.full_row_indices, a.topX = T["full_rows"].data_ptr(), T["full_row_indices"].data_ptr(), T["full_rows"].shape[1]
    rc = lib.sqllm_lutgemv(ctypes.byref(a), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.sqllm_last_error()


def module_call(mod, T, x, mul, batched):
    """The way squeezellm/quant.py:225-309 / :323-379 picks one of the 12 symbols."""
    b, sfx = T["bits"], "_batched" if batched else ""
    if T["rows"] is not None and T["full_rows"] is not None:
        getattr(mod, f"vecquant{b}matmul_spmv_hybrid_nuq_perchannel{sfx}")(
            T["rows"], T["cols"], T["vals"], x, T["full_rows"], T["full_row_indices"], mul, T["outfeatures"], T["qweight"], T["lookup_table"])
    elif T["rows"] is not None:
        getattr(mod, f"vecquant{b}matmul_spmv_nuq_perchannel{sfx}")(
            T["rows"], T["cols"], T["vals"], x, mul, T["outfeatures"], T["qweight"], T["lookup_table"])
    else:
        getattr(mod, f"vecquant{b}matmul_nuq_perchannel{sfx}")(x, T["qweight"], mul, T["lookup_table"])


def oracle_chain(layers, dims, x, lut_fp16=False):
    """fp64 truth of a chain of matvecs, dims = [(K, N, x_offset into the previous output), ...]; the hand-over between two
    matvecs is rounded to fp16, as in the model (and in the sequence kernel)."""
    outs, prev = [], None
    for L, (K, N, off) in zip(layers, dims):
        xin = x if prev is None else prev[off:off + K]
        LL = dict(L)
        if lut_fp16:
            LL["lookup_table"] = L["lookup_table"].astype(np.float16).astype(np.float32)
        y = orc.forward_f64(LL, xin.astype(np.float32).reshape(1, K)).reshape(N)
        prev = y.astype(np.float16).astype(np.float64)
        outs.append(prev)
    return outs
