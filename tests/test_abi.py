"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every symbol include/sqllm_b200.h
declares, argument validation answers without touching a GPU, and the `quant_cuda` module carries the
reference's 12 names (squeezellm/quant_cuda.cpp:258-269)."""
import ctypes
import os

import pytest

from util import GOLDEN, Args, buffer_signature, header_symbols, load_lib

REFERENCE_SYMBOLS = [
    "vecquant3matmul_nuq_perchannel", "vecquant4matmul_nuq_perchannel",
    "vecquant3matmul_nuq_perchannel_batched", "vecquant4matmul_nuq_perchannel_batched",
    "vecquant3matmul_spmv_nuq_perchannel", "vecquant4matmul_spmv_nuq_perchannel",
    "vecquant3matmul_spmv_nuq_perchannel_batched", "vecquant4matmul_spmv_nuq_perchannel_batched",
    "vecquant3matmul_spmv_hybrid_nuq_perchannel", "vecquant4matmul_spmv_hybrid_nuq_perchannel",
    "vecquant3matmul_spmv_hybrid_nuq_perchannel_batched", "vecquant4matmul_spmv_hybrid_nuq_perchannel_batched",
]


def test_library_exports_every_declared_symbol():
    lib = load_lib()
    syms = header_symbols()
    assert len(syms) >= 12 + 6
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/sqllm_b200.h but not exported"
    for s in REFERENCE_SYMBOLS:
        assert "sqllm_" + s in syms


def test_abi_version_and_error_string():
    lib = load_lib()
    assert lib.sqllm_abi_version() == 4
    assert isinstance(lib.sqllm_last_error(), bytes)


@pytest.mark.parametrize("field,value,frag", [("bits", 5, b"bits"), ("in_features", 100, b"in_features"),
                                              ("out_features", 6, b"out_features")])
def test_argument_validation_without_gpu(field, value, frag):
    lib = load_lib()
    a = Args(bits=4, in_features=128, out_features=128, batch=1, qweight=16, lookup_table=16, vec=16, mul=16)
    setattr(a, field, value)
    rc = lib.sqllm_lutgemv(ctypes.byref(a), None)
    assert rc == -1  # SQLLM_EINVAL
    assert frag in lib.sqllm_last_error()


def test_null_and_misaligned_pointers_rejected():
    lib = load_lib()
    a = Args(bits=4, in_features=128, out_features=128, batch=1, qweight=0, lookup_table=16, vec=16, mul=16)
    assert lib.sqllm_lutgemv(ctypes.byref(a), None) == -1
    a.qweight = 20  # not 16-byte aligned
    assert lib.sqllm_lutgemv(ctypes.byref(a), None) == -1
    assert b"aligned" in lib.sqllm_last_error()
    assert lib.sqllm_lutgemv(None, None) == -1


def test_reference_launcher_shape_checks():
    lib = load_lib()
    # height must be a multiple of bits (height = in/32*bits)
    assert lib.sqllm_vecquant3matmul_nuq_perchannel(16, 16, 16, 16, 13, 128, None) == -1
    # batched: vec_height must equal the in_features implied by the packed matrix
    assert lib.sqllm_vecquant4matmul_nuq_perchannel_batched(16, 16, 16, 16, 16, 128, 2, 64, None) == -1
    assert b"features" in lib.sqllm_last_error()


def test_quant_cuda_module_has_the_reference_names():
    from squeezellm_b200.quant import quant_cuda
    for s in REFERENCE_SYMBOLS:
        assert callable(getattr(quant_cuda, s))
    assert not any("balanced" in n for n in dir(quant_cuda))  # absent in the reference build too
    assert quant_cuda.abi_version() == 4


def test_quant_cuda_rejects_cpu_tensors_loudly():
    """No CPU fallback: calling the extension with host tensors raises instead of computing something."""
    import torch
    from squeezellm_b200.quant import quant_cuda
    x = torch.zeros(128); q = torch.zeros((16, 128), dtype=torch.int32); y = torch.zeros(128); lut = torch.zeros((128, 16))
    with pytest.raises(RuntimeError, match="CUDA"):
        quant_cuda.vecquant4matmul_nuq_perchannel(x, q, y, lut)
    with pytest.raises(RuntimeError):
        quant_cuda.lutgemv_fused(x, q, lut, 4)


class Exchange(ctypes.Structure):  # mirrors sqllm_exchange
    _fields_ = [("world", ctypes.c_int), ("rank", ctypes.c_int), ("members", ctypes.c_int), ("out_features_full", ctypes.c_int),
                ("peer_base", ctypes.c_void_p), ("out_offset", ctypes.c_size_t), ("flag_offset", ctypes.c_size_t),
                ("state_offset", ctypes.c_size_t), ("error_offset", ctypes.c_size_t)]


@pytest.mark.parametrize("change,frag", [(dict(rank=2), b"rank"), (dict(members=3), b"members"), (dict(out_features_full=64), b"out_features_full"),
                                         (dict(peer_base=0), b"peer_base"), (dict(out_offset=4100), b"misaligned"), (dict(flag_offset=4), b"misaligned")])
def test_exchange_descriptor_validation_without_gpu(change, frag):
    """sqllm_lutgemv_fused_exchange rejects inconsistent descriptors before it touches the device."""
    lib = load_lib()
    lib.sqllm_lutgemv_fused_exchange.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                                 ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]
    a = Args(bits=4, in_features=128, out_features=128, batch=1, qweight=16, lookup_table=16)
    x = Exchange(world=2, rank=0, members=2, out_features_full=128, peer_base=16, out_offset=4096, flag_offset=0, state_offset=64, error_offset=128)
    for k, v in change.items():
        setattr(x, k, v)
    rc = lib.sqllm_lutgemv_fused_exchange(ctypes.byref(a), 16, 1, 1, None, 16, 1 << 20, ctypes.byref(x), None)
    assert rc == -1 and frag in lib.sqllm_last_error(), lib.sqllm_last_error()
    assert lib.sqllm_lutgemv_fused_exchange(ctypes.byref(a), 16, 1, 1, None, 16, 1 << 20, None, None) == -1


def test_reference_quant_py_imports_against_our_extension():
    """Option A of INTEGRATION.md: the reference's own squeezellm/quant.py, unmodified, imports `quant_cuda` by name and finds every
    symbol it calls in OUR extension (except the *_balanced_* ones, which the reference's extension does not define either), and its
    QuantLinearLUT registers the same buffers as ours.  What quant.py calls and registers is recorded in
    tests/golden/reference_quant_api.json (tests/golden/make_golden_reference_api.py)."""
    import json
    import squeezellm_b200.quant as ours            # registers the in-tree extension as top-level module `quant_cuda`
    import quant_cuda                                # what quant.py:5 runs
    assert quant_cuda is ours.quant_cuda
    with open(os.path.join(GOLDEN, "reference_quant_api.json")) as f:
        rec = json.load(f)
    called = set(rec["quant_cuda_calls"])
    missing = {n for n in called if not hasattr(quant_cuda, n)}
    assert len(called - missing) == 12
    assert missing and all("balanced" in n for n in missing), missing
    assert rec["modules"]
    for mod in rec["modules"]:
        bits, K, N, bias, sparse, numvals, topx = mod["args"]
        m = ours.QuantLinearLUT(bits, K, N, bias, include_sparse=sparse, numvals=numvals, topX=topx)
        assert {k: buffer_signature(v) for k, v in m.state_dict().items()} == mod["buffers"], mod["args"]
