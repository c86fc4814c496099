"""GPU parity tests (run on the B200 with `-m gpu`): our CUDA path, called through the C ABI (ctypes on
libsqllm_b200.so) and through the `quant_cuda` module, against the CPU oracle on the same seeded inputs, and
against the outputs of the reference's own kernels for the same inputs (tests/golden/refparity_*.npz, written on a
B200 by tests/golden/make_golden_parity.py)."""
import os

import numpy as np
import pytest
import torch

from util import GOLDEN, REL_TOL, TIGHT_TOL, load_lib, orc, rel_err, to_torch
from util import abi_call as _abi_call, module_call as _module_call

pytestmark = pytest.mark.gpu

SHAPES = [  # (bits, K, N, sparsity, topX, nonzero_full_rows, skew)
    (4, 128, 128, 0.0, 0, False, False),
    (3, 128, 128, 0.0, 0, False, False),
    (4, 256, 64, 0.02, 0, False, False),
    (3, 256, 192, 0.02, 4, True, False),
    (4, 512, 132, 0.01, 10, True, False),       # out not a multiple of 64 (ragged last strip), out % 4 == 0
    (3, 192, 68, 0.01, 3, True, True),          # in a multiple of 64 only; ragged strip
    (4, 4096, 4096, 0.0, 0, False, False),      # BASELINE configs[0]
    (4, 4096, 4096, 0.0045, 10, False, False),  # w4-s45 as llama.py runs it (hybrid, zero full_rows)
    (3, 4096, 4096, 0.0045, 10, True, True),    # w3-s45, skewed outliers, non-zero dense rows
    (4, 4096, 11008, 0.0045, 10, True, False),
    (3, 11008, 4096, 0.0045, 0, False, True),
    (4, 5120, 5120, 0.0005, 10, True, False),   # 13B w4-s5
    # BASELINE shapes that round 1 left out (VERDICT r01, "parity gaps")
    (3, 4096, 11008, 0.0045, 10, False, False), # 7B w3-s45 gate/up
    (4, 5120, 13824, 0.0005, 10, False, False), # 13B gate/up
    (4, 13824, 5120, 0.0005, 10, False, False), # 13B down
    (3, 8192, 8192, 0.0045, 10, False, False),  # 65B q/k/v/o
    (3, 8192, 22016, 0.0045, 10, False, False), # 65B gate/up
    (3, 22016, 8192, 0.0045, 10, True, False),  # 65B down
    (3, 8192, 2752, 0.0045, 10, False, False),  # 65B gate/up, 1 of 8 column shards: 43 strips, not a multiple of 128
    (3, 22016, 1024, 0.0045, 10, False, False), # 65B down, 1 of 8 column shards
    (4, 4096, 22016, 0.0045, 10, False, False), # 7B gate+up stacked (fusion.py)
    (4, 4096, 12288, 0.0045, 10, True, True),   # 7B q+k+v stacked, skewed outliers
    (4, 256, 44032, 0.01, 4, True, False),      # more CSR rows per CTA than the shared row accumulator holds (mailbox fallback path)
    (3, 11008, 64, 0.01, 4, True, False),       # one strip, every CTA inside it: 147 mailbox rows for one owner
]
IDS = [f"w{b}-{k}x{n}-s{int(s*1e4)}-t{t}{'-nz' if z else ''}{'-skew' if sk else ''}" for b, k, n, s, t, z, sk in SHAPES]
BATCHED_SHAPES = [s for s in SHAPES if s[1] <= 512] + [(4, 4096, 4096, 0.0045, 10, True, False), (3, 11008, 4096, 0.0045, 10, True, True)]
BATCHES = [2, 5, 16, 64]


def batched_id(s):
    return f"w{s[0]}-{s[1]}x{s[2]}-t{s[4]}"


def _layer(shape, seed):
    bits, K, N, sp, topx, nz, skew = shape
    L = orc.make_layer(bits, K, N, sparsity=sp, topX=topx, seed=seed, skew=skew, nonzero_full_rows=nz)
    if topx and sp == 0:
        L["full_rows"] = L["full_row_indices"] = None
    return L


def matvec_case(shape):
    """Layer and x of test_matvec_module_vs_reference_kernel."""
    return _layer(shape, shape[1] + shape[2] + shape[0]), orc.make_vec(shape[1], seed=2)


def batched_case(shape, batch):
    """Layer and x [batch, K] of test_batched_symbols_vs_oracle_and_reference."""
    return _layer(shape, 3), orc.make_vec(shape[1], batch=batch, seed=3)


def fingerprint(L, x):
    """Sums of every input array: stored reference outputs are only valid for the inputs they were computed from."""
    keys = ("qweight", "lookup_table", "rows", "cols", "vals", "full_rows", "full_row_indices")
    return np.array([np.asarray(a, dtype=np.float64).sum() for a in [L[k] for k in keys if L[k] is not None] + [x]])


def vs_reference(got, stored, key, L, x):
    """rel_err of our output against the reference kernel's, at the output positions stored for case `key`."""
    assert f"{key}.ref" in stored.files, f"no stored reference output for {key}: run tests/golden/make_golden_parity.py"
    assert np.allclose(stored[f"{key}.fingerprint"], fingerprint(L, x), rtol=1e-9, atol=0), f"{key}: inputs differ from the stored ones"
    return rel_err(np.asarray(got).reshape(-1)[stored[f"{key}.idx"]], stored[f"{key}.ref"])


@pytest.fixture(scope="module")
def lib():
    return load_lib()


@pytest.fixture(scope="module")
def qc():
    from squeezellm_b200.quant import quant_cuda
    return quant_cuda


@pytest.fixture(scope="module")
def ref():
    """Outputs of the reference's kernels: {"matvec": npz, "batched": npz}."""
    return {k: np.load(os.path.join(GOLDEN, f"refparity_{k}.npz")) for k in ("matvec", "batched")}


@pytest.mark.parametrize("bits", [3, 4])
def test_integer_unpack_bit_exact(qc, bits):
    """north_star: 'the integer unpack path alone is bit-exact' - the kernels' shift/mask/PRMT expressions vs the oracle."""
    rng = np.random.default_rng(bits)
    q = rng.integers(-2**31, 2**31, size=(bits * 16, 200), dtype=np.int64).astype(np.int32)
    got = qc.unpack_indices(torch.from_numpy(q).cuda(), bits).cpu().numpy()
    assert np.array_equal(got, orc.unpack(q, bits))


@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_matvec_c_abi_vs_oracle(lib, shape):
    bits, K, N, sp, topx, nz, skew = shape
    L = orc.make_layer(bits, K, N, sparsity=sp, topX=topx, seed=K + N + bits, skew=skew, nonzero_full_rows=nz)
    if topx and sp == 0:
        L["full_rows"] = L["full_row_indices"] = None
    x = orc.make_vec(K, seed=1)
    init = np.random.default_rng(0).standard_normal((1, N)).astype(np.float32)  # "bias.clone()" pre-fill (quant.py:215)
    T = to_torch(L)
    mul = torch.from_numpy(init.copy()).cuda()
    _abi_call(lib, T, torch.from_numpy(x).cuda(), mul)
    torch.cuda.synchronize()
    want = orc.forward_f64(L, x, mul_init=init)
    e = rel_err(mul.cpu().numpy(), want)
    assert e < REL_TOL and e < TIGHT_TOL, e


@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_matvec_module_vs_reference_kernel(qc, ref, shape):
    """Identical packed weights and inputs through the reference's own kernels on a B200 (north_star's parity statement; shapes
    that are not multiples of 128 ran zero-padded, see make_golden_parity.py)."""
    L, x = matvec_case(shape)
    T = to_torch(L)
    ours = torch.zeros(shape[2], device="cuda")
    _module_call(qc, T, torch.from_numpy(x).cuda().reshape(-1), ours, batched=False)
    torch.cuda.synchronize()
    assert vs_reference(ours.cpu().numpy(), ref["matvec"], IDS[SHAPES.index(shape)], L, x) < REL_TOL


@pytest.mark.parametrize("shape", BATCHED_SHAPES, ids=batched_id)
@pytest.mark.parametrize("batch", BATCHES)
def test_batched_symbols_vs_oracle_and_reference(qc, ref, shape, batch):
    L, x = batched_case(shape, batch)
    T = to_torch(L)
    xs = torch.from_numpy(x).cuda()
    ours = torch.zeros((batch, shape[2]), device="cuda")
    _module_call(qc, T, xs, ours, batched=True)
    torch.cuda.synchronize()
    want = orc.forward_f64(L, x)
    assert rel_err(ours.cpu().numpy(), want) < TIGHT_TOL
    assert vs_reference(ours.cpu().numpy(), ref["batched"], f"{batched_id(shape)}-b{batch}", L, x) < REL_TOL


@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32], ids=["fp16", "fp32"])
def test_fused_forward_vs_oracle(qc, shape, dtype):
    """The single-launch module path: fp16/fp32 x -> y in x's dtype, bias folded, no pre-zeroed output, deterministic."""
    bits, K, N, sp, topx, nz, skew = shape
    L = orc.make_layer(bits, K, N, sparsity=sp, topX=topx, seed=K + 7 * N, skew=skew, nonzero_full_rows=nz, bias=True)
    if topx and sp == 0:
        L["full_rows"] = L["full_row_indices"] = None
    x = orc.make_vec(K, seed=4)  # fp16-representable values, as decode activations are
    T = to_torch(L)
    xt = torch.from_numpy(x).cuda().reshape(-1).to(dtype)
    args = (xt, T["qweight"], T["lookup_table"], bits, T["bias"], T["rows"], T["cols"], T["vals"], T["full_rows"], T["full_row_indices"])
    y1 = qc.lutgemv_fused(*args)           # default: red.add accumulation (order may vary, like the reference's atomics)
    qc.set_deterministic(True)             # fixed-order reduction: must be bit-reproducible
    try:
        d1 = qc.lutgemv_fused(*args)
        d2 = qc.lutgemv_fused(*args)
        torch.cuda.synchronize()
    finally:
        qc.set_deterministic(False)
    assert y1.dtype == dtype and y1.shape == (N,)
    assert torch.equal(d1, d2), "deterministic fused mode must be bit-reproducible"
    want = orc.forward_f64(L, x, mul_init=L["bias"][None, :])
    for y in (y1, d1):
        e = rel_err(y.float().cpu().numpy(), want)
        assert e < (REL_TOL if dtype == torch.float16 else TIGHT_TOL), e  # fp16 output rounding is 2^-11 = 4.9e-4


def test_module_forward_matches_reference_sequence(qc):
    """QuantLinearLUT.forward fused vs the reference's zeros + float() + symbol + to(dtype) sequence (quant.py:212-312)."""
    from squeezellm_b200.quant import QuantLinearLUT
    for bits, sparse, topx in [(4, False, 0), (3, True, 0), (4, True, 10)]:
        K, N = 4096, 4096
        L = orc.make_layer(bits, K, N, sparsity=0.0045 if sparse else 0.0, topX=topx, seed=9, nonzero_full_rows=True)
        m = QuantLinearLUT(bits, K, N, False, include_sparse=sparse, numvals=len(L["vals"]) if sparse else 0, topX=topx)
        sd = {k: torch.from_numpy(v) for k, v in L.items() if isinstance(v, np.ndarray) and k in m.state_dict()}
        m.load_state_dict(sd, strict=False)
        m = m.cuda()
        x = torch.from_numpy(orc.make_vec(K, seed=8)).cuda().half().reshape(1, 1, K)
        QuantLinearLUT.use_fused = True
        y_f = m(x)
        QuantLinearLUT.use_fused = False
        y_r = m(x)
        QuantLinearLUT.use_fused = True
        assert y_f.shape == (1, 1, N) and y_f.dtype == torch.float16
        want = orc.forward_f64(L, x.float().cpu().numpy().reshape(1, K))
        assert rel_err(y_f.float().cpu().numpy(), want) < REL_TOL
        assert rel_err(y_r.float().cpu().numpy(), want) < REL_TOL
        # batched branch (prefill-style input)
        xb = torch.from_numpy(orc.make_vec(K, batch=3, seed=10)).cuda().half().reshape(1, 3, K)
        yb = m(xb)
        assert yb.shape == (1, 3, N)
        assert rel_err(yb.float().cpu().numpy(), orc.forward_f64(L, xb.float().cpu().numpy().reshape(3, K))) < REL_TOL


def test_full_size_properties_linearity_and_accumulate(qc):
    """BASELINE full-size shapes through size-independent properties: linearity in x and the accumulate contract."""
    K, N = 11008, 4096
    L = orc.make_layer(4, K, N, sparsity=0.0045, topX=10, seed=21, nonzero_full_rows=True)
    T = to_torch(L)
    x1 = torch.from_numpy(orc.make_vec(K, seed=1)).cuda().reshape(-1)
    x2 = torch.from_numpy(orc.make_vec(K, seed=2)).cuda().reshape(-1)
    def run(x, init=None):
        y = torch.zeros(N, device="cuda") if init is None else init.clone()
        _module_call(qc, T, x.contiguous(), y, batched=False)
        return y
    y1, y2, y12 = run(x1), run(x2), run(x1 + 2 * x2)
    assert rel_err((y1 + 2 * y2).cpu().numpy(), y12.cpu().numpy()) < TIGHT_TOL
    init = torch.randn(N, device="cuda")
    assert rel_err(run(x1, init).cpu().numpy(), (y1 + init).cpu().numpy()) < TIGHT_TOL
    # calling twice accumulates twice (the reference's atomicAdd contract)
    y = torch.zeros(N, device="cuda")
    _module_call(qc, T, x1, y, batched=False)
    _module_call(qc, T, x1, y, batched=False)
    assert rel_err(y.cpu().numpy(), (2 * y1).cpu().numpy()) < TIGHT_TOL


def test_edge_cases_empty_csr_and_duplicate_dense_rows(qc):
    """nnz = 0 CSR, a CSR with one enormous row (> the staging chunk), all-zero full_row_indices with non-zero rows."""
    K, N = 4096, 256
    L = orc.make_layer(4, K, N, sparsity=0.0, topX=0, seed=5)
    L["rows"] = np.zeros(N + 1, dtype=np.int32); L["cols"] = np.zeros(0, dtype=np.int32); L["vals"] = np.zeros(0, dtype=np.float32)
    x = orc.make_vec(K, seed=5)
    T = to_torch(L)
    y = torch.zeros(N, device="cuda")
    _module_call(qc, T, torch.from_numpy(x).cuda().reshape(-1), y, batched=False)
    assert rel_err(y.cpu().numpy(), orc.forward_f64(L, x)) < TIGHT_TOL
    # one output channel holds 3000 outliers, its neighbours few
    rng = np.random.default_rng(1)
    counts = rng.integers(0, 5, size=N); counts[37] = 3000; counts[38] = 100
    rows = np.zeros(N + 1, dtype=np.int32); rows[1:] = np.cumsum(counts)
    cols = np.concatenate([np.sort(rng.permutation(K)[:c]) for c in counts]).astype(np.int32)
    L["rows"], L["cols"], L["vals"] = rows, cols, (rng.standard_normal(len(cols)) * 0.1).astype(np.float32)
    L["full_rows"] = (rng.standard_normal((K, 10)) * 0.05).astype(np.float32)
    L["full_row_indices"] = np.zeros(10, dtype=np.int32)  # what a checkpoint without them leaves (all map to channel 0)
    T = to_torch(L)
    y = torch.zeros(N, device="cuda")
    _module_call(qc, T, torch.from_numpy(x).cuda().reshape(-1), y, batched=False)
    want = orc.forward_f64(L, x)
    assert rel_err(y.cpu().numpy(), want) < TIGHT_TOL
    yf = qc.lutgemv_fused(torch.from_numpy(x).cuda().reshape(-1), T["qweight"], T["lookup_table"], 4, None, T["rows"], T["cols"], T["vals"], T["full_rows"], T["full_row_indices"])
    assert rel_err(yf.cpu().numpy(), want) < TIGHT_TOL


def test_current_stream_and_graph_capture(qc):
    """Launches go to PyTorch's current stream (the reference uses the legacy stream): capturable in a CUDA graph."""
    K, N = 4096, 4096
    L = orc.make_layer(4, K, N, sparsity=0.0045, topX=10, seed=3)
    T = to_torch(L)
    x = torch.from_numpy(orc.make_vec(K, seed=3)).cuda().half().reshape(-1)
    args = (x, T["qweight"], T["lookup_table"], 4, None, T["rows"], T["cols"], T["vals"], T["full_rows"], T["full_row_indices"])
    eager = qc.lutgemv_fused(*args)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        qc.lutgemv_fused(*args)  # warm the per-stream workspace outside capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = qc.lutgemv_fused(*args)
    x.copy_(x)  # no-op write; replay
    g.replay(); g.replay()
    torch.cuda.synchronize()
    assert rel_err(out.float().cpu().numpy(), eager.float().cpu().numpy()) < REL_TOL  # default mode: last-bit differences allowed


def test_errors_raise_runtimeerror(qc):
    x = torch.zeros(128, device="cuda"); q = torch.zeros((16, 128), dtype=torch.int32, device="cuda")
    y = torch.zeros(128, device="cuda"); lut = torch.zeros((128, 16), device="cuda")
    with pytest.raises(RuntimeError, match="dtype"):
        qc.vecquant4matmul_nuq_perchannel(x.half(), q, y, lut)
    with pytest.raises(RuntimeError, match="features"):
        qc.vecquant4matmul_nuq_perchannel(torch.zeros(64, device="cuda"), q, y, lut)
    with pytest.raises(RuntimeError, match="contiguous"):
        qc.vecquant4matmul_nuq_perchannel(x, q.t().contiguous().t(), y, lut)
