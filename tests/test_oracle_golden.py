"""CPU tests: the oracle (C restatement + numpy restatement) against fixtures produced by the
REFERENCE's own code - tests/golden/pack2_*.npz (reference pack2 run on CPU, make_golden_pack2.py) and
tests/golden/refkernel_*.npz (reference CUDA kernels run on a B200, make_golden_gpu.py)."""
import numpy as np
import pytest
import torch

from util import orc, golden_files, rel_err, REL_TOL, TIGHT_TOL

PACK2 = golden_files("pack2_")
REFK = golden_files("refkernel_")


def test_fixtures_present():
    assert len(PACK2) >= 6, "run tests/golden/make_golden_pack2.py where /root/reference exists"


@pytest.mark.parametrize("path", PACK2, ids=lambda p: p.split("pack2_")[-1][:-4])
def test_unpack_matches_reference_pack2(path):
    g = np.load(path)
    bits = int(g["bits"])
    want = g["indices"].T  # [K, N]
    assert np.array_equal(orc.unpack(g["qweight"], bits), want), "C oracle unpack != indices the reference packed"
    assert np.array_equal(orc.unpack_np(g["qweight"], bits), want), "numpy restatement disagrees"


@pytest.mark.parametrize("path", PACK2, ids=lambda p: p.split("pack2_")[-1][:-4])
def test_pack_is_bit_identical_to_reference_pack2(path):
    from squeezellm_b200.quant import pack_indices
    g = np.load(path)
    bits = int(g["bits"])
    idx = g["indices"].T
    for name, fn in (("C oracle", orc.pack), ("numpy oracle", orc.pack_np), ("squeezellm_b200.pack_indices", pack_indices)):
        assert np.array_equal(fn(idx, bits), g["qweight"]), f"{name} differs from the reference's qweight"


@pytest.mark.parametrize("path", PACK2, ids=lambda p: p.split("pack2_")[-1][:-4])
def test_our_pack2_reproduces_reference_buffers(path):
    """QuantLinearLUT.pack2 (vectorised) must emit the reference's buffers: qweight, lookup_table and the
    'outlier - zero centroid' CSR (reference quant.py:117-131)."""
    from squeezellm_b200.quant import QuantLinearLUT
    g = np.load(path)
    bits, K, N = int(g["bits"]), int(g["K"]), int(g["N"])
    sparse = "rows" in g.files
    lut = [[(g["centroids"][c], g["indices"][c])] for c in range(N)]
    outl = torch.from_numpy(g["outliers_dense"]).to_sparse() if sparse else None
    q = QuantLinearLUT(bits, K, N, False, include_sparse=sparse)
    q.pack2(torch.nn.Linear(K, N, bias=False), (lut, outl), sparse)
    assert q.qweight.dtype == torch.int32 and np.array_equal(q.qweight.numpy(), g["qweight"])
    assert q.lookup_table.dtype == torch.float32 and np.array_equal(q.lookup_table.numpy(), g["lookup_table"])
    if sparse:
        assert np.array_equal(q.rows.numpy(), g["rows"]) and q.rows.dtype == torch.int32
        assert np.array_equal(q.cols.numpy(), g["cols"]) and q.cols.dtype == torch.int32
        assert np.array_equal(q.vals.numpy(), g["vals"]) and q.vals.dtype == torch.float32
        assert set(q.state_dict().keys()) == {"qweight", "lookup_table", "rows", "cols", "vals"}


@pytest.mark.parametrize("bits", [3, 4])
def test_pack_unpack_roundtrip_random_words(bits):
    """Every int32 bit pattern is a valid packed weight: unpack -> pack is the identity."""
    rng = np.random.default_rng(7)
    q = rng.integers(-2**31, 2**31, size=(bits * 8, 96), dtype=np.int64).astype(np.int32)
    idx = orc.unpack(q, bits)
    assert idx.max() < 2**bits
    assert np.array_equal(orc.pack(idx, bits), q)
    assert np.array_equal(orc.pack_np(orc.unpack_np(q, bits), bits), q)


@pytest.mark.parametrize("bits,K,N,sp,topx", [(4, 128, 64, 0.0, 0), (3, 128, 64, 0.0, 0), (4, 256, 128, 0.02, 0),
                                                (3, 256, 128, 0.02, 3), (4, 128, 192, 0.01, 10), (4, 256, 192, 0.01, 64)])
def test_oracle_forward_against_plain_numpy(bits, K, N, sp, topx):
    """forward_f64 == dequantise with the (golden-pinned) unpack, then a float64 matmul + dense CSR + dense rows."""
    L = orc.make_layer(bits, K, N, sparsity=sp, topX=topx, seed=11, nonzero_full_rows=True)
    if topx:  # several dense rows on one output channel: every odd row shares the channel of the row before it, a quarter share channel 0
        fri = L["full_row_indices"]
        fri[1::2] = fri[0::2][:len(fri[1::2])]
        fri[3::4] = 0
    x = orc.make_vec(K, batch=3, seed=5)
    idx = orc.unpack_np(L["qweight"], bits).astype(np.int64)             # [K, N]
    W = np.take_along_axis(L["lookup_table"].astype(np.float64).T, idx, axis=0)  # W[k, c] = LUT[c, idx[k, c]]
    want = x.astype(np.float64) @ W
    if L["rows"] is not None:
        S = np.zeros((N, K))
        for c in range(N):
            S[c, L["cols"][L["rows"][c]:L["rows"][c + 1]]] = L["vals"][L["rows"][c]:L["rows"][c + 1]]
        want += x.astype(np.float64) @ S.T
    if L["full_rows"] is not None:
        part = x.astype(np.float64) @ L["full_rows"].astype(np.float64)
        for j, c in enumerate(L["full_row_indices"]):
            want[:, c] += part[:, j]
    init = np.random.default_rng(3).standard_normal((3, N)).astype(np.float32)
    got = orc.forward_f64(L, x, mul_init=init)
    assert np.allclose(got, want + init, rtol=1e-12, atol=1e-12)
    # the fp32 "one legal reference ordering" emulation and the fp16-dequant baseline stay inside north_star's tolerance
    assert rel_err(orc.forward_f32_blocked(L, x, mul_init=init), got) < TIGHT_TOL
    y16, _ = orc.cpu_dequant_matmul(L, x, compute_dtype="float32")
    assert rel_err(y16 + init, got) < TIGHT_TOL


def test_cpu_baseline_fp16_dequant_within_north_star_tolerance():
    """BASELINE.json configs[0]: single w4-s0 NUQ matvec, fp16 dequant + torch.matmul on CPU (small here)."""
    L = orc.make_layer(4, 512, 256, seed=2)
    x = orc.make_vec(512, seed=2)
    y16, _ = orc.cpu_dequant_matmul(L, x, compute_dtype="float16")
    assert rel_err(y16, orc.forward_f64(L, x)) < 2e-2  # fp16 weights+accumulate: a baseline, not a parity bar


@pytest.mark.skipif(not REFK, reason="tests/golden/refkernel_*.npz not generated yet (needs one GPU run)")
@pytest.mark.parametrize("path", REFK, ids=lambda p: p.split("refkernel_")[-1][:-4])
def test_oracle_matches_reference_kernel_outputs(path):
    """Pins the oracle's arithmetic: outputs of the reference's own CUDA kernels (oracle/_ref, run on a B200)
    for the inputs stored next to them."""
    g = np.load(path, allow_pickle=False)
    L = {k: (g[k] if k in g.files else None) for k in ("qweight", "lookup_table", "rows", "cols", "vals", "full_rows", "full_row_indices")}
    L.update(bits=int(g["bits"]), infeatures=int(g["K"]), outfeatures=int(g["N"]))
    want = g["mul_out"]
    got = orc.forward_f64(L, g["vec"], mul_init=g["mul_init"])
    assert rel_err(want, got) < REL_TOL
    assert rel_err(want, got) < TIGHT_TOL  # in practice the reference's fp32 atomics sit ~1e-6 from fp64
