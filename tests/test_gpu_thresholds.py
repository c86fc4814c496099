"""GPU tests on both sides of the kernels' internal size thresholds, against the fp64 oracle.

  * dense rows per launch (topX): up to 32 the contributors combine rows that feed one channel and the finisher lists its rows with a
    ballot; past 32 every row travels alone and the list is built with a shared-memory atomic.  128 (quant_cuda.MAX_TOPX_FUSED) is
    the last value the fused path takes; past it QuantLinearLUT.forward runs the reference sequence and the batched symbols take the
    dense rows in blocks of 256.
  * owned strips per CTA of the fused finisher: past 8 (SOWN) the strip sums and the dense-row sums go through the workspace
    accumulator, which the finisher reads and re-zeroes.  Which CTA owns how many strips depends on the SM count, so those tests
    recompute the launch plan and assert that they reach the path.
  * out_features < 64 (one strip not even full): the v1 kernel, accumulate and fused.
  * out_features = 262144 (quant_cuda.MAX_N_FUSED): the last fused width; one more strip and the fused path refuses.
"""
import ctypes
import functools

import numpy as np
import pytest
import torch

from util import REL_TOL, TIGHT_TOL, abi_call, load_lib, module_call, oracle_chain, orc, rel_err, to_torch

pytestmark = pytest.mark.gpu

STRIP = 64   # output columns per strip
SOWN = 8     # owned strips whose sums a finishing CTA keeps in shared memory (lutgemv_v2.cuh, lutgemv_seq.cuh)


@pytest.fixture(scope="module")
def lib():
    lib = load_lib()
    lib.sqllm_debug_last_grid.restype = ctypes.c_int
    return lib


@pytest.fixture(scope="module")
def qc():
    from squeezellm_b200.quant import quant_cuda
    return quant_cuda


def module_from_layer(L):
    """QuantLinearLUT on the GPU holding the buffers of the oracle layer L."""
    from squeezellm_b200.quant import QuantLinearLUT
    has_csr = L["rows"] is not None
    topX = L["full_rows"].shape[1] if L["full_rows"] is not None else 0
    m = QuantLinearLUT(L["bits"], L["infeatures"], L["outfeatures"], L.get("bias") is not None, include_sparse=has_csr,
                       numvals=len(L["vals"]) if has_csr else 0, topX=topX)
    sd = m.state_dict()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in L.items() if isinstance(v, np.ndarray) and k in sd}, strict=False)
    return m.cuda()


def fused(qc, L, T, x, dtype=torch.float32):
    """quant_cuda.lutgemv_fused on x (numpy, fp16-representable) and the check that no bounded in-kernel wait gave up."""
    xt = torch.from_numpy(x).cuda().reshape(-1).to(dtype)
    y = qc.lutgemv_fused(xt, T["qweight"], T["lookup_table"], L["bits"], T.get("bias"), T["rows"], T["cols"], T["vals"],
                         T["full_rows"], T["full_row_indices"])
    assert not qc.workspace_error(), "a bounded wait of the fused kernel gave up (partial sums)"
    return y


def want_fused(L, x):
    bias = L.get("bias")
    return orc.forward_f64(L, x, mul_init=None if bias is None else bias[None, :])


# =====================================================================================================================================
# (a) dense-row count sweep
# =====================================================================================================================================
TOPX = [1, 31, 32, 33, 64, 127, 128]
SHAPES_A = [(4096, 4096), (512, 132)]   # (512, 132): three strips, the last one ragged
PATTERNS = ["distinct", "dup", "zero"]


def dense_indices(pattern, topX, N, rng):
    """distinct: channels spread evenly over all strips (so over the CTAs that own them), the first row on the last column N - 1;
    dup: pairs on one channel, pairs in one strip on neighbouring channels, and a quarter of the rows on one channel;
    zero: every row on channel 0, what a checkpoint without dense rows loads to."""
    if pattern == "zero":
        return np.zeros(topX, dtype=np.int32)
    if pattern == "distinct":
        c = np.round(np.linspace(N - 1, 0, topX)).astype(np.int64)
        assert len(np.unique(c)) == topX
        return np.concatenate([c[:1], rng.permutation(c[1:])]).astype(np.int32)
    c = rng.integers(0, N, size=topX)
    c[1::4] = c[0::4][:len(c[1::4])]
    c[2::4] = c[0::4][:len(c[2::4])] ^ 1   # same 64-column strip, other channel (N is a multiple of 4, so c ^ 1 < N)
    c[3::4] = c[0]
    return c.astype(np.int32)


@functools.lru_cache(maxsize=None)
def _base_layer(bits, K, N):
    return orc.make_layer(bits, K, N, sparsity=0.0045 if K >= 4096 else 0.01, seed=bits * 1000 + K + N, bias=True)


def dense_layer(bits, K, N, topX, pattern):
    rng = np.random.default_rng(topX * 31 + bits * 7 + PATTERNS.index(pattern))
    L = dict(_base_layer(bits, K, N))
    L["full_rows"] = (rng.standard_normal((K, topX)) * 0.05).astype(np.float32)
    L["full_row_indices"] = dense_indices(pattern, topX, N, rng)
    return L


def a_id(v):
    return f"{v[0]}x{v[1]}" if isinstance(v, tuple) else None


a_params = pytest.mark.parametrize("pattern", PATTERNS)
a_topx = pytest.mark.parametrize("topX", TOPX)
a_shape = pytest.mark.parametrize("shape", SHAPES_A, ids=a_id)
a_bits = pytest.mark.parametrize("bits", [3, 4])


@a_bits
@a_shape
@a_topx
@a_params
def test_dense_rows_c_abi_accumulate(lib, bits, shape, topX, pattern):
    K, N = shape
    L = dense_layer(bits, K, N, topX, pattern)
    x = orc.make_vec(K, seed=topX)
    init = np.random.default_rng(1).standard_normal((1, N)).astype(np.float32)
    T = to_torch(L)
    mul = torch.from_numpy(init.copy()).cuda()
    abi_call(lib, T, torch.from_numpy(x).cuda(), mul)
    torch.cuda.synchronize()
    assert rel_err(mul.cpu().numpy(), orc.forward_f64(L, x, mul_init=init)) < TIGHT_TOL


@a_bits
@a_shape
@a_topx
@a_params
@pytest.mark.parametrize("dtype", [torch.float16, torch.float32], ids=["fp16", "fp32"])
def test_dense_rows_fused(qc, bits, shape, topX, pattern, dtype):
    K, N = shape
    L = dense_layer(bits, K, N, topX, pattern)
    x = orc.make_vec(K, seed=topX + 1)
    T = to_torch(L)
    y1 = fused(qc, L, T, x, dtype)
    qc.set_deterministic(True)
    try:
        d1 = fused(qc, L, T, x, dtype)
        d2 = fused(qc, L, T, x, dtype)
        torch.cuda.synchronize()
    finally:
        qc.set_deterministic(False)
    assert torch.equal(d1, d2), "deterministic fused mode must be bit-reproducible"
    want = want_fused(L, x)
    for y in (y1, d1):
        assert y.dtype == dtype and y.shape == (N,)
        assert rel_err(y.float().cpu().numpy(), want) < (REL_TOL if dtype == torch.float16 else TIGHT_TOL)


@a_bits
@a_shape
@a_topx
@a_params
def test_dense_rows_module_forward(qc, bits, shape, topX, pattern):
    K, N = shape
    L = dense_layer(bits, K, N, topX, pattern)
    m = module_from_layer(L)
    assert m.fused_ok()
    x = torch.from_numpy(orc.make_vec(K, seed=topX + 2)).cuda().half().reshape(1, 1, K)
    y = m(x)
    assert not qc.workspace_error()
    assert y.shape == (1, 1, N) and y.dtype == torch.float16
    assert rel_err(y.float().cpu().numpy(), want_fused(L, x.float().cpu().numpy().reshape(1, K))) < REL_TOL


@a_bits
@a_shape
@pytest.mark.parametrize("topX", [129, 256, 384])
@pytest.mark.parametrize("pattern", ["dup", "zero"])
def test_module_forward_past_fused_topx_limit(qc, bits, shape, topX, pattern):
    """More dense rows than the fused path takes: forward() runs the reference sequence (bias.clone + symbol + to(dtype))."""
    K, N = shape
    L = dense_layer(bits, K, N, topX, pattern)
    m = module_from_layer(L)
    assert topX > qc.MAX_TOPX_FUSED and not m.fused_ok()
    with pytest.raises(RuntimeError, match="topX"):
        fused(qc, L, to_torch(L), orc.make_vec(K, seed=0))
    x = torch.from_numpy(orc.make_vec(K, seed=topX + 3)).cuda().half().reshape(1, 1, K)
    y = m(x)
    assert y.shape == (1, 1, N) and y.dtype == torch.float16
    assert rel_err(y.float().cpu().numpy(), want_fused(L, x.float().cpu().numpy().reshape(1, K))) < REL_TOL


BATCHED_CASES = [(bits, shape, topX, pattern) for bits in (3, 4) for shape in SHAPES_A for topX in (33, 128, 200, 256, 257, 384)
                 for pattern in ("distinct", "dup") if not (pattern == "distinct" and topX > shape[1])]


@pytest.mark.parametrize("case", BATCHED_CASES, ids=lambda c: f"w{c[0]}-{c[1][0]}x{c[1][1]}-t{c[2]}-{c[3]}")
@pytest.mark.parametrize("batch", [3, 16])
def test_dense_rows_batched_symbols(qc, case, batch):
    """The batched symbols take the dense rows in blocks of at most 256 (one launch per block)."""
    bits, (K, N), topX, pattern = case
    L = dense_layer(bits, K, N, topX, pattern)
    x = orc.make_vec(K, batch=batch, seed=topX + batch)
    T = to_torch(L)
    out = torch.zeros((batch, N), device="cuda")
    module_call(qc, T, torch.from_numpy(x).cuda(), out, batched=True)
    torch.cuda.synchronize()
    assert rel_err(out.cpu().numpy(), orc.forward_f64(L, x)) < TIGHT_TOL


@pytest.mark.parametrize("bits", [3, 4])
def test_stacked_siblings_past_fused_topx_limit(qc, bits):
    """Three siblings with topX = 50 each: every member is within the fused limit, the stacked layer (150 dense rows) is not.
    Each member's output must match its own oracle before and after fuse_siblings."""
    from squeezellm_b200.fusion import fuse_siblings
    K, N = 512, 256
    Ls = [orc.make_layer(bits, K, N, sparsity=0.01, topX=50, seed=40 + i, nonzero_full_rows=True, bias=True) for i in range(3)]
    Ls[1]["full_row_indices"][:10] = Ls[1]["full_row_indices"][0]   # several rows on one channel inside a member
    model = torch.nn.Module()
    for name, L in zip(("q_proj", "k_proj", "v_proj"), Ls):
        setattr(model, name, module_from_layer(L))
    x = torch.from_numpy(orc.make_vec(K, seed=41)).cuda().half().reshape(1, 1, K)
    xb = torch.from_numpy(orc.make_vec(K, batch=3, seed=42)).cuda().half().reshape(1, 3, K)
    wants = [want_fused(L, x.float().cpu().numpy().reshape(1, K)) for L in Ls]
    # the batched branch rounds to x's dtype before it adds the bias (reference quant.py:376-379)
    wants_b = [orc.forward_f64(L, xb.float().cpu().numpy().reshape(3, K)).astype(np.float16) + L["bias"] for L in Ls]
    members = (model.q_proj, model.k_proj, model.v_proj)
    for m, w in zip(members, wants):
        assert rel_err(m(x).float().cpu().numpy(), w) < REL_TOL
    groups = fuse_siblings(model)
    assert len(groups) == 1 and groups[0].layer.topX == 150
    for _ in range(2):
        ys = [m(x) for m in members]
        for y, w in zip(ys, wants):
            assert y.shape == (1, 1, N)
            assert rel_err(y.float().cpu().numpy(), w) < REL_TOL
    assert groups[0].launches == 2
    for m, w in zip(members, wants_b):  # prefill-shaped input: the batched symbols
        assert rel_err(m(xb).float().cpu().numpy(), w) < REL_TOL
    assert all(m.fused_ok() for m in members) and not groups[0].layer.fused_ok()


# =====================================================================================================================================
# (b) wide layers: more than SOWN owned strips per CTA
# =====================================================================================================================================
def plan(bits, K, N, sm):
    """make_plan2's arithmetic (lutgemv_kernels.cu) and the finisher's ownership rule (lutgemv_v2.cuh): CTA b covers work units
    [b * chunk, (b + 1) * chunk) of T = strips * R and owns the strips that START in that range, so0 .. so1 - 1; the last of them is
    its last segment when it touches at least two strips or starts on a strip boundary."""
    R = K // 8 if bits == 4 else K // 32
    strips = -(-N // STRIP)
    T = strips * R
    chunk = max(2, 2 * -(-T // (2 * sm)))
    G = -(-T // chunk)
    ctas = []
    for b in range(G):
        cb0, cb1 = b * chunk, min(T, (b + 1) * chunk)
        so0, so1 = -(-cb0 // R), -(-cb1 // R)
        nseg = (cb1 - 1) // R - cb0 // R + 1
        last = so1 - so0 - 1 if (nseg >= 2 or cb0 % R == 0) else -1
        ctas.append((so0, so1, last))
    return G, ctas


def owner(ctas, strip):
    """(CTA, index of the strip among the CTA's owned strips, whether it is the CTA's last segment)."""
    for b, (so0, so1, last) in enumerate(ctas):
        if so0 <= strip < so1:
            return b, strip - so0, strip - so0 == last
    raise AssertionError(f"strip {strip} has no owner")


def wide_channels(ctas, N, topX):
    """Dense-row channels: evenly over all strips (the first on column N - 1), plus, in a CTA that owns at least 10 strips, one at
    owned index 5 (kept in shared memory), two rows on one channel at owned index 8 (past SOWN, not the last segment) and one in
    the CTA's last segment."""
    b = next(b for b, (so0, so1, _) in enumerate(ctas) if so1 - so0 >= SOWN + 2)
    so0, so1, last = ctas[b]
    c8 = (so0 + SOWN) * STRIP + 17
    designed = [(so0 + 5) * STRIP + 63, c8, c8, (so0 + last) * STRIP + 40]
    spread = np.round(np.linspace(N - 1, 0, topX - len(designed))).astype(np.int64)
    return np.concatenate([spread[:1], designed, spread[1:]]).astype(np.int32)


def assert_reaches_sown_path(ctas, fri):
    assert max(so1 - so0 for so0, so1, _ in ctas) >= SOWN + 1, "no CTA owns more than SOWN strips"
    where = [owner(ctas, int(c) // STRIP) for c in fri]
    assert any(4 <= u < SOWN and not lst for _, u, lst in where), "no dense row in an owned strip kept in shared memory past FAST"
    assert any(u >= SOWN and not lst for _, u, lst in where), "no dense row in an owned strip past SOWN"
    assert any(lst for _, u, lst in where), "no dense row in a CTA's last segment"


def wide_layer(bits, K, N, topX, sm, seed, sparsity=0.01):
    """Random layer in the reference's buffer format, CSR built with numpy (make_layer's per-channel loop is slow at these widths)."""
    rng = np.random.default_rng(seed)
    L = dict(bits=bits, infeatures=K, outfeatures=N)
    L["qweight"] = rng.integers(-2**31, 2**31, size=(K // 32 * bits, N), dtype=np.int64).astype(np.int32)
    L["lookup_table"] = np.sort(rng.standard_normal((N, 2**bits)).astype(np.float32) * 0.02, axis=1)
    L["bias"] = (rng.standard_normal(N) * 0.1).astype(np.float32)
    mask = rng.random((N, K), dtype=np.float32) < sparsity
    rows = np.zeros(N + 1, dtype=np.int32)
    rows[1:] = np.cumsum(mask.sum(axis=1))
    L["rows"], L["cols"] = rows, np.nonzero(mask)[1].astype(np.int32)   # row-major: sorted columns inside a row
    L["vals"] = (rng.standard_normal(len(L["cols"])) * 0.1).astype(np.float32)
    L["full_rows"] = (rng.standard_normal((K, topX)) * 0.05).astype(np.float32)
    L["full_row_indices"] = wide_channels(plan(bits, K, N, sm)[1], N, topX) if N <= 262144 else \
        np.round(np.linspace(N - 1, 0, topX)).astype(np.int32)
    return L


WIDE = [(4, 64, 131072), (3, 64, 131072), (4, 128, 262144)]


@pytest.mark.parametrize("shape", WIDE, ids=lambda s: f"w{s[0]}-{s[1]}x{s[2]}")
@pytest.mark.parametrize("topX", [10, 128])
def test_wide_layer_owned_strips_past_sown(qc, lib, shape, topX):
    bits, K, N = shape
    sm = qc.sm_count()
    G, ctas = plan(bits, K, N, sm)
    L = wide_layer(bits, K, N, topX, sm, seed=N + topX + bits)
    assert_reaches_sown_path(ctas, L["full_row_indices"])
    T = to_torch(L)
    x = orc.make_vec(K, seed=topX)
    want = want_fused(L, x)
    y1 = fused(qc, L, T, x)
    assert lib.sqllm_debug_last_grid() == G, "the launch plan differs from the one the reach assertions were computed for"
    assert rel_err(y1.cpu().numpy(), want) < TIGHT_TOL
    # the same layer again on the same stream: an accumulator column left non-zero would be counted twice
    y2 = fused(qc, L, T, x)
    assert rel_err(y2.cpu().numpy(), y1.cpu().numpy()) < TIGHT_TOL
    yh = fused(qc, L, T, x, torch.float16)
    assert rel_err(yh.float().cpu().numpy(), want) < REL_TOL
    # then a different, smaller layer through the same workspace
    S = orc.make_layer(bits, 4096, 4096, sparsity=0.0045, topX=10, seed=5, nonzero_full_rows=True, bias=True)
    xs = orc.make_vec(4096, seed=6)
    assert rel_err(fused(qc, S, to_torch(S), xs).cpu().numpy(), want_fused(S, xs)) < TIGHT_TOL
    # the accumulate entry point on the same layer
    mul = torch.zeros(N, device="cuda")
    abi_call(lib, T, torch.from_numpy(x).cuda(), mul)
    torch.cuda.synchronize()
    assert rel_err(mul.cpu().numpy(), orc.forward_f64(L, x)) < TIGHT_TOL


def test_width_past_max_n_fused(qc, lib):
    """One strip past MAX_N_FUSED: the fused path refuses with a message naming out_features; the accumulate symbols and the module
    (which then runs the reference sequence) compute it."""
    bits, K, N = 4, 128, qc.MAX_N_FUSED + 4
    L = wide_layer(bits, K, N, 10, qc.sm_count(), seed=3)
    T = to_torch(L)
    x = orc.make_vec(K, seed=3)
    with pytest.raises(RuntimeError, match="out_features"):
        fused(qc, L, T, x)
    mul = torch.zeros(N, device="cuda")
    abi_call(lib, T, torch.from_numpy(x).cuda(), mul)
    torch.cuda.synchronize()
    assert rel_err(mul.cpu().numpy(), orc.forward_f64(L, x)) < TIGHT_TOL
    m = module_from_layer(L)
    assert not m.fused_ok()
    xh = torch.from_numpy(x).cuda().half().reshape(1, 1, K)
    assert rel_err(m(xh).float().cpu().numpy(), want_fused(L, x)) < REL_TOL


# =====================================================================================================================================
# (c) narrow layers: the v1 kernel
# =====================================================================================================================================
@pytest.mark.parametrize("N", [4, 12, 60, 64])
@pytest.mark.parametrize("bits", [3, 4])
def test_narrow_layers(qc, bits, N):
    """out_features < 64 runs the v1 kernel (64: the v2 kernel, the other side).  All 12 symbols at batch 1 and 3, and the fused
    path in both summation modes.  (The reference's kernels read out of bounds at these widths: oracle only.)"""
    K = 512
    L = orc.make_layer(bits, K, N, sparsity=0.02, seed=N + bits, bias=True)
    L["full_rows"] = (np.random.default_rng(N).standard_normal((K, 5)) * 0.05).astype(np.float32)
    L["full_row_indices"] = np.array([N - 1, 0, N - 1, 1, N // 2], dtype=np.int32)
    for batch in (1, 3):
        x = orc.make_vec(K, batch=batch, seed=batch)
        for kind in ("dense", "spmv", "hybrid"):
            Lk = dict(L)
            if kind == "dense":
                Lk["rows"] = Lk["cols"] = Lk["vals"] = None
            if kind != "hybrid":
                Lk["full_rows"] = Lk["full_row_indices"] = None
            T = to_torch(Lk)
            out = torch.zeros((batch, N), device="cuda")
            module_call(qc, T, torch.from_numpy(x).cuda().reshape(-1) if batch == 1 else torch.from_numpy(x).cuda(), out.reshape(-1) if batch == 1 else out,
                        batched=batch > 1)
            torch.cuda.synchronize()
            assert rel_err(out.cpu().numpy(), orc.forward_f64(Lk, x)) < TIGHT_TOL, (kind, batch)
    T = to_torch(L)
    x = orc.make_vec(K, seed=7)
    want = want_fused(L, x)
    for dtype in (torch.float32, torch.float16):
        y = fused(qc, L, T, x, dtype)
        qc.set_deterministic(True)
        try:
            d1 = fused(qc, L, T, x, dtype)
            d2 = fused(qc, L, T, x, dtype)
            torch.cuda.synchronize()
        finally:
            qc.set_deterministic(False)
        assert torch.equal(d1, d2)
        for v in (y, d1):
            assert rel_err(v.float().cpu().numpy(), want) < (REL_TOL if dtype == torch.float16 else TIGHT_TOL), dtype


# =====================================================================================================================================
# (d) the sequence kernel past SOWN
# =====================================================================================================================================
@pytest.mark.parametrize("bits", [3, 4])
def test_sequence_wide_item_past_sown(qc, bits):
    """A chain (64 -> 131072) -> (4096 -> 4096) reading a 4096-slice of the wide output: the wide item's finishers own more than SOWN
    strips (lutgemv_seq.cuh).  Checked against the fp64 oracle chain with fp16 hand-overs, over three replays.  The wide item has dense
    rows but no CSR: the sequence kernel keeps a CTA's outlier rows in shared memory and refuses more than 255 of them per CTA, i.e.
    a CSR layer wider than about 255 x SMs columns, which leaves no CTA with more than SOWN strips."""
    from squeezellm_b200.runtime import DecodeSequence
    sm = qc.sm_count()
    K0, N0, off = 64, 131072, 65536 + 512
    _, ctas = plan(bits, K0, N0, sm)
    L0 = wide_layer(bits, K0, N0, 10, sm, seed=90 + bits)
    L0["rows"] = L0["cols"] = L0["vals"] = None
    assert_reaches_sown_path(ctas, L0["full_row_indices"])
    L1 = orc.make_layer(bits, 4096, 4096, sparsity=0.0045, topX=10, seed=91, nonzero_full_rows=True)
    layers = [L0, L1]
    for L in layers:  # keep activations O(1) through the chain, as in test_sequence_gpu
        L["lookup_table"] = (L["lookup_table"] * (50.0 / np.sqrt(L["infeatures"]))).astype(np.float32)
        L["bias"] = None
    dims = [(K0, N0, 0), (4096, 4096, off)]
    mods = [module_from_layer(L) for L in layers]
    mods[0]._sparse_args = lambda: (None, None, None, mods[0].full_rows, mods[0].full_row_indices)  # dense rows without CSR
    seq = DecodeSequence(K0, "cuda", lut_mode="exact")
    vecs, prev = [], seq.input
    for m, (K, N, o) in zip(mods, dims):
        prev = seq.matvec(m, prev[o:o + K])
        vecs.append(prev)
    seq.compile(outputs=vecs)
    x = orc.make_vec(K0, seed=5).reshape(-1).astype(np.float16)
    for rep in range(3):
        xr = x if rep < 2 else (x.astype(np.float32) * 0.5).astype(np.float16)
        seq.x.copy_(torch.from_numpy(xr).cuda())
        outs = [o.clone() for o in seq.replay()]
        torch.cuda.synchronize()
        assert not seq.error(), "a bounded in-kernel wait of the sequence gave up"
        want = oracle_chain(layers, dims, xr.astype(np.float64))
        for i, (o, w) in enumerate(zip(outs, want)):
            got = o.float().cpu().numpy().astype(np.float64)
            err = np.abs(got - w).max() / max(np.abs(w).max(), 1e-30)
            assert err < 2 * REL_TOL, f"rep {rep} item {i}: max-norm error {err:.3e} vs the oracle chain"
        assert rel_err(outs[0].float().cpu().numpy(), want[0]) < REL_TOL

