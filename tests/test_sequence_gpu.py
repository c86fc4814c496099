"""GPU parity of the sequence kernel (csrc/lutgemv_seq.cuh, runtime.DecodeSequence): a chain of dependent matvecs run as ONE
persistent launch must give what the same layers give when called one by one (squeezellm/llama.py:226-234 drives
QuantLinearLUT.forward layer by layer), and what the fp64 oracle gives for the same chain with fp16 hand-overs."""
import numpy as np
import pytest
import torch

from util import REL_TOL, oracle_chain as _oracle_chain, orc, rel_err

pytestmark = pytest.mark.gpu


def _module(L, bits, K, N, topX):
    from squeezellm_b200.quant import QuantLinearLUT
    has_csr = L.get("rows") is not None
    m = QuantLinearLUT(bits, K, N, False, include_sparse=has_csr, numvals=len(L["vals"]) if has_csr else 0, topX=topX if has_csr else 0)
    sd = m.state_dict()
    m.load_state_dict({k: torch.from_numpy(v) for k, v in L.items() if isinstance(v, np.ndarray) and k in sd}, strict=False)
    return m.cuda()


def _scaled_layer(bits, K, N, sparsity, topX, seed, dup):
    L = orc.make_layer(bits, K, N, sparsity=sparsity, topX=topX, seed=seed, nonzero_full_rows=True)
    if topX and sparsity == 0:
        L["full_rows"] = L["full_row_indices"] = None
    elif topX >= 3 and dup:  # dense rows that feed the same output channel (their parts travel combined), one of them channel 0
        L["full_row_indices"][1] = L["full_row_indices"][0]
        L["full_row_indices"][2] = 0
    # keep activations O(1) through the chain
    L["lookup_table"] = (L["lookup_table"] * (50.0 / np.sqrt(K))).astype(np.float32)  # centroids ~ N(0, 1/K): |y| ~ |x|
    return L


def _stack_layers(Ls):
    """numpy restatement of stacking sibling layers along the output dimension (fusion.stack_buffers), for the oracle."""
    offs = np.cumsum([0] + [L["outfeatures"] for L in Ls])
    S = dict(bits=Ls[0]["bits"], infeatures=Ls[0]["infeatures"], outfeatures=int(offs[-1]), bias=None)
    S["qweight"] = np.concatenate([L["qweight"] for L in Ls], axis=1)
    S["lookup_table"] = np.concatenate([L["lookup_table"] for L in Ls], axis=0)
    S["rows"] = np.concatenate([[0]] + [L["rows"][1:] + sum(int(P["rows"][-1]) for P in Ls[:i]) for i, L in enumerate(Ls)]).astype(np.int32)
    S["cols"] = np.concatenate([L["cols"] for L in Ls])
    S["vals"] = np.concatenate([L["vals"] for L in Ls])
    S["full_rows"] = np.concatenate([L["full_rows"] for L in Ls], axis=1)
    S["full_row_indices"] = np.concatenate([L["full_row_indices"] + o for L, o in zip(Ls, offs)]).astype(np.int32)
    return S


def _chain(bits, dims, sparsity, topX, seed):
    """dims: [(K, N, x_offset into the previous output[, members])]; returns oracle layers + modules.  An item with members > 1 is
    the stacked layer that fusion.fuse_siblings builds from that many sibling layers of N / members columns and topX dense rows each."""
    from squeezellm_b200.fusion import SiblingGroup
    layers, mods = [], []
    for i, d in enumerate(dims):
        K, N = d[0], d[1]
        members = d[3] if len(d) > 3 else 1
        if members == 1:
            L = _scaled_layer(bits, K, N, sparsity, topX, seed + 17 * i, dup=i % 2 == 0)
            m = _module(L, bits, K, N, topX)
        else:
            Ls = [_scaled_layer(bits, K, N // members, sparsity, topX, seed + 17 * i + 1000 * j, dup=j == 0) for j in range(members)]
            L = _stack_layers(Ls)
            m = SiblingGroup([_module(Lj, bits, K, N // members, topX) for Lj in Ls]).layer
            assert m.topX == members * topX
        layers.append(L)
        mods.append(m)
    return layers, mods


CASES = [  # (bits, dims, sparsity, topX)
    (4, [(256, 768, 0), (256, 256, 512), (256, 704, 0), (704, 256, 0)], 0.0, 0),
    (4, [(256, 768, 0), (256, 256, 512), (256, 704, 0), (704, 256, 0)], 0.02, 4),
    (3, [(256, 768, 0), (256, 256, 512), (256, 704, 0), (704, 256, 0)], 0.02, 4),
    (4, [(512, 132, 0), (128, 200, 4), (192, 64, 8), (64, 512, 0), (512, 132, 0)], 0.01, 3),   # ragged strips, one-strip items
    (4, [(4096, 12288, 0), (4096, 4096, 8192), (4096, 22016, 0), (11008, 4096, 0)], 0.0045, 10, 3),  # LLaMA-7B decoder layer, three times over
    (3, [(4096, 12288, 0), (4096, 4096, 8192), (4096, 22016, 0), (11008, 4096, 0)], 0.0045, 10, 2),
    (4, [(256, 768, 0), (256, 256, 512), (256, 704, 0), (704, 256, 0)], 0.02, 43),        # > 32 dense rows per item, duplicate channels
    (4, [(512, 768, 0, 3), (256, 256, 512), (256, 768, 0, 3), (768, 132, 0)], 0.02, 11),  # stacked q+k+v of topX = 11: 33 dense rows
]
IDS = [f"w{c[0]}-{len(c[1])}items-K{c[1][0][0]}-s{int(c[2] * 1e4)}-t{c[3]}{'-stacked' if len(c[1][0]) > 3 else ''}" for c in CASES]


@pytest.mark.parametrize("case", CASES, ids=IDS)
@pytest.mark.parametrize("mode", ["exact", "fp16"])
def test_sequence_matches_layer_by_layer_and_oracle(case, mode):
    from squeezellm_b200.quant import quant_cuda
    from squeezellm_b200.runtime import DecodeSequence
    bits, dims, sp, topX = case[:4]
    layers, mods = _chain(bits, dims, sp, topX, seed=bits * 100 + len(dims))
    rep_n = case[4] if len(case) > 4 else 1  # the same matrices again (the generator is slow for 22016 channels): a longer chain
    dims, layers, mods = dims * rep_n, layers * rep_n, mods * rep_n
    x = orc.make_vec(dims[0][0], seed=5).reshape(-1).astype(np.float16)
    seq = DecodeSequence(dims[0][0], "cuda", lut_mode=mode)
    vecs, prev = [], seq.input
    dims = [d[:3] for d in dims]
    for m, (K, N, off) in zip(mods, dims):
        prev = seq.matvec(m, prev[off:off + K])
        vecs.append(prev)
    seq.compile(outputs=vecs)
    seq.x.copy_(torch.from_numpy(x).cuda())
    want = _oracle_chain(layers, dims, x.astype(np.float64), lut_fp16=(mode == "fp16"))
    # the same layers one by one through the module path
    quant_cuda.set_lut_mode(mode)
    try:
        ys, cur = [], torch.from_numpy(x).cuda()
        for m, (K, N, off) in zip(mods, dims):
            cur = m(cur[off:off + K].clone() if ys else cur)  # (a fresh allocation: the module path wants a 16-byte aligned x)
            ys.append(cur)
    finally:
        quant_cuda.set_lut_mode("exact")
    for rep in range(3):  # replays: the tags of the previous token must not be taken for this one's
        if rep == 2:
            seq.x.copy_(torch.from_numpy((x.astype(np.float32) * 0.5).astype(np.float16)).cuda())
        outs = [o.clone() for o in seq.replay()]
        torch.cuda.synchronize()
        assert not seq.error(), "a bounded in-kernel wait of the sequence gave up"
        if rep == 2:
            want = _oracle_chain(layers, dims, (x.astype(np.float32) * 0.5).astype(np.float16).astype(np.float64), lut_fp16=(mode == "fp16"))
        for i, (o, w) in enumerate(zip(outs, want)):
            got = o.float().cpu().numpy().astype(np.float64)
            # fp16 hand-overs: one fp16 ulp of an input moves later outputs; compare in the max norm at the north_star tolerance,
            # plus the strict per-element metric for the first item (no hand-over before it)
            err = np.abs(got - w).max() / max(np.abs(w).max(), 1e-30)
            assert err < 2 * REL_TOL, f"rep {rep} item {i}: max-norm error {err:.3e} vs the oracle chain"
            if i == 0 and mode == "exact":
                assert rel_err(got, w) < REL_TOL
            if rep < 2:
                ref = ys[i].float().cpu().numpy().astype(np.float64)
                err2 = np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30)
                assert err2 < 2 * REL_TOL, f"rep {rep} item {i}: {err2:.3e} vs the layer-by-layer module path"


def test_sequence_in_cuda_graph_and_plain_copies():
    """The two launches of a run are capturable; replays keep working (the token counter lives in device memory)."""
    from squeezellm_b200.runtime import DecodeSequence, GraphedDecodeStep
    bits, dims = 4, [(256, 768, 0), (256, 256, 512), (256, 704, 0), (704, 256, 0)]
    layers, mods = _chain(bits, dims, 0.02, 4, seed=77)
    seq = DecodeSequence(256, "cuda", lut_mode="exact")
    prev = seq.input
    for m, (K, N, off) in zip(mods, dims):
        prev = seq.matvec(m, prev[off:off + K])
    seq.compile(outputs=[prev])
    runner = GraphedDecodeStep(lambda x: seq.replay()[0], seq.x, warmup=2, static_input=True)
    for s in (1, 2, 3):
        x = orc.make_vec(256, seed=s).reshape(-1).astype(np.float16)
        y = runner(torch.from_numpy(x)).clone().float().numpy().astype(np.float64)
        w = _oracle_chain(layers, dims, x.astype(np.float64))[-1]
        assert np.abs(y - w).max() / np.abs(w).max() < 2 * REL_TOL
    assert not seq.error()
