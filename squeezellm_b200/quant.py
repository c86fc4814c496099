"""QuantLinearLUT / make_quant_lut - host-side mirror of the reference's module interface
(squeezellm/quant.py:28-435) on top of the B200-native `quant_cuda` extension.

Same class name, constructor signature, buffer names (= checkpoint keys: qweight, lookup_table, bias,
rows, cols, vals, full_rows, full_row_indices, startrows), `pack2`, `forward` and `make_quant_lut`
as the reference, so `llama.py`-style loaders work unchanged.  Differences, all behind the same API:

  * `forward` (batch-1 branch, reference quant.py:212-312) uses ONE fused launch
    (`quant_cuda.lutgemv_fused`: fp16/fp32 x in, y out in x's dtype, bias + CSR + dense rows fused;
    `quant_cuda.set_deterministic(True)` selects the bit-reproducible summation) instead of
    zeros + x.float() + 1-3 launches + y.to(dtype).  Layers past the fused limits (more than
    quant_cuda.MAX_TOPX_FUSED dense rows or quant_cuda.MAX_N_FUSED output channels) keep the reference sequence.  Set
    `QuantLinearLUT.use_fused = False` to go through the reference's 12 symbols exactly as quant.py does.
  * `balanced=True` raises NotImplementedError up front: the reference dispatches it to
    `vecquant{3,4}matmul_spmv_balanced_nuq_perchannel`, which its extension never defines
    (quant.py:238,282 vs quant_cuda.cpp:257-270), i.e. an AttributeError at the first forward.
  * the device is the buffers' device, not the hard-coded "cuda" (quant.py:218,317).
  * `pack2` is vectorised (numpy) instead of a Python row loop; output is bit-identical
    (tests/test_oracle_golden.py checks it against buffers produced by the reference's pack2).

There is NO CPU fallback: importing this module requires the compiled extension, and forward() requires
CUDA tensors (the extension raises otherwise).
"""
import glob
import importlib.util
import math
import os
import sys

import numpy as np
import torch
import torch.nn as nn

_PKG = os.path.dirname(os.path.abspath(__file__))


def _load_extension():
    """Load the in-tree extension as top-level module `quant_cuda` (the name the reference's quant.py:5 imports) WITHOUT touching
    sys.path: putting the package directory there would make build / quant / runtime / ... importable as top-level modules and
    shadow a user's own modules of those names."""
    if "quant_cuda" in sys.modules and hasattr(sys.modules["quant_cuda"], "lutgemv_fused"):
        return sys.modules["quant_cuda"]
    cands = sorted(glob.glob(os.path.join(_PKG, "quant_cuda*.so")))
    if not cands:
        raise ImportError(
            "squeezellm_b200: the compiled CUDA extension `quant_cuda` is missing; build it with "
            "`python -m squeezellm_b200.build` (needs nvcc, sm_100a). No CPU fallback exists.")
    spec = importlib.util.spec_from_file_location("quant_cuda", cands[0])
    mod = importlib.util.module_from_spec(spec)
    try:
        spec.loader.exec_module(mod)
    except ImportError as e:  # fail loudly: no silent eager fallback
        raise ImportError(f"squeezellm_b200: cannot load {cands[0]}: {e}. Rebuild with `python -m squeezellm_b200.build`. "
                          "No CPU fallback exists.") from e
    sys.modules["quant_cuda"] = mod
    return mod


quant_cuda = _load_extension()
# limits of the single-launch fused path (the 12 reference symbols have none)
MAX_TOPX_FUSED, MAX_N_FUSED = quant_cuda.MAX_TOPX_FUSED, quant_cuda.MAX_N_FUSED


def round_to_nearest_pole_sim(w, poles):
    """Round the numbers in w to the nearest value in poles (reference quant.py:8-24)."""
    poles_t = torch.as_tensor(np.asarray(poles), dtype=w.dtype)
    idx = (w.unsqueeze(0) - poles_t.reshape(-1, *([1] * w.dim()))).abs().argmin(dim=0)
    return poles_t[idx]


def pack_indices(idx_kn, bits):
    """uint8/int idx [K, N] -> packed int32 [K/32*bits, N] in the reference layout (quant.py:171-208)."""
    v = np.ascontiguousarray(idx_kn).astype(np.uint32)
    K, N = v.shape
    assert K % 32 == 0, "infeatures must be a multiple of 32"
    if bits == 4:
        v = v.reshape(K // 8, 8, N)
        sh = (4 * np.arange(8, dtype=np.uint32))[None, :, None]
        return np.bitwise_or.reduce(v << sh, axis=1).astype(np.uint32).view(np.int32)
    if bits != 3:
        raise NotImplementedError("Only 3 and 4 bits is supported.")
    v = v.reshape(K // 32, 32, N)
    s = (3 * np.arange(10, dtype=np.uint32))[None, :, None]
    w0 = np.bitwise_or.reduce(v[:, 0:10] << s, axis=1) | (v[:, 10] << 30)
    w1 = ((v[:, 10] >> 2) & 1) | np.bitwise_or.reduce(v[:, 11:21] << (s + 1), axis=1) | (v[:, 21] << 31)
    w2 = ((v[:, 21] >> 1) & 3) | np.bitwise_or.reduce(v[:, 22:32] << (s + 2), axis=1)
    q = np.empty((K // 32 * 3, N), dtype=np.uint32)
    q[0::3], q[1::3], q[2::3] = w0, w1, w2
    return q.view(np.int32)


class QuantLinearLUT(nn.Module):
    """Drop-in layer replacement (reference quant.py:28)."""

    use_fused = True  # class-wide switch: fused single-launch forward vs the reference's 12-symbol sequence
    # codebook precision of the fused path is process-wide: quant_cuda.set_lut_mode("exact" | "fp16")  (include/sqllm_b200.h)

    def __init__(self, bits, infeatures, outfeatures, bias, include_sparse=False, numvals=0, topX=0,
                 balanced=False, num_nonzero_per_thread=10):
        super().__init__()
        if bits not in [3, 4]:
            raise NotImplementedError("Only 3 and 4 bits is supported.")
        if balanced:
            raise NotImplementedError(
                "balanced SpMV is not available: the reference dispatches to quant_cuda.*_spmv_balanced_*, "
                "which its extension never defines (quant_cuda.cpp:257-270)")
        self.infeatures = infeatures
        self.outfeatures = outfeatures
        self.bits = bits
        self.register_buffer("qweight", torch.zeros((infeatures // 32 * self.bits, outfeatures), dtype=torch.int32))
        if bias:
            self.include_bias = True
            self.register_buffer("bias", torch.zeros((outfeatures)))
        else:
            self.include_bias = False
            self.bias = None
        self.register_buffer("lookup_table", torch.zeros((outfeatures, 2**self.bits), dtype=torch.float32))
        self.include_sparse = include_sparse
        self.numvals = numvals
        self.topX = topX
        if numvals > 0:
            self.register_buffer("rows", torch.zeros(outfeatures + 1, dtype=torch.int32))
            self.register_buffer("cols", torch.zeros(numvals, dtype=torch.int32))
            self.register_buffer("vals", torch.zeros(numvals, dtype=torch.float32))
        if topX > 0:
            self.register_buffer("full_rows", torch.zeros((infeatures, topX), dtype=torch.float32))
            self.register_buffer("full_row_indices", torch.zeros(topX, dtype=torch.int32))
        self.balanced = balanced
        self._sibling_group = None  # (SiblingGroup, index) once fusion.fuse_siblings has stacked this layer with its siblings

    # ------------------------------------------------------------------------------------------
    def pack2(self, linear, lookup_table, include_sparse, num_nonzero_per_thread=-1):
        """Fill the buffers from per-channel (centroids, indices) and an outlier matrix
        (reference quant.py:97-208).  lookup_table = (lut, outliers); lut[c][0] = (centroids, indices)."""
        if self.include_bias:
            self.bias = linear.bias.clone()
        lut, outliers = lookup_table
        num_channels = len(lut)
        K = linear.weight.shape[1]
        idx = np.empty((num_channels, K), dtype=np.uint8)
        cent = np.empty((num_channels, 2**self.bits), dtype=np.float32)
        for channel in range(num_channels):
            centroid, indices = lut[channel][0]  # last 0 is for group 0
            idx[channel] = np.asarray(indices)
            cent[channel] = np.asarray(centroid, dtype=np.float32)
        self.lookup_table = torch.from_numpy(cent)
        if include_sparse:
            outliers = outliers.to_dense().clone() if outliers.layout != torch.strided else outliers.clone()
            # the dense index at an outlier position encodes the centroid nearest to zero, so the sparse
            # value stored is (outlier - that centroid)  (reference quant.py:117-123)
            zero_map = torch.from_numpy(cent[np.arange(num_channels), np.abs(cent).argmin(axis=1)])
            nz = outliers != 0
            outliers = torch.where(nz, outliers - zero_map[:, None].to(outliers.dtype), outliers)
            csr = outliers.to_sparse(layout=torch.sparse_csr)
            self.register_buffer("rows", csr.crow_indices().to(torch.int32))
            self.register_buffer("cols", csr.col_indices().to(torch.int32))
            self.register_buffer("vals", csr.values().to(torch.float32))
            self.numvals = int(self.vals.shape[0])
        self.qweight = torch.from_numpy(pack_indices(idx.T, self.bits))

    # ------------------------------------------------------------------------------------------
    def _sparse_args(self):
        if not (self.include_sparse and hasattr(self, "rows")):
            return None, None, None, None, None
        fr = fri = None
        if self.topX > 0:
            fr, fri = self.full_rows, self.full_row_indices
        return self.rows, self.cols, self.vals, fr, fri

    def fused_ok(self):
        """True if the single-launch fused path takes this layer: at most MAX_TOPX_FUSED dense rows and at most MAX_N_FUSED
        output channels.  Past either limit forward() runs the reference sequence, whose symbols have
        no such limit (a stacked sibling group of three layers with topX = 50 each has 150 dense rows)."""
        fr = self._sparse_args()[3]
        topX = fr.shape[1] if fr is not None else 0
        return topX <= MAX_TOPX_FUSED and self.outfeatures <= MAX_N_FUSED

    def forward(self, x):
        if self._sibling_group is not None:
            group, index = self._sibling_group
            return group.member_forward(index, x)
        dev = self.qweight.device
        if x.shape[-1] == x.numel():
            outshape = list(x.shape)
            outshape[-1] = self.outfeatures
            if QuantLinearLUT.use_fused and x.dtype in (torch.float16, torch.float32) and self.fused_ok():
                rows, cols, vals, fr, fri = self._sparse_args()
                y = quant_cuda.lutgemv_fused(x.contiguous(), self.qweight, self.lookup_table, self.bits,
                                             self.bias, rows, cols, vals, fr, fri)
                return y.reshape(outshape)
            # reference sequence (quant.py:213-312)
            y = self.bias.clone() if self.bias is not None else torch.zeros((self.outfeatures), device=dev, dtype=torch.float32)
            dtype = x.dtype
            x = x.float().contiguous()
            self._dispatch(x, y, batched=False)
            return y.to(dtype).reshape(outshape)
        out_shape = x.shape[:-1] + (self.outfeatures,)
        x = x.reshape(-1, x.shape[-1])
        out = torch.zeros((x.shape[0], self.outfeatures), device=dev, dtype=torch.float32)
        dtype = x.dtype
        x = x.float().contiguous()
        self._dispatch(x, out, batched=True)
        out = out.to(dtype).reshape(out_shape)
        return out + self.bias if self.bias is not None else out

    def _dispatch(self, x, y, batched):
        """Pick 1 of the 12 quant_cuda symbols by (bits, batched, dense|spmv|hybrid) - reference quant.py:222-309,320-379."""
        b = self.bits
        sfx = "_batched" if batched else ""
        if self.include_sparse and self.topX > 0:
            fn = getattr(quant_cuda, f"vecquant{b}matmul_spmv_hybrid_nuq_perchannel{sfx}")
            fn(self.rows, self.cols, self.vals, x, self.full_rows, self.full_row_indices, y, self.outfeatures,
               self.qweight, self.lookup_table)
        elif self.include_sparse:
            fn = getattr(quant_cuda, f"vecquant{b}matmul_spmv_nuq_perchannel{sfx}")
            fn(self.rows, self.cols, self.vals, x, y, self.outfeatures, self.qweight, self.lookup_table)
        else:
            fn = getattr(quant_cuda, f"vecquant{b}matmul_nuq_perchannel{sfx}")
            fn(x, self.qweight, y, self.lookup_table)


def make_quant_lut(module, names, bits, name="", include_sparse=False, numvals=None, topX=0, balanced=False,
                   num_nonzero_per_thread=10):
    """Recursively replace the nn.Linear attributes listed in `names` by QuantLinearLUT
    (reference quant.py:386-435; same signature)."""
    if isinstance(module, QuantLinearLUT):
        return
    for attr in dir(module):
        tmp = getattr(module, attr)
        name1 = name + "." + attr if name != "" else attr
        if name1 in names:
            num = numvals[name1] if numvals is not None else 0
            delattr(module, attr)
            setattr(module, attr, QuantLinearLUT(bits, tmp.in_features, tmp.out_features, tmp.bias is not None,
                                                 include_sparse=include_sparse, numvals=num, topX=topX, balanced=balanced,
                                                 num_nonzero_per_thread=num_nonzero_per_thread))
    for name1, child in module.named_children():
        make_quant_lut(child, names, bits, name + "." + name1 if name != "" else name1, include_sparse=include_sparse,
                       numvals=numvals, topX=topX, balanced=balanced, num_nonzero_per_thread=num_nonzero_per_thread)
