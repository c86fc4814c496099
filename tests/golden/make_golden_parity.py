#!/usr/bin/env python3
"""Generate tests/golden/refparity_{matvec,batched}.npz on a B200: outputs of the REFERENCE's own CUDA kernels
(oracle/_ref/quant_cuda_ref*.so, built by oracle/build_ref.py) for the inputs of
tests/test_gpu_parity.py::test_matvec_module_vs_reference_kernel and ::test_batched_symbols_vs_oracle_and_reference.

    python tests/golden/make_golden_parity.py [OUT_DIR]        # default: tests/golden

The reference kernels read out of bounds unless in % 128 == 0 and out % 128 == 0 (SURVEY 2.1), so other shapes run
zero-padded to multiples of 128: padded inputs are 0, padded weights are index 0 of an all-zero table row, and the padded
outputs are dropped, so every stored output is a sum over the layer's own terms only.  For every case the files hold,
under the case's key,
  <key>.idx          int32   flat output positions: one seeded random position in each of min(numel, SAMPLES) equal
                             chunks of the output, so every region of the output is checked while the files stay small
  <key>.ref          float32 the reference kernel's outputs at those positions
  <key>.fingerprint  float64 sums of the inputs (test_gpu_parity.fingerprint), checked before the comparison
"""
import os
import sys
import zlib

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import build_ref  # noqa: E402
import test_gpu_parity as P  # noqa: E402
from util import rel_err, to_torch  # noqa: E402

SAMPLES = 256


def sample_index(numel, seed):
    rng = np.random.default_rng(seed)
    bounds = np.linspace(0, numel, min(numel, SAMPLES) + 1).astype(np.int64)
    return (bounds[:-1] + (rng.random(len(bounds) - 1) * np.diff(bounds)).astype(np.int64)).astype(np.int32)


def padded(L, x):
    bits, K, N = L["bits"], L["infeatures"], L["outfeatures"]
    Kp, Np = -(-K // 128) * 128, -(-N // 128) * 128
    Lp = dict(L, infeatures=Kp, outfeatures=Np, qweight=np.zeros((Kp // 32 * bits, Np), np.int32),
              lookup_table=np.zeros((Np, 2 ** bits), np.float32))
    Lp["qweight"][:K // 32 * bits, :N] = L["qweight"]
    Lp["lookup_table"][:N] = L["lookup_table"]
    if L["rows"] is not None:
        Lp["rows"] = np.concatenate([L["rows"], np.full(Np - N, L["rows"][-1], np.int32)])
    if L["full_rows"] is not None:
        Lp["full_rows"] = np.zeros((Kp, L["full_rows"].shape[1]), np.float32)
        Lp["full_rows"][:K] = L["full_rows"]
    xp = np.zeros(x.shape[:-1] + (Kp,), np.float32)
    xp[..., :K] = x
    return Lp, xp


def run_reference(ref, L, x, batch):
    """The reference symbol squeezellm/quant.py would pick, on the layer padded to multiples of 128; outputs [batch, N]."""
    Lp, xp = padded(L, x)
    theirs = torch.zeros((batch, Lp["outfeatures"]), device="cuda")
    xs = torch.from_numpy(xp).cuda()
    P._module_call(ref, to_torch(Lp), xs.reshape(-1) if batch == 1 else xs, theirs.reshape(-1) if batch == 1 else theirs, batched=batch > 1)
    torch.cuda.synchronize()
    return theirs.cpu().numpy()[:, :L["outfeatures"]]


def store(d, key, L, x, theirs):
    idx = sample_index(theirs.size, zlib.crc32(key.encode()))
    d[f"{key}.idx"], d[f"{key}.ref"] = idx, theirs.reshape(-1)[idx].astype(np.float32)
    d[f"{key}.fingerprint"] = P.fingerprint(L, x)
    # the stored values must describe the same computation as the fp64 oracle
    want = P.orc.forward_f64(L, x).reshape(-1)[idx]
    print(f"{key}: {idx.size} of {theirs.size} outputs, rel_err vs fp64 oracle {rel_err(d[f'{key}.ref'], want):.2e}")


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(out, exist_ok=True)
    ref = build_ref.load()
    matvec = {}
    for shape, key in zip(P.SHAPES, P.IDS):
        L, x = P.matvec_case(shape)
        store(matvec, key, L, x, run_reference(ref, L, x, 1))
    batched = {}
    for shape in P.BATCHED_SHAPES:
        for batch in P.BATCHES:
            L, x = P.batched_case(shape, batch)
            store(batched, f"{P.batched_id(shape)}-b{batch}", L, x, run_reference(ref, L, x, batch))
    for name, d in (("matvec", matvec), ("batched", batched)):
        np.savez_compressed(os.path.join(out, f"refparity_{name}.npz"), **d)


if __name__ == "__main__":
    main()
