#!/usr/bin/env python3
"""Generate tests/golden/reference_quant_api.json from the REFERENCE's squeezellm/quant.py (CPU only).

    SQLLM_REFERENCE_DIR=<reference checkout> python tests/golden/make_golden_reference_api.py

Records what the drop-in boundary has to offer the reference's module code: every `quant_cuda.<name>` that
quant.py calls, and the buffers (name, shape, dtype) its QuantLinearLUT registers for a few constructor calls.
The module is imported with the same stub `quant_cuda` as make_golden_pack2.py (its constructor never calls
the extension).  tests/test_abi.py checks our extension and our QuantLinearLUT against this record.
"""
import json
import os
import re
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))
from make_golden_pack2 import REF, load_reference_quant  # noqa: E402
from util import buffer_signature  # noqa: E402

OUT = os.path.join(HERE, "reference_quant_api.json")

# (bits, infeatures, outfeatures, bias, include_sparse, numvals, topX)
CONFIGS = [(4, 128, 128, False, True, 5, 10), (3, 256, 64, True, False, 0, 0), (3, 128, 96, True, True, 7, 0)]


def main():
    src = open(os.path.join(REF, "squeezellm", "quant.py")).read()
    QuantLinearLUT = load_reference_quant()
    modules = []
    for cfg in CONFIGS:
        bits, K, N, bias, sparse, numvals, topx = cfg
        m = QuantLinearLUT(bits, K, N, bias, include_sparse=sparse, numvals=numvals, topX=topx)
        buffers = {k: buffer_signature(v) for k, v in m.state_dict().items()}
        modules.append({"args": list(cfg), "buffers": buffers})
    rec = {"source": "squeezellm/quant.py", "quant_cuda_calls": sorted(set(re.findall(r"quant_cuda\.(\w+)", src))),
           "modules": modules}
    with open(OUT, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
        f.write("\n")
    print(OUT, len(rec["quant_cuda_calls"]), "symbols,", len(modules), "modules")


if __name__ == "__main__":
    main()
