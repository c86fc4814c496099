#!/usr/bin/env python3
"""bench.py - BASELINE.json's metric on BASELINE.json's config: LLaMA-7B w4-s45 decode tokens/s at batch 1
(QuantLinear layers), plus the per-layer HBM roofline fraction.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload llama7b-w4-s45] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one decode token's pass over the hot path: the 7 QuantLinearLUT matvecs (q, k, v, o, gate, up, down) of
each of the model's decoder layers, in model order, chained through their real shapes (x -> q,k,v ; v -> o ; o -> gate,up ;
gate -> down -> next layer's x), on synthetic random-init weights in the reference's buffer format (distinct per layer:
3.6 GB per token for 7B w4-s45, far beyond the 126 MB L2, so every step streams from HBM).  Attention, norms, rotary,
lm_head and the KV cache are NOT part of the step (they are not on the path this repo replaces) and that is stated in
`config`.  As `llama.py --include_sparse` always runs (llama.py:301-306), sparse layers use the hybrid symbol with
topX=10 dense rows that are zero (a checkpoint without them, llama.py:182).

  value  : tokens/s, device-timed, inputs resident in HBM, one CUDA-graph replay per step; --steps K timed steps in all, in
           --blocks (5) blocks of near-equal size, the MEDIAN per-step time of the blocks is reported (ms_per_step; block
           times in `blocks_ms`, their step counts in `block_steps`).  --dump-outputs DIR writes the last timed step's outputs.
  lut_fp16: the same measurement with the fp16 pair-table mode of the kernel (quant_cuda.set_lut_mode("fp16"), north_star's
           "per-channel fp16 LUT"); the headline `value` always uses the exact fp32 codebook.  `--lut fp16` makes it the only run.
  parity_check: outside the timed region, one sampled layer group per rank against the fp64 CPU oracle on the same buffers.
  e2e    : same metric through the public API (squeezellm_b200.runtime.GraphedDecodeStep over QuantLinearLUT.forward)
           with the token's activation coming from pinned host memory and the result read back every step.
  roofline: algorithmic bytes of all launches of the step / step time vs the measured HBM copy bandwidth.
  cpu_baseline / --impl reference: the reference has no CPU path; this is the restatement north_star names
           (unpack -> LUT gather -> fp16 W -> torch.matmul, + CSR + dense rows) on the box's host cores, on ONE decoder
           layer per step (bounded sample), extrapolated to the model's layer count.
  N > 1  : every QuantLinear is column-sharded N ways (qweight[:, c0:c1], LUT rows, CSR rows re-based) and the output
           vector is summed with one NCCL all-reduce per matvec (north_star); "scaling": "strong".
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: hidden, ffn, layers, bits, sparsity, topX
    "llama7b-w4-s45": dict(hidden=4096, ffn=11008, layers=32, bits=4, sparsity=0.0045, topX=10),
    "llama7b-w4-s0": dict(hidden=4096, ffn=11008, layers=32, bits=4, sparsity=0.0, topX=0),
    "llama7b-w3-s45": dict(hidden=4096, ffn=11008, layers=32, bits=3, sparsity=0.0045, topX=10),
    "llama13b-w4-s5": dict(hidden=5120, ffn=13824, layers=40, bits=4, sparsity=0.0005, topX=10),
    "llama65b-w3-s45": dict(hidden=8192, ffn=22016, layers=80, bits=3, sparsity=0.0045, topX=10),
}
MATS = [("q_proj", "hidden", "hidden"), ("k_proj", "hidden", "hidden"), ("v_proj", "hidden", "hidden"),
        ("o_proj", "hidden", "hidden"), ("gate_proj", "hidden", "ffn"), ("up_proj", "hidden", "ffn"),
        ("down_proj", "ffn", "hidden")]


def alg_bytes(bits, K, N, nnz, topx):
    """SURVEY.md 8(d): packed words + fp32 LUT + fp32 x + fp32 y (+ CSR cols/vals/rows) (+ dense rows)."""
    b = K // 32 * bits * N * 4 + N * (2 ** bits) * 4 + K * 4 + N * 4
    if nnz:
        b += nnz * 8 + (N + 1) * 4
    if topx:
        b += K * topx * 4 + topx * 4
    return b


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, bf16 copy read+write)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------------------------
# synthetic model in the reference's buffer format, generated on the device
# ------------------------------------------------------------------------------------------------------------------
def synth_matrix(bits, K, N, sparsity, topx, gen, dev, c0=0, c1=None):
    """Buffers of one QuantLinearLUT [K -> N]; columns [c0, c1) only (column shard) if given."""
    c1 = N if c1 is None else c1
    n = c1 - c0
    d = {}
    d["qweight"] = torch.randint(-2**31, 2**31 - 1, (K // 32 * bits, n), dtype=torch.int64, device=dev, generator=gen).to(torch.int32)
    # per-channel sorted centroids, scaled so that a matvec keeps |x| ~ O(1) through 224 chained layers
    d["lookup_table"] = torch.sort(torch.randn((n, 2 ** bits), device=dev, generator=gen) * (K ** -0.5), dim=1).values.contiguous()
    nnz = int(round(sparsity * K * n))
    if nnz:
        counts = torch.bincount(torch.randint(0, n, (nnz,), device=dev, generator=gen), minlength=n)
        rows = torch.zeros(n + 1, dtype=torch.int32, device=dev)
        rows[1:] = torch.cumsum(counts, 0).to(torch.int32)
        d["rows"] = rows
        d["cols"] = torch.randint(0, K, (nnz,), device=dev, generator=gen).to(torch.int32)
        d["vals"] = torch.randn(nnz, device=dev, generator=gen) * (0.5 * K ** -0.5)
    if topx and nnz:
        d["full_rows"] = torch.zeros((K, topx), device=dev)
        d["full_row_indices"] = torch.zeros(topx, dtype=torch.int32, device=dev)
    return d, nnz


def build_model(cfg, dev, rank, world, seed=0):
    from squeezellm_b200.quant import QuantLinearLUT
    gen = torch.Generator(device=dev).manual_seed(seed + 1000 * rank)
    layers, nbytes, nlaunch = [], 0, 0
    for li in range(cfg["layers"]):
        mods = {}
        for name, kin, kout in MATS:
            K, N = cfg[kin], cfg[kout]
            assert N % (4 * world) == 0, f"{name}: out_features {N} does not split into {world} shards of a multiple of 4"
            w = N // world
            d, nnz = synth_matrix(cfg["bits"], K, N, cfg["sparsity"], cfg["topX"], gen, dev, rank * w, (rank + 1) * w)
            m = QuantLinearLUT(cfg["bits"], K, w, False, include_sparse=nnz > 0, numvals=nnz, topX=cfg["topX"] if nnz else 0)
            for k, v in d.items():
                setattr(m, k, v)  # registered buffers: assignment keeps them buffers
            mods[name] = m
            nbytes += alg_bytes(cfg["bits"], K, w, nnz, cfg["topX"] if nnz else 0)
            nlaunch += 1
        layers.append(mods)
    return layers, nbytes, nlaunch


def make_step(layers, world, peer=None, keep=None):
    """Returns (step, run_layer).  step: x [hidden] -> x' [hidden], the 7 matvecs per decoder layer in model order (see module
    docstring).  run_layer(L, x) runs ONE decoder layer the same way and returns [(name, input, full-length output)] for the 7
    matvecs - what parity_check compares with the oracle (at N > 1: after the exchange, i.e. the vectors the next matvec reads).
    keep: a list that step() refills with run_layer's result for every layer, so that the 7 x layers output tensors of its last
    call (in a CUDA graph: of its last replay) stay readable."""
    QKV, GU = ("q_proj", "k_proj", "v_proj"), ("gate_proj", "up_proj")
    if world == 1:
        def run_layer(L, x):
            q, k, v = L["q_proj"](x), L["k_proj"](x), L["v_proj"](x)
            o = L["o_proj"](v)
            g, u = L["gate_proj"](o), L["up_proj"](o)
            d = L["down_proj"](g)
            return [("q_proj", x, q), ("k_proj", x, k), ("v_proj", x, v), ("o_proj", v, o), ("gate_proj", o, g), ("up_proj", o, u), ("down_proj", g, d)]
    else:
        import torch.distributed as dist
        from squeezellm_b200.sharding import exchange_stacked
        rank = dist.get_rank()
        bufs = {}

        def group_layer(L, names):
            g = L[names[0]]._sibling_group
            return g[0].layer if g is not None else None

        if peer is not None:
            # the kernel's finishing CTAs store their slice into every rank's arena over NVLink and wait for the peers': no collective
            def run(layer, x, slot, members):
                return peer.forward(layer, x, slot, members, layer.outfeatures // members * world)

            def stacked(L, names, x, slot):
                layer = group_layer(L, names)
                if layer is not None:
                    return run(layer, x, slot, len(names))
                return [run(L[n], x, slot + n, 1)[0] for n in names]

            def single(L, name, x, slot):
                return run(L[name], x, slot, 1)[0]
        else:
            def exchange(name, y, members):
                """this rank's (stacked) column shard -> zero-padded full-length vectors -> ONE all-reduce (north_star)."""
                w = y.shape[-1] // members
                if name not in bufs:
                    bufs[name] = torch.zeros((members, w * world), dtype=y.dtype, device=y.device)
                return exchange_stacked(y, members, rank, world, out=bufs[name])

            def stacked(L, names, x, slot):
                layer = group_layer(L, names)
                if layer is not None:  # q/k/v (gate/up) shards stacked: one launch, one all-reduce for all members
                    return exchange(names[0], layer(x), len(names))
                return [exchange(n, L[n](x), 1)[0] for n in names]

            def single(L, name, x, slot):
                return exchange(slot, L[name](x), 1)[0]

        def run_layer(L, x):
            q, k, v = stacked(L, QKV, x, "qkv")
            o = single(L, "o_proj", v, "o")
            g, u = stacked(L, GU, o, "gu")
            d = single(L, "down_proj", g, "d")
            return [("q_proj", x, q), ("k_proj", x, k), ("v_proj", x, v), ("o_proj", v, o), ("gate_proj", o, g), ("up_proj", o, u), ("down_proj", g, d)]

    def step(x):
        if keep is not None:
            keep.clear()
        for L in layers:
            outs = run_layer(L, x)
            if keep is not None:
                keep.append(outs)
            x = outs[-1][2]
        return x.clone() if world > 1 else x
    return step, run_layer


def seq_record_layer(seq, L, x, world=1):
    """Record the 7 matvecs of decoder layer L into the DecodeSequence `seq`, reading the SeqVec `x`; same wiring as make_step.
    Returns [(name, input SeqVec, output SeqVec)] in model order."""
    def stacked(names, xin):
        g = L[names[0]]._sibling_group
        if g is not None:
            y = seq.matvec(g[0].layer, xin, members=len(names))
            n = len(y) // len(names)
            return [y[i * n:(i + 1) * n] for i in range(len(names))]
        return [seq.matvec(L[n], xin) for n in names]
    q, k, v = stacked(("q_proj", "k_proj", "v_proj"), x)
    o = seq.matvec(L["o_proj"], v)
    g, u = stacked(("gate_proj", "up_proj"), o)
    d = seq.matvec(L["down_proj"], g)
    return [("q_proj", x, q), ("k_proj", x, k), ("v_proj", x, v), ("o_proj", v, o), ("gate_proj", o, g), ("up_proj", o, u), ("down_proj", g, d)]


def make_seq_step(layers, cfg, dev, mode, peer=None):
    """The whole token as ONE persistent launch (squeezellm_b200.runtime.DecodeSequence): returns (sequence, step(x) -> x')."""
    from squeezellm_b200.runtime import DecodeSequence
    seq = DecodeSequence(cfg["hidden"], dev, lut_mode=mode, peer=peer)
    x = seq.input
    for L in layers:
        x = seq_record_layer(seq, L, x, peer.world if peer is not None else 1)[-1][2]
    seq.compile(outputs=[x])

    def step(xin):
        if xin is not seq.x:
            seq.x.copy_(xin)
        return seq.replay()[0]
    return seq, step


def make_seq_run_layer(cfg, dev, quant_cuda, peer=None):
    """run_layer for parity_check: the sampled layer as a (one-layer) sequence, every matvec's full-length output exported."""
    from squeezellm_b200.runtime import DecodeSequence

    def run_layer(L, x):
        seq = DecodeSequence(cfg["hidden"], dev, lut_mode=quant_cuda.get_lut_mode(), peer=peer)
        rec = seq_record_layer(seq, L, seq.input, peer.world if peer is not None else 1)
        seq.compile(outputs=[r[2] for r in rec] + [r[1] for r in rec if r[1].item >= 0])
        seq.x.copy_(x)
        outs = [o.clone() for o in seq.replay()]
        torch.cuda.synchronize()
        if seq.error():
            print("[bench] parity_check: a bounded in-kernel wait of the sequence gave up; its vectors are incomplete", file=sys.stderr)
        ys, xs = outs[:len(rec)], iter(outs[len(rec):])
        return [(r[0], x if r[1].item < 0 else next(xs), y) for r, y in zip(rec, ys)]
    return run_layer


# ------------------------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc, self.thread = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        def pump():
            for line in self.proc.stdout:
                self.samples.append(line.strip())
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [t.strip() for t in s.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------
# CPU baseline (oracle port) - bench.py's only use of oracle/
# ------------------------------------------------------------------------------------------------------------------
def cpu_layer_sample(cfg, reps, seed=0):
    """Seconds per decoder layer for the 'dequant-to-fp16 + torch.matmul' CPU path, timed on host cores."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    mats = []
    for i, (name, kin, kout) in enumerate(MATS):
        L = orc.make_layer(cfg["bits"], cfg[kin], cfg[kout], sparsity=cfg["sparsity"], topX=cfg["topX"] if cfg["sparsity"] else 0, seed=seed + i)
        mats.append((L, orc.make_vec(cfg[kin], seed=i)))
    times, fused_times, mm_times = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        Ws = [orc.cpu_dequant_matmul(L, x, compute_dtype="float16")[1] for L, x in mats]
        times.append(time.perf_counter() - t0)
        if len(mm_times) < 3:  # (ii) of SURVEY 8(d): the same matmul (+CSR, dense rows) on the already dequantized fp16 matrices;
            t0 = time.perf_counter()   # three samples are enough, the reference arm must stay within minutes
            for (L, x), W in zip(mats, Ws):
                orc.cpu_dequant_matmul(L, x, predequantized=W, compute_dtype="float16")
            mm_times.append(time.perf_counter() - t0)
        del Ws
        t0 = time.perf_counter()
        for L, x in mats:
            orc.forward_f32_blocked(L, x)
        fused_times.append(time.perf_counter() - t0)
    cpu_layer_sample.matmul_only = mm_times
    return times, fused_times, orc.threads()


def leave(world):
    """Multi-rank exit.  destroy_process_group() can block for ever while CUDA graphs that captured NCCL kernels are alive
    (seen on 2 x B200: both ranks stuck after the JSON line was out), so ranks leave without tearing the communicator down."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        torch.cuda.synchronize()
        os._exit(0)


def metric_name(workload):
    if workload == "llama7b-w4-s45":
        return "LLaMA-7B w4-s45 decode tokens/s at batch=1 (QuantLinear layers); per-layer HBM GB/s vs peak"
    return f"{workload} decode tokens/s at batch=1 (QuantLinear layers)"


def base_config(args, cfg):
    return {"workload": args.workload, "batch": 1, "layers": cfg["layers"], "hidden": cfg["hidden"], "ffn": cfg["ffn"], "bits": cfg["bits"],
            "sparsity": cfg["sparsity"], "topX": cfg["topX"], "matvecs_per_step": len(MATS) * cfg["layers"],
            "scope": "QuantLinearLUT matvecs only; attention/norms/lm_head/KV cache excluded", "layers_overridden": bool(args.layers)}


def run_reference_arm(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nthr = host_threads()  # physical cores of one NUMA node, affinity pinned: the 128-thread oversubscribed run of round 1 varied 8x
    torch.set_num_threads(nthr)
    times, fused, thr = cpu_layer_sample(cfg, args.warmup + args.steps)
    t = times[args.warmup:]
    layer_s = statistics.median(t)
    per_tok = layer_s * cfg["layers"]
    val = 1.0 / per_tok
    fused_val = 1.0 / (statistics.median(fused[args.warmup:]) * cfg["layers"])
    sample = (f"each step = 1 of {cfg['layers']} decoder layers (7 matvecs: fp16 dequant + torch.matmul + CSR + dense rows), median of {len(t)} steps; "
              f"tokens/s = 1 / (layer time x {cfg['layers']}); ms_per_step is the MEASURED layer time")
    config = {**base_config(args, cfg), "launches_per_step": 0, "matvec_items_per_step": 0, "sibling_fusion": "n/a (CPU)", "l2": "n/a (CPU)", "parallelism": "host threads",
              "exchange": "none", "launch": "n/a (CPU)", "lut": "exact", "timing": f"median of {len(t)} steps", "layers_timed": 1}
    out = {"metric": metric_name(args.workload), "value": val, "unit": "tokens/s", "impl": "reference",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": layer_s * 1e3, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f16 weights x f16 activations (torch CPU matmul)", "data": "synthetic",
           "config": config,
           "cpu_baseline": {"value": val, "unit": "tokens/s", "cores": nthr, "kind": "port", "sample": sample,
                            "note": "the reference has no CPU path; this arm is the CPU restatement north_star names (oracle/), pinned to the physical cores of one NUMA node",
                            "layer_ms": layer_s * 1e3, "layers_per_token": cfg["layers"],
                            "fused_lookup_gemv_port_tokens_per_s": fused_val, "fused_port_threads": thr, "host_cpus": os.cpu_count(),
                            "matmul_only_on_predequantized_fp16_tokens_per_s": 1.0 / (min(cpu_layer_sample.matmul_only) * cfg["layers"])},
           "e2e": {"value": val, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="llama7b-w4-s45", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--layers", type=int, default=0, help="override the layer count (debug only; the JSON says so)")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N>1: how column shards are reassembled - p2p: stores into every rank's symmetric arena from inside the GEMV "
                         "kernel (falls back to nccl if symmetric memory is unavailable or the self-check fails); nccl: one all-reduce per launch")
    ap.add_argument("--launch", default="auto", choices=["auto", "seq", "graph"],
                    help="graph: one launch per (stacked) matvec, chained with PDL inside a CUDA graph; seq: the whole token as ONE persistent "
                         "kernel launch (runtime.DecodeSequence, csrc/lutgemv_seq.cuh; on several GPUs its input poll is the exchange); "
                         "auto (default): what measured faster - graph on one GPU (547 vs 481 tokens/s), seq on several (509 vs 371 at N=2)")
    ap.add_argument("--no-fuse", action="store_true", help="one launch per QuantLinearLUT (no q/k/v and gate/up sibling stacking)")
    ap.add_argument("--lut", default="both", choices=["both", "exact", "fp16"],
                    help="codebook precision: exact = fp32 as stored (headline), fp16 = pair tables; both = headline exact + a lut_fp16 object")
    ap.add_argument("--blocks", type=int, default=5,
                    help="the --steps timed steps are split into this many blocks (at most --steps) of near-equal size; the median "
                         "per-step time of the blocks is reported")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32): step_output "
                         "[hidden] and, with one launch per (stacked) matvec, every matvec's full-length output as <matvec name>.npy "
                         "[layers, out_features] (an evenly spaced subset of the layers if all of them would exceed 64 MB).  The inputs "
                         "are seeded; the default summation order is not, so two runs differ by fp16 roundings that grow along the "
                         "chain (LLaMA-7B w4-s45, two runs on one B200: up to 5e-4 of max|y| in layer 0, 4e-3 in layer 31)")
    ap.add_argument("--per-shape", action="store_true",
                    help="also time each of the step's launch types on its own (one CUDA graph of `layers` launches over every layer's "
                         "distinct weights, CUDA events) and add a per_shape object: us per launch, GB/s and roofline fraction per type")
    args = ap.parse_args()
    cfg = dict(WORKLOADS[args.workload])
    if args.layers:
        cfg["layers"] = args.layers
    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    assert args.steps >= 1 and args.blocks >= 1, "--steps and --blocks must be at least 1"

    if args.impl == "reference":
        run_reference_arm(args, cfg)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run for N>1)"
    assert torch.cuda.is_available(), "bench.py needs a CUDA device; there is no CPU fallback for the product path"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when the first communicator comes up; rank 0's stdout must carry exactly one
        # line (the JSON), so stdout points at stderr until the communicator exists
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    layers, nbytes, nmat = build_model(cfg, dev, rank, world)
    nlaunch = nmat
    if not args.no_fuse:
        # squeezellm_b200.fusion: siblings that read the same input run as one stacked launch (same packed words, same LUT rows)
        from squeezellm_b200.fusion import SiblingGroup, LLAMA_SIBLINGS
        for L in layers:
            for names in LLAMA_SIBLINGS:
                SiblingGroup([L[n] for n in names])
                nlaunch -= len(names) - 1
        torch.cuda.empty_cache()
    exchange_used, peer_used = "none", None
    use_seq = args.launch == "seq" or (args.launch == "auto" and world > 1)
    seq_peer = None
    if world > 1 and use_seq:
        from squeezellm_b200.sharding import PeerArena
        seq_peer = PeerArena(rank, world, dev)
    keep = [] if args.dump_outputs and not use_seq else None  # the sequence kernel hands out the step's output only
    if world > 1:
        import torch.distributed as dist
        step_nccl, run_layer_nccl = make_step(layers, world, keep=keep)
        run_layer = run_layer_nccl
        step, exchange_used = step_nccl, "nccl all-reduce per launch"
        if use_seq:
            exchange_used = ("sequence kernel: strip owners store tagged result words into every rank's arena over NVLink; the next matvec's "
                             "input poll is the exchange (no collective)")
        elif args.exchange == "p2p":
            why, ok, step_p2p = None, 0.0, None
            try:
                from squeezellm_b200.sharding import PeerExchange
                peer = PeerExchange(rank, world, dev)
                step_p2p, run_layer_p2p = make_step(layers, world, peer, keep=keep)
                xs = torch.randn(cfg["hidden"], device=dev, generator=torch.Generator(device=dev).manual_seed(7)).half()
                a, b = step_p2p(xs).float(), step_nccl(xs).float()
                torch.cuda.synchronize()
                # start-up smoke check only (does the exchange deliver at all?); the parity statement is parity_check, against the fp64 oracle
                good = (not peer.error()) and bool(torch.isfinite(a).all()) and bool((a - b).abs().max() <= 2e-2 * b.abs().max().clamp_min(1e-3))
                ok = 1.0 if good else 0.0
                if not good:
                    why = "self-check against the NCCL path failed"
            except Exception as e:  # noqa: BLE001 - symmetric memory unavailable: keep the NCCL path
                why = f"{type(e).__name__}: {e}"
            vote = torch.tensor([ok], device=dev)
            dist.all_reduce(vote, op=dist.ReduceOp.MIN)  # every rank takes the same decision
            if vote.item() == 1.0:
                step, exchange_used, peer_used = step_p2p, "in-kernel stores to every rank's symmetric arena over NVLink (no collective)", peer
                run_layer = run_layer_p2p
            elif why or rank == 0:
                print(f"[bench] rank {rank}: p2p exchange not used ({why or 'another rank declined'}); falling back to NCCL", file=sys.stderr)
    else:
        step, run_layer = make_step(layers, world, keep=keep)
    x0 = torch.randn(cfg["hidden"], device=dev, generator=torch.Generator(device=dev).manual_seed(99)).half()  # same on every rank

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    from squeezellm_b200.quant import quant_cuda
    from squeezellm_b200.runtime import GraphedDecodeStep
    xh = torch.randn(cfg["hidden"], generator=torch.Generator().manual_seed(98)).half().pin_memory()
    sampler = ClockSampler(torch.cuda.current_device() if "CUDA_VISIBLE_DEVICES" not in os.environ else local)

    def measure(lut_mode, sample_clocks, dump=False):
        """One full measurement (device-resident blocks, then end to end from host memory) with the given codebook mode.
        The mode is baked into the graph at capture time (the kernel variant is chosen per launch).
        dump: also return the outputs of the last timed step (name -> float32 host tensor)."""
        quant_cuda.set_lut_mode(lut_mode)
        graphed = True
        seq = None
        try:
            if use_seq:
                seq, _ = make_seq_step(layers, cfg, dev, lut_mode, peer=seq_peer)
                seq.x.copy_(x0)
                runner = GraphedDecodeStep(lambda x: seq.replay()[0], seq.x, warmup=3, static_input=True)
            else:
                runner = GraphedDecodeStep(step, x0, warmup=3)
        except Exception as e:  # e.g. NCCL refusing capture: fall back to eager launches, and say so
            if world == 1:
                raise
            graphed, runner = False, None
            print(f"[bench] graph capture failed on rank {rank}: {e}; timing eager", file=sys.stderr)
            torch.cuda.synchronize()

        def one_step():
            return runner.replay() if graphed else step(x0)

        for _ in range(args.warmup):
            one_step()
        barrier()
        warm_timeout = False
        if seq is not None and seq.error():  # start-up skew between ranks (> 2 s) during warm-up: note it, clear it, go on aligned
            warm_timeout = True
            seq.reset_error()
            print(f"[bench] rank {rank}: a bounded in-kernel wait timed out during warm-up (start-up skew); cleared", file=sys.stderr)
            barrier()
        if sample_clocks and rank == 0:
            sampler.start()
        nblocks = min(args.blocks, args.steps)
        sizes = [args.steps // nblocks + (b < args.steps % nblocks) for b in range(nblocks)]  # args.steps timed steps in all
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(nblocks + 1)]
        evs[0].record()
        for b in range(nblocks):
            for _ in range(sizes[b]):
                y = one_step()
            evs[b + 1].record()
        barrier()
        blocks = [evs[b].elapsed_time(evs[b + 1]) for b in range(nblocks)]
        clocks = sampler.stop() if (sample_clocks and rank == 0) else None
        outputs = None
        if dump:  # read before the end-to-end run below overwrites the graph's buffers
            outputs = {"step_output": y.float().cpu()}
            for j, name in enumerate([o[0] for o in keep[0]] if keep else []):
                outputs[name] = torch.stack([outs[j][2].reshape(-1) for outs in keep]).float().cpu()
        # end to end from host memory through the public API
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if graphed:
            for _ in range(args.warmup):
                runner(xh)
            barrier()
            ev0.record()
            for _ in range(args.steps):
                runner(xh)
            ev1.record()
        else:
            yh = torch.empty(cfg["hidden"], dtype=torch.float16).pin_memory()
            for _ in range(args.warmup):
                yh.copy_(step(xh.to(dev, non_blocking=True)))
            barrier()
            ev0.record()
            for _ in range(args.steps):
                yh.copy_(step(xh.to(dev, non_blocking=True)))
            ev1.record()
        barrier()
        e2e_ms = ev0.elapsed_time(ev1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor(blocks + [e2e_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)  # every block: max over ranks
            blocks, e2e_ms = t.tolist()[:-1], t.tolist()[-1]
        ms_step = statistics.median([ms / n for ms, n in zip(blocks, sizes)])
        quant_cuda.set_lut_mode("exact")
        seq_timeout = False
        if seq is not None:
            seq_timeout = bool(seq.error())  # a bounded in-kernel wait gave up during the timed run: the numbers of this run are void
            if seq_timeout:
                print(f"[bench] rank {rank}: the sequence kernel's error word is set after the timed region - THIS RUN'S NUMBERS ARE VOID", file=sys.stderr)
            del runner, seq
            torch.cuda.empty_cache()
        return {"seq_timeout": seq_timeout, "warm_timeout": warm_timeout, "ms_step": ms_step, "e2e_ms_step": e2e_ms / args.steps, "blocks_ms": [round(b, 4) for b in blocks],
                "block_steps": sizes, "graphed": graphed, "clocks": clocks, "outputs": outputs}

    def per_shape(lut_mode):
        """us per launch for each launch type of the step: a graph with one launch per decoder layer (every layer's own weights, LUT
        and outlier arrays, so nothing is L2-resident), replayed 3 + 10 times, device-timed."""
        quant_cuda.set_lut_mode(lut_mode)
        peak = peaks()[0]
        groups = [("qkv" if not args.no_fuse else "q", ("q_proj", "k_proj", "v_proj") if not args.no_fuse else ("q_proj",), "hidden"),
                  ("o", ("o_proj",), "hidden"), ("gate_up" if not args.no_fuse else "gate", ("gate_proj", "up_proj") if not args.no_fuse else ("gate_proj",), "hidden"),
                  ("down", ("down_proj",), "ffn")]
        out = {}
        for gname, names, kin in groups:
            xin = torch.randn(cfg[kin], device=dev).half()

            def run():
                for L in layers:
                    for n in names:
                        L[n](xin)
            st = torch.cuda.Stream()
            st.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(st):
                run(); run()
            torch.cuda.current_stream().wait_stream(st)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=st):
                run()
            for _ in range(3):
                g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            us = e0.elapsed_time(e1) * 1e3 / (10 * len(layers))
            nb = 0
            for n in names:
                m = layers[0][n]
                nnz = int(m.vals.numel()) if hasattr(m, "vals") and m.vals is not None and m.include_sparse else 0
                nb += alg_bytes(cfg["bits"], m.infeatures, m.outfeatures, nnz, cfg["topX"] if nnz else 0)
            if not args.no_fuse and len(names) > 1:   # stacked: one x read and one launch for all members
                nb -= (len(names) - 1) * cfg[kin] * 4
            out[gname] = {"us_per_launch": us, "algorithmic_bytes": nb, "GBps": nb / us / 1e3, "frac": nb / us / 1e3 / peak,
                          "K": cfg[kin], "N": sum(layers[0][n].outfeatures for n in names)}
        quant_cuda.set_lut_mode("exact")
        return out

    head_mode = "fp16" if args.lut == "fp16" else "exact"
    shapes = None
    if args.per_shape and world == 1:
        shapes = {"exact": per_shape("exact"), "fp16": per_shape("fp16")}
    main_run = measure(head_mode, True, dump=bool(args.dump_outputs))
    extra_run = measure("fp16", False) if args.lut == "both" else None

    # ---- parity: one sampled layer group per rank against the fp64 oracle on the same buffers (outside every timed region) ----------
    if use_seq:
        run_layer = make_seq_run_layer(cfg, dev, quant_cuda, peer=seq_peer)
    parity = parity_check(layers, run_layer, cfg, rank, world, dev, quant_cuda)
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([parity["max_rel_err"], parity["fp16_max_norm_err"]], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        parity["max_rel_err"], parity["fp16_max_norm_err"] = t.tolist()
        parity["ranks"] = world

    if main_run.get("seq_timeout") or (extra_run or {}).get("seq_timeout"):
        parity["sequence_wait_timeout_in_timed_region"] = True
        parity["ok"] = False
    if main_run.get("warm_timeout"):
        parity["sequence_wait_timeout_during_warmup_cleared"] = True
    if peer_used is not None and peer_used.error():  # a bounded in-kernel wait gave up: the numbers of this run are not valid
        exchange_used += " - ERROR: a peer wait timed out during this run"
        print(f"[bench] rank {rank}: exchange error word is set", file=sys.stderr)
    if quant_cuda.workspace_error():
        print(f"[bench] rank {rank}: the fused-path workspace error word is set (a bounded in-kernel wait timed out)", file=sys.stderr)
        parity["workspace_error"] = True
    if world > 1:
        import torch.distributed as dist
        tot = torch.tensor([float(nbytes)], device=dev, dtype=torch.float64)
        dist.all_reduce(tot)
        nbytes_all = tot.item()
    else:
        nbytes_all = float(nbytes)

    if rank != 0:
        leave(world)
        return

    ms_step = main_run["ms_step"]
    tok_s = 1e3 / ms_step
    e2e_tok_s = 1e3 / main_run["e2e_ms_step"]
    graphed = main_run["graphed"]
    peak, peak_src = peaks()
    achieved = nbytes / (ms_step * 1e-3) / 1e9  # per GPU: this rank's bytes over the step time
    traffic = None
    if world == 1:  # measured with ncu on the default single-GPU command (profiles/); not meaningful for column shards
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.workload)
        except Exception:
            pass
    kern = f"{'lutgemv_seq_kernel' if use_seq else 'lutgemv2_kernel'}<{cfg['bits']}, {'fp16 pair table' if head_mode == 'fp16' else 'exact fp32 table'}{'' if use_seq else ', fused'}>"
    launches = 2 if use_seq else nlaunch  # seq: token counter + the persistent kernel
    out = {
        "metric": metric_name(args.workload),
        "value": tok_s, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": ("f32 accumulate (fp16-rounded LUT x fp16 activations, exact products, fp16 outputs)" if head_mode == "fp16" else
                  "f32 accumulate (fp32 LUT x fp16->fp32 activations, fp16 outputs)"), "data": "synthetic",
        "config": {**base_config(args, cfg), "launches_per_step": launches, "matvec_items_per_step": nlaunch,
                   "sibling_fusion": "q/k/v and gate/up stacked (squeezellm_b200.fusion)" if nlaunch != nmat else "off",
                   "l2": f"{nbytes_all / 1e9:.2f} GB of distinct weights per step >> 126 MB L2 (inputs larger than L2)",
                   "parallelism": "single GPU" if world == 1 else f"column-sharded x{world}, {nlaunch} launches per step", "exchange": exchange_used,
                   "launch": ("one CUDA-graph replay per step" if graphed else "eager launches (graph capture unavailable)") +
                             (": ONE persistent kernel runs all matvecs of the token (runtime.DecodeSequence)" if use_seq else ": one PDL-chained launch per (stacked) matvec"),
                   "lut": head_mode, "timing": f"{args.steps} timed steps in {len(main_run['block_steps'])} blocks, median per-step time of the blocks",
                   "layers_timed": cfg["layers"]},
        "blocks_ms": main_run["blocks_ms"], "block_steps": main_run["block_steps"],
        "e2e": {"value": e2e_tok_s, "unit": "tokens/s", "h2d_bytes_per_step": cfg["hidden"] * 2, "d2h_bytes_per_step": cfg["hidden"] * 2,
                "api": ("squeezellm_b200.runtime.GraphedDecodeStep over runtime.DecodeSequence (QuantLinearLUT modules)" if use_seq else
                        "squeezellm_b200.runtime.GraphedDecodeStep over QuantLinearLUT.forward") if graphed else "QuantLinearLUT.forward eager"},
        "gpu_launches": launches * args.steps,
        "clocks": main_run["clocks"],
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "peak_source": peak_src, "kernel": kern,
                     "algorithmic_bytes_per_step_per_gpu": nbytes, "frac_of_nominal_8000": achieved / 8000.0},
        "parity_check": parity,
    }
    if shapes is not None:
        out["per_shape"] = shapes
    if extra_run is not None:
        a2 = nbytes / (extra_run["ms_step"] * 1e-3) / 1e9
        out["lut_fp16"] = {"value": 1e3 / extra_run["ms_step"], "unit": "tokens/s", "ms_per_step": extra_run["ms_step"],
                           "e2e": 1e3 / extra_run["e2e_ms_step"], "blocks_ms": extra_run["blocks_ms"],
                           "roofline_frac": a2 / peak, "achieved_GBps": a2,
                           "note": "same graph with the kernel's fp16 pair-table mode (centroids rounded to fp16, fp16 x fp16 -> fp32 FMAs); "
                                   "max-norm error vs the fp64 oracle in parity_check.fp16_max_norm_err"}
    if not args.no_cpu_baseline:
        torch.set_num_threads(host_threads())
        times, fused, thr = cpu_layer_sample(cfg, 2)
        per_tok = min(times) * cfg["layers"]
        out["cpu_baseline"] = {"value": 1.0 / per_tok, "unit": "tokens/s", "cores": torch.get_num_threads(), "kind": "port",
                               "sample": f"1 of {cfg['layers']} decoder layers (7 matvecs), best of 2, fp16 dequant + torch.matmul (+CSR, dense rows), x{cfg['layers']}",
                               "layer_ms": min(times) * 1e3,
                               "fused_lookup_gemv_port_tokens_per_s": 1.0 / (min(fused) * cfg["layers"]), "fused_port_threads": thr,
                               "matmul_only_on_predequantized_fp16_tokens_per_s": 1.0 / (min(cpu_layer_sample.matmul_only) * cfg["layers"]),
                               "host_cpus": os.cpu_count()}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, main_run["outputs"])
    print(json.dumps(out), flush=True)
    leave(world)


DUMP_BYTES = 64 << 20


def dump_outputs(path, outputs):
    """outputs: name -> float32 tensor on the host; [layers, N] arrays keep an evenly spaced subset of their rows (first and last
    layer included) if all of them would exceed DUMP_BYTES."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    per_layer = sum(v[0].numel() * 4 for k, v in outputs.items() if k != "step_output")
    nlayers = max((len(v) for k, v in outputs.items() if k != "step_output"), default=0)
    nrows = min(nlayers, (DUMP_BYTES - outputs["step_output"].numel() * 4) // per_layer) if per_layer else 0
    rows = np.unique(np.linspace(0, nlayers - 1, nrows).round().astype(np.int64))
    for name, v in outputs.items():
        a = v.numpy().astype(np.float32)
        if name != "step_output":
            a = a[rows]
        np.save(os.path.join(path, f"{name}.npy"), a)


def parity_check(layers, run_layer, cfg, rank, world, dev, quant_cuda):
    """One sampled decoder layer (the same on every rank, so that the exchange is part of what is checked): its 7 matvecs run exactly as
    in the timed step (run_layer: same module objects, sibling stacking, the exchange at N > 1) and every full-length output vector
    is compared with the fp64 oracle evaluated on the same buffers and the same fp16 inputs.  At N > 1 each rank evaluates the
    oracle on its own column shard and the slices are all-gathered, so every rank checks every rank's columns as delivered to it.
    max_rel_err: exact codebook, the strict per-element metric of tests/util.py (floor 1 % of max|y|), tolerance 1e-3 (north_star).
    fp16_max_norm_err: fp16 pair-table mode, max|y - o| / max|o| (tests/test_lut_fp16.py says why that mode is stated in the max norm)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle as orc
    li = len(layers) // 2
    L = layers[li]

    def rel_err(a, b):
        den = np.maximum(np.abs(b), 1e-2 * max(np.abs(b).max(), 1e-30))
        return float((np.abs(a - b) / den).max())

    def to_oracle(m):
        d = dict(bits=m.bits, infeatures=m.infeatures, outfeatures=m.outfeatures, bias=None)
        for k in ("qweight", "lookup_table", "rows", "cols", "vals", "full_rows", "full_row_indices"):
            d[k] = getattr(m, k).detach().cpu().numpy() if hasattr(m, k) and getattr(m, k) is not None else None
        return d

    x = torch.randn(cfg["hidden"], device=dev, generator=torch.Generator(device=dev).manual_seed(4321)).half()  # same on every rank
    worst = {"exact": 0.0, "fp16": 0.0}
    for mode in ("exact", "fp16"):
        quant_cuda.set_lut_mode(mode)
        outs = run_layer(L, x)
        torch.cuda.synchronize()
        for name, xin, y in outs:
            want = orc.forward_f64(to_oracle(L[name]), xin.float().cpu().numpy().reshape(1, -1)).reshape(-1)  # this rank's columns
            if world > 1:
                import torch.distributed as dist
                parts = [torch.empty(want.shape[0], dtype=torch.float64, device=dev) for _ in range(world)]
                dist.all_gather(parts, torch.from_numpy(want).to(dev))
                want = torch.cat(parts).cpu().numpy()
            got = y.float().cpu().numpy().reshape(-1)
            if mode == "exact":
                worst[mode] = max(worst[mode], rel_err(got, want))
            else:
                worst[mode] = max(worst[mode], float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)))
    quant_cuda.set_lut_mode("exact")
    return {"max_rel_err": worst["exact"], "tol": 1e-3, "fp16_max_norm_err": worst["fp16"], "fp16_tol": 1e-3,
            "metric": "exact: max_i |y_i - o_i| / max(|o_i|, 1e-2 max|o|); fp16: max|y - o| / max|o|; o = fp64 oracle, y = fp16 output as the next matvec reads it",
            "sample": f"decoder layer {li} of {len(layers)}, all 7 matvecs, run exactly as in the timed step" + (", after the exchange" if world > 1 else ""),
            "ok": bool(worst["exact"] <= 1e-3 and worst["fp16"] <= 1e-3)}


def host_threads():
    """Threads for the CPU arm: the physical cores of ONE NUMA node (hyper-threads and the second socket only add noise here)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except Exception:
        cpus = list(range(os.cpu_count() or 1))
    node0 = set()
    try:
        for part in open("/sys/devices/system/node/node0/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            node0.update(range(int(a), int(b or a) + 1))
    except Exception:
        node0 = set(cpus)
    phys = {}
    for c in cpus:
        if c not in node0:
            continue
        try:
            core = open(f"/sys/devices/system/cpu/cpu{c}/topology/core_id").read().strip()
        except Exception:
            core = str(c)
        phys.setdefault(core, c)
    chosen = sorted(phys.values()) or cpus
    try:
        os.sched_setaffinity(0, chosen)
    except Exception:
        pass
    os.environ["OMP_NUM_THREADS"] = str(len(chosen))
    return len(chosen)


if __name__ == "__main__":
    main()
