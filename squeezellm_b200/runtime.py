"""Decode-time runtime helpers around QuantLinearLUT (public API).

`GraphedDecodeStep` turns a token step made of QuantLinearLUT calls (224 of them per LLaMA-7B token, each a
~2-10 us kernel) into ONE CUDA-graph replay with static device buffers and pinned host staging:

    runner = GraphedDecodeStep(step_fn, example_x)      # captures step_fn(x_dev) -> y_dev
    y_host = runner(x_host)                             # H2D copy, replay, D2H copy, all on one stream

It exists because the reference drives the path from Python one launch at a time on the legacy stream
(llama.py:226-234, quant_cuda_kernel.cu:147), which costs more host time per call than the kernels take on a
B200; our kernels launch on the current stream precisely so that they can be captured.
"""
import torch


class GraphedDecodeStep:
    def __init__(self, step_fn, example_x, warmup=3, static_input=False):
        """static_input=True: `example_x` itself is the static input buffer (a DecodeSequence's `x`), not a clone of it."""
        assert example_x.is_cuda, "example_x must be a CUDA tensor (static input buffer is cloned from it)"
        self.step_fn = step_fn
        self.x_dev = example_x if static_input else example_x.clone()
        self.x_host = torch.empty(example_x.shape, dtype=example_x.dtype, pin_memory=True)
        self.stream = torch.cuda.Stream()
        self.stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.stream):
            for _ in range(warmup):  # also sizes the per-stream fused-path workspace before capture
                y = step_fn(self.x_dev)
        torch.cuda.current_stream().wait_stream(self.stream)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph, stream=self.stream):
            self.y_dev = step_fn(self.x_dev)
        self.y_host = torch.empty(self.y_dev.shape, dtype=self.y_dev.dtype, pin_memory=True)
        self.h2d_bytes = self.x_host.numel() * self.x_host.element_size()
        self.d2h_bytes = self.y_host.numel() * self.y_host.element_size()

    def replay(self):
        """Device-only: replay on the current stream with whatever is in the static input buffer."""
        self.graph.replay()
        return self.y_dev

    def __call__(self, x_host):
        """End to end from host memory: pinned H2D, replay, pinned D2H, synchronise; returns the pinned host result."""
        self.x_host.copy_(x_host)
        self.x_dev.copy_(self.x_host, non_blocking=True)
        self.graph.replay()
        self.y_host.copy_(self.y_dev, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self.y_host


class SeqVec:
    """A vector inside a DecodeSequence: the token's input (item -1) or (a slice of) the output of one of its matvecs."""

    def __init__(self, item, offset, length):
        self.item, self.offset, self.length = item, offset, length

    def __getitem__(self, sl):
        assert isinstance(sl, slice) and sl.step in (None, 1), "SeqVec supports contiguous slices only"
        a, b, _ = sl.indices(self.length)
        return SeqVec(self.item, self.offset + a, max(0, b - a))

    def __len__(self):
        return self.length


class DecodeSequence:
    """A token step recorded as a list of dependent QuantLinearLUT matvecs and run as ONE persistent kernel launch
    (csrc/lutgemv_seq.cuh): the weight stream never stops between two matvecs and results travel from one matvec to the
    next as self-validating tagged words - no launch, no grid barrier in between.

        seq = DecodeSequence(hidden, device)                  # seq.x: static fp16 input buffer [hidden]
        qkv = seq.matvec(stacked_qkv_layer, seq.input)        # -> SeqVec over the full output
        o   = seq.matvec(o_proj, qkv[2 * hidden:3 * hidden])
        ...
        seq.compile(outputs=[d])                              # d: the SeqVec whose plain fp16 copy is wanted
        y = seq.replay()[0]                                   # run on the current stream (CUDA-graph capturable)

    It replaces the per-layer launch loop of the reference's decode (llama.py:226-234) for the QuantLinear layers; whatever
    sits between them in a real model (attention, norms) has to run as its own launches, i.e. a model is cut into sequences
    at those points.  Layers must be QuantLinearLUT modules of one bit width, on one device, used with fp16 activations.
    On several GPUs pass `peer` (sharding.PeerArena): every layer is this rank's column shard."""

    def __init__(self, in_features, device, lut_mode=None, peer=None):
        self.device = torch.device(device)
        self.x = torch.zeros(in_features, dtype=torch.float16, device=self.device)
        self.input = SeqVec(-1, 0, in_features)
        self._items, self._lens, self._keep = [], [], []
        self._handle, self.outputs, self._out_vecs = None, [], []
        self.lut_mode = lut_mode
        self.peer = peer

    def matvec(self, layer, x, members=1):
        """Record y = layer(x).  `members`: on several GPUs, how many equal column shards `layer` stacks (q/k/v: 3)."""
        assert self._handle is None, "sequence already compiled"
        assert isinstance(x, SeqVec) and x.length == layer.infeatures, f"input has {len(x)} elements, layer wants {layer.infeatures}"
        assert x.item < len(self._items)
        world = self.peer.world if self.peer is not None else 1
        assert layer.outfeatures % members == 0
        nfull = layer.outfeatures // members * world
        rows, cols, vals, fr, fri = layer._sparse_args()
        from .quant import MAX_N_FUSED, MAX_TOPX_FUSED
        topX = fr.shape[1] if fr is not None else 0
        if topX > MAX_TOPX_FUSED:
            raise ValueError(f"DecodeSequence: layer has {topX} dense rows; the sequence kernel takes at most MAX_TOPX_FUSED = {MAX_TOPX_FUSED}")
        if layer.outfeatures > MAX_N_FUSED:
            raise ValueError(f"DecodeSequence: layer has out_features = {layer.outfeatures}; the sequence kernel takes at most "
                             f"MAX_N_FUSED = {MAX_N_FUSED}")
        self._items.append((layer.qweight, layer.lookup_table, layer.bits, layer.bias, rows, cols, vals, fr, fri,
                            x.item, x.offset, self.x if x.item < 0 else None, members, nfull))
        self._keep.append(layer)
        self._lens.append(members * nfull)
        return SeqVec(len(self._items) - 1, 0, members * nfull)

    def compile(self, outputs):
        from .quant import quant_cuda
        assert self._handle is None and self._items
        mode = self.lut_mode or quant_cuda.get_lut_mode()
        exports, bufs = [], {}
        for v in outputs:
            assert v.item >= 0, "the input is not an output"
            if v.item not in bufs:
                bufs[v.item] = torch.zeros(self._lens[v.item], dtype=torch.float16, device=self.device)
                exports.append((v.item, bufs[v.item]))
        self.outputs = [bufs[v.item][v.offset:v.offset + v.length] for v in outputs]
        with torch.cuda.device(self.device):
            if self.peer is not None:
                arena, peer_base = self.peer.arena_for(quant_cuda.sequence_arena_bytes(self._lens))
                self._handle = quant_cuda.sequence_create(self._items, exports, mode, self.peer.world, self.peer.rank, arena, peer_base)
                self._arena = arena
            else:
                self._handle = quant_cuda.sequence_create(self._items, exports, mode)
        self._exports = exports
        self._quant_cuda = quant_cuda
        return self

    def replay(self):
        """Run on the current stream with whatever is in `self.x`; returns the output views (static buffers)."""
        self._quant_cuda.sequence_run(self._handle)
        return self.outputs

    def error(self):
        """True if a bounded in-kernel wait (2 s) ever gave up: a result since then is incomplete.  Synchronises the current stream."""
        return self._quant_cuda.sequence_error(self._handle)

    def check(self):
        if self.error():
            raise RuntimeError("DecodeSequence: an in-kernel wait timed out (2 s) - on several GPUs a rank was late or absent; results since then "
                               "are incomplete.  Bring the ranks together (barrier) and call reset_error() on every rank.")

    def reset_error(self):
        self._quant_cuda.sequence_reset_error(self._handle)

    def __del__(self):
        try:
            if self._handle is not None:
                self._quant_cuda.sequence_destroy(self._handle)
                self._handle = None
        except Exception:
            pass
