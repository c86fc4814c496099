"""CPU tests of the sequence API's host side: SeqVec slicing, arena sizing and the argument validation of sqllm_sequence_create
(include/sqllm_b200.h; everything is checked before the first CUDA call, so it runs without a GPU)."""
import ctypes

import pytest

from util import Args, load_lib


class SeqItem(ctypes.Structure):  # mirrors sqllm_seq_item
    _fields_ = [("a", Args), ("bias", ctypes.c_void_p), ("x_from", ctypes.c_int), ("x_offset", ctypes.c_int), ("x_ext", ctypes.c_void_p),
                ("y", ctypes.c_void_p), ("members", ctypes.c_int), ("out_features_full", ctypes.c_int)]


class SeqOptions(ctypes.Structure):  # mirrors sqllm_seq_options
    _fields_ = [("lut_mode", ctypes.c_int), ("world", ctypes.c_int), ("rank", ctypes.c_int), ("arena", ctypes.c_void_p),
                ("arena_bytes", ctypes.c_size_t), ("peer_base", ctypes.c_void_p), ("n_export", ctypes.c_int),
                ("export_items", ctypes.c_void_p), ("export_dst", ctypes.c_void_p), ("trace", ctypes.c_void_p)]


def _item(bits=4, K=256, N=256, x_from=-1, x_offset=0, members=1, nfull=0):
    it = SeqItem()
    it.a = Args(bits=bits, in_features=K, out_features=N, batch=1, qweight=4096, lookup_table=8192, vec=0, mul=0)
    it.x_from, it.x_offset, it.x_ext, it.members, it.out_features_full = x_from, x_offset, (16384 if x_from < 0 else 0), members, nfull or N
    return it


def _create(lib, items, **opt):
    arr = (SeqItem * len(items))(*items)
    o = SeqOptions(lut_mode=0, world=opt.get("world", 1), rank=opt.get("rank", 0))
    h = ctypes.c_void_p()
    rc = lib.sqllm_sequence_create(arr, len(items), ctypes.byref(o), ctypes.byref(h))
    return rc, lib.sqllm_last_error().decode()


def test_seqvec_slicing():
    from squeezellm_b200.runtime import SeqVec
    v = SeqVec(3, 0, 12288)
    w = v[8192:12288]
    assert (w.item, w.offset, len(w)) == (3, 8192, 4096)
    u = w[1024:2048]
    assert (u.item, u.offset, len(u)) == (3, 9216, 1024)
    with pytest.raises(AssertionError):
        v[::2]


def test_arena_bytes_rounding():
    lib = load_lib()
    lib.sqllm_sequence_arena_bytes.restype = ctypes.c_size_t
    items = (SeqItem * 3)(_item(N=256), _item(N=4096 + 4, x_from=0), _item(N=64, x_from=1, members=1, nfull=512))
    # 4 bytes per output element (fp16 value + 16-bit tag), each vector rounded up to 128 bytes
    assert lib.sqllm_sequence_arena_bytes(items, 3) == 1024 + (16400 + 127) // 128 * 128 + 2048
    assert lib.sqllm_sequence_arena_bytes(None, 0) == 0


@pytest.mark.parametrize("items,kw,needle", [
    ([], {}, "null / empty"),
    ([_item(), _item(bits=3, x_from=0)], {}, "one sequence, one width"),
    ([_item(), _item(x_from=1)], {}, "must name an earlier item"),
    ([_item(N=256), _item(K=256, x_from=0, x_offset=2)], {}, "reads ["),          # offset not a multiple of 4
    ([_item(N=256), _item(K=512, x_from=0)], {}, "reads ["),                      # reads past the producer's vector
    ([_item(N=32)], {}, "out_features=32 <"),
    ([_item(N=256, members=3)], {}, "members of a multiple of 4"),
    ([_item()], {"world": 2, "rank": 0}, "peer-visible arena"),
    ([_item()], {"world": 2, "rank": 5}, "bad world / rank"),
])
def test_create_rejects_bad_arguments(items, kw, needle):
    lib = load_lib()
    rc, msg = _create(lib, items, **kw) if items else (lib.sqllm_sequence_create(None, 0, None, None), lib.sqllm_last_error().decode())
    assert rc == -1 and needle in msg, (rc, msg)


@pytest.mark.parametrize("topX,N,needle", [(129, 128, "MAX_TOPX_FUSED"), (10, 262148, "MAX_N_FUSED")])
def test_matvec_rejects_layers_past_the_fused_limits(topX, N, needle):
    """DecodeSequence.matvec refuses, when the layer is recorded, what the sequence kernel cannot run (not later, inside compile)."""
    from squeezellm_b200.quant import QuantLinearLUT, quant_cuda
    from squeezellm_b200.runtime import DecodeSequence
    assert (quant_cuda.MAX_TOPX_FUSED, quant_cuda.MAX_N_FUSED) == (128, 262144)
    seq = DecodeSequence(64, "cpu")
    ok = QuantLinearLUT(4, 64, 128, False, include_sparse=True, numvals=1, topX=quant_cuda.MAX_TOPX_FUSED)
    seq.matvec(ok, seq.input)
    with pytest.raises(ValueError, match=needle):
        seq.matvec(QuantLinearLUT(4, 64, N, False, include_sparse=True, numvals=1, topX=topX), seq.input)
