"""CPU tests of the C-ABI library: it loads, exports every declared symbol, its host-side logic
(graph reader, glibc rand / random_shuffle restatement) matches the golden fixtures, and the compute
entry points fail loudly without a CUDA device (no CPU fallback)."""
import ctypes as C
import os

import numpy as np
import pytest

from ppo_cpp_b200 import _lib, core
from ppo_cpp_b200.meta_graph import TENSOR_ORDER, parse_meta_txt, write_meta_txt


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = _lib.declared_symbols()
    assert len(names) >= 45
    for n in names:
        assert hasattr(lib, n), n
    assert lib.ppo_abi_version() == 1


def test_tensor_names_follow_graph_gradient_order():
    lib = _lib.load()
    assert lib.ppo_core_num_tensors() == 15
    assert [lib.ppo_core_tensor_name(i).decode() for i in range(15)] == TENSOR_ORDER


def test_host_rand_bit_exact(kat):
    for seed, vals in kat["glibc"]["rand"].items():
        assert core.host_rand(int(seed), len(vals)).tolist() == vals


def test_host_random_shuffle_bit_exact(kat):
    for key, perms in kat["glibc"]["shuffle"].items():
        seed, n, epochs = (int(x) for x in key.split("_"))
        assert core.host_random_shuffle(seed, n, epochs).tolist() == perms


def test_host_rand_matches_live_libc():
    libc = C.CDLL("libc.so.6")
    libc.rand.restype = C.c_int
    libc.srand(987654321)
    assert core.host_rand(987654321, 5000).tolist() == [libc.rand() for _ in range(5000)]


def test_meta_parse_written_graph(tmp_path):
    """Round trip through a graph file written by our own writer (wide net, no TensorFlow needed)."""
    rng = np.random.default_rng(0)
    shapes = {"model/pi_fc0/w": (18, 64), "model/pi_fc0/b": (64,), "model/vf_fc0/w": (18, 64), "model/vf_fc0/b": (64,),
              "model/pi_fc1/w": (64, 32), "model/pi_fc1/b": (32,), "model/vf_fc1/w": (64, 32), "model/vf_fc1/b": (32,),
              "model/vf/w": (32, 1), "model/vf/b": (1,), "model/pi/w": (32, 18), "model/pi/b": (18,),
              "model/pi/logstd": (1, 18), "model/q/w": (32, 18), "model/q/b": (18,)}
    tensors = {k: rng.standard_normal(s).astype(np.float32) for k, s in shapes.items()}
    tensors["model/pi/b"][:] = 0  # exercises the "all-zero tensor has no value field" path
    path = str(tmp_path / "g.meta.txt")
    write_meta_txt(path, tensors, ent_coef=0.01, vf_coef=0.25, clip_norm=0.7, beta1=0.8, beta2=0.99, adam_eps=1e-7)
    info, params = core.meta_parse(path)
    assert (info.hidden1, info.hidden2, info.n_params_total) == (64, 32, sum(int(np.prod(s)) for s in shapes.values()))
    assert info.ent_coef == np.float32(0.01) and info.vf_coef == 0.25 and info.max_grad_norm == np.float32(0.7)
    assert np.array_equal(params, np.concatenate([tensors[n].ravel() for n in TENSOR_ORDER]))
    py = parse_meta_txt(path)
    assert py.hidden == [64, 32] and np.array_equal(py.flat_params(), params)


def test_meta_parse_errors():
    lib = _lib.load()
    info = _lib.MetaInfo()
    assert lib.ppo_meta_parse(b"/nonexistent/graph.meta.txt", C.byref(info), None, 0) == -3
    assert b"cannot open" in lib.ppo_last_error()


def _parse_bundle_index(buf):
    """Independent reader of a Saver-V2 `.index` (LevelDB table, one data block): {key: BundleEntryProto fields}."""
    def varint(b, i):
        v = s = 0
        while True:
            c = b[i]; i += 1
            v |= (c & 0x7F) << s; s += 7
            if c < 0x80:
                return v, i
    assert buf[-8:] == (0xdb4775248b80fb57).to_bytes(8, "little")
    foot = buf[-48:]
    _, i = varint(foot, 0); _, i = varint(foot, i)          # meta-index handle
    ioff, i = varint(foot, i); isz, i = varint(foot, i)      # index handle
    iblk = buf[ioff:ioff + isz]
    _, j = varint(iblk, 0); kl, j = varint(iblk, j); vl, j = varint(iblk, j)
    doff, k = varint(iblk, j + kl); dsz, k = varint(iblk, k)
    blk = buf[doff:doff + dsz]
    nrest = int.from_bytes(blk[-4:], "little")
    end = len(blk) - 4 - 4 * nrest
    out, key, i = {}, b"", 0
    while i < end:
        sh, i = varint(blk, i); un, i = varint(blk, i); vl, i = varint(blk, i)
        key = key[:sh] + blk[i:i + un]; i += un
        val = blk[i:i + vl]; i += vl
        f, j = {"shape": []}, 0
        while j < len(val):
            tag = val[j]; j += 1
            if tag == 0x35:
                f["crc"] = int.from_bytes(val[j:j + 4], "little"); j += 4
            elif tag in (0x12, 0x1a):
                ln, j = varint(val, j); sub = val[j:j + ln]; j += ln
                q = 0
                while tag == 0x12 and q < len(sub):  # TensorShapeProto.dim { size }
                    assert sub[q] == 0x12
                    dl, q = varint(sub, q + 1)
                    assert sub[q] == 0x08
                    f["shape"].append(varint(sub, q + 1)[0]); q += dl
            else:
                v, j = varint(val, j)
                f[{0x08: "dtype", 0x20: "offset", 0x28: "size"}[tag]] = v
        out[key.decode()] = f
    return out


def test_checkpoint_index_is_tensorflows(tmp_path):
    """The `.index` we write for the reference's shipped checkpoint is TensorFlow's own file, byte for byte
    (resources/ppo_cl/2019-08-20_21_13_01_2859_0.pkl.71.index, copied to tests/golden/ckpt_71.index), and an independent reader
    finds the 15 tensors with the offsets of the `.data` file; other widths parse with consistent offsets / sizes."""
    import numpy as np
    lib = _lib.load()
    ck = np.load(os.path.join(os.path.dirname(__file__), "golden", "ckpt_71_weights.npz"))
    names = sorted(k.replace("__", "/") for k in ck.files)
    payload = np.concatenate([ck[n.replace("/", "__")].astype(np.float32).ravel() for n in names])
    fp = payload.ctypes.data_as(C.POINTER(C.c_float))
    assert lib.ppo_checkpoint_write_index(str(tmp_path / "a").encode(), 18, 18, 4, 5, fp, payload.size) == 0
    got = open(tmp_path / "a.index", "rb").read()
    want = open(os.path.join(os.path.dirname(__file__), "golden", "ckpt_71.index"), "rb").read()
    assert got == want
    ent = _parse_bundle_index(got)
    assert list(ent)[0] == "" and list(ent)[1:] == names
    off = 0
    for n in names:
        e = ent[n]
        assert e["dtype"] == 1 and tuple(e["shape"]) == ck[n.replace("/", "__")].shape
        assert e.get("offset", 0) == off and e["size"] == 4 * ck[n.replace("/", "__")].size
        off += e["size"]
    assert off == 1768
    # a [64,64] policy on (36, 18): several restart-free entries with multi-byte varints
    big = np.arange(36 * 64 * 2 + 64 * 64 * 2 + 64 * 4 + 64 * 18 * 2 + 18 * 3 + 64 + 1, dtype=np.float32)
    assert lib.ppo_checkpoint_write_index(str(tmp_path / "b").encode(), 36, 18, 64, 64, big.ctypes.data_as(C.POINTER(C.c_float)), big.size) == 0
    ent = _parse_bundle_index(open(tmp_path / "b.index", "rb").read())
    assert ent["model/pi_fc0/w"]["shape"] == [36, 64] and ent["model/vf/w"]["shape"] == [64, 1]
    assert sum(e["size"] for k, e in ent.items() if k) == 4 * big.size
    assert lib.ppo_checkpoint_write_index(str(tmp_path / "c").encode(), 36, 18, 64, 64, fp, payload.size) == -1  # wrong payload size


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    with pytest.raises(core.PPOError, match="no CUDA device"):
        core.PPOCore()


def test_desc_validation():
    lib = _lib.load()
    d = _lib.CoreDesc()
    assert lib.ppo_core_desc_default(C.byref(d)) == 0
    assert (d.obs_dim, d.hidden1, d.hidden2, d.nminibatches, d.noptepochs) == (18, 4, 5, 32, 10)
    h = C.c_void_p()
    d.n_envs, d.n_steps, d.nminibatches = 1, 100, 32  # 100 % 32 != 0: the reference asserts (ppo2.hpp:265)
    assert lib.ppo_core_create(C.byref(d), C.byref(h)) == -1
    assert b"not divisible" in lib.ppo_last_error()
    d.abi_version = 99
    assert lib.ppo_core_create(C.byref(d), C.byref(h)) == -1
