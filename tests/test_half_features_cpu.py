"""16-bit node features without a GPU: packed feature files in fp16 / bf16, the old fp32 format, and the `_x` entry points of the
C ABI (symbols, prototypes, rejection of an unknown element kind before any device work)."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest
import torch

import gcn_mtmc_b200 as m
from gcn_mtmc_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
X_ENTRY_POINTS = ["mpn_edge_features_x", "mpn_forward_x", "mpn_forward_with_edge_features_x", "mpn_forward_sharded_x",
                  "mpn_forward_sharded_with_edge_features_x", "mpn_plan_node_encoder_x", "mpn_normalize_columns_x",
                  "mpn_normalize_columns_batched_x"]


def _features(n=37, d=24, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, d, generator=g) * 3, np.arange(n) % 5, np.arange(n) * 7


def _header(path):
    with open(path, "rb") as f:
        assert f.read(8) == m.graph_inputs.MAGIC
        hlen = int(np.frombuffer(f.read(8), dtype=np.int64)[0])
        return json.loads(f.read(hlen).decode())


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16], ids=["f16", "bf16"])
@pytest.mark.parametrize("spelling", ["torch", "str"])
def test_pack_read_round_trip_half(tmp_path, dt, spelling):
    x, cam, tid = _features()
    p = str(tmp_path / "feat.bin")
    m.pack_reid_features(p, x, cam, tid, dtype=dt if spelling == "torch" else str(dt).replace("torch.", ""))
    assert _header(p)["dtype"] == str(dt).replace("torch.", "")
    assert os.path.getsize(p) % 4096 == x.numel() * 2 % 4096                    # 2 bytes per element after the aligned prefix
    xr, cr, tr = m.read_packed_features(p)
    got = xr if torch.is_tensor(xr) else torch.from_numpy(np.array(xr))
    assert got.dtype == dt and got.shape == x.shape
    assert torch.equal(got.view(torch.int16), x.to(dt).view(torch.int16))       # bit-exact: round to nearest even, raw words
    assert np.array_equal(cr, cam) and np.array_equal(tr, tid)


def test_pack_half_from_half_tensor_and_list(tmp_path):
    x, cam, tid = _features(9, 8, 1)
    xb = x.to(torch.bfloat16)
    p1, p2 = str(tmp_path / "a.bin"), str(tmp_path / "b.bin")
    m.pack_reid_features(p1, xb, cam, tid, dtype="bfloat16")                   # exact: no second rounding
    m.pack_reid_features(p2, list(xb), cam, tid, dtype="bfloat16")
    for p in (p1, p2):
        assert torch.equal(m.read_packed_features(p)[0].view(torch.int16), xb.view(torch.int16))


def _parent_format(path, x, cam, tid):
    """The fp32 layout as the format has always been written: magic, header length, JSON header, ids, pad to 4096, features."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    cam, tid = np.asarray(cam, dtype=np.int64), np.asarray(tid, dtype=np.int64)
    header = json.dumps({"n": int(x.shape[0]), "d": int(x.shape[1]), "dtype": "float32"}).encode()
    pre = 8 + 8 + len(header) + cam.nbytes + tid.nbytes
    with open(path, "wb") as f:
        f.write(b"MPNFEAT1" + np.int64(len(header)).tobytes() + header + cam.tobytes() + tid.tobytes() + b"\0" * ((-pre) % 4096)
                + x.tobytes())


def test_fp32_files_unchanged(tmp_path):
    x, cam, tid = _features(50, 16, 2)
    old, new = str(tmp_path / "old.bin"), str(tmp_path / "new.bin")
    _parent_format(old, x.numpy(), cam, tid)
    m.pack_reid_features(new, x, cam, tid)
    with open(old, "rb") as a, open(new, "rb") as b:
        assert a.read() == b.read()                                           # the default still writes the same bytes
    xr, cr, tr = m.read_packed_features(old)
    assert isinstance(xr, np.ndarray) and xr.dtype == np.float32 and np.array_equal(xr, x.numpy())
    assert np.array_equal(cr, cam) and np.array_equal(tr, tid)


def test_unknown_dtype_rejected(tmp_path):
    x, cam, tid = _features(4, 4, 3)
    with pytest.raises(ValueError):
        m.pack_reid_features(str(tmp_path / "x.bin"), x, cam, tid, dtype="float64")
    p = str(tmp_path / "bad.bin")
    _parent_format(p, x.numpy(), cam, tid)
    with open(p, "r+b") as f:                                               # same length: "float32" -> "float64"
        data = f.read()
        f.seek(0)
        f.write(data.replace(b'"dtype": "float32"', b'"dtype": "float64"', 1))
    with pytest.raises(ValueError):
        m.read_packed_features(p)


def test_x_entry_points_in_header_library_and_bindings():
    header = open(os.path.join(ROOT, "include", "mpn_b200.h")).read()
    for k, v in (("MPN_X_F32", 0), ("MPN_X_F16", 1), ("MPN_X_BF16", 2)):
        assert re.search(r"#define %s %d\b" % (k, v), header)
        assert getattr(_lib, k) == v
    lib = _lib.lib()
    assert lib.mpn_abi_version() == 6
    for name in X_ENTRY_POINTS:
        assert name in _lib.EXPORTED_SYMBOLS and hasattr(lib, name), name
        proto = re.search(r"\b%s\(([^;]*)\);" % name, header)
        assert proto, name
        params = [p for p in proto.group(1).split(",") if p.strip()]
        assert len(params) == len(_lib._PROTOS[name][1]), name
        assert "const void* x_dev, int32_t x_kind" in proto.group(1), name
        # the fp32 entry point takes the same arguments without x_kind
        assert len(_lib._PROTOS[name[:-2]][1]) == len(params) - 1, name


def test_unknown_x_kind_is_an_error_before_device_work():
    lib = _lib.lib()
    fake = C.c_void_p(256)
    g = _lib.MpnGraph()
    w = _lib.MpnWeights()
    calls = [
        lambda k: lib.mpn_normalize_columns_x(fake, k, 4, 4, fake, fake, 1 << 20, None),
        lambda k: lib.mpn_normalize_columns_batched_x(fake, k, 4, 4, fake, 2, fake, None, 0, None),
        lambda k: lib.mpn_edge_features_x(C.byref(g), fake, k, 4, fake, 1, fake, 1 << 20, None),
        lambda k: lib.mpn_forward_x(C.byref(g), C.byref(w), fake, k, fake, 1, 1, fake, None, None, None, 1, fake, 1 << 20, None),
    ]
    for call in calls:
        assert call(3) == _lib.MPN_ERR_INVALID
        assert b"element kind 3" in lib.mpn_last_error()
        assert call(-1) == _lib.MPN_ERR_INVALID
