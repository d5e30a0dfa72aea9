"""CPU: the C-ABI library loads, exports every symbol ``include/mlv_index.h`` declares, and the
product fails loudly without a GPU (no CPU fallback, no oracle behind the product)."""
import ast
import ctypes as C
import os
import re

import numpy as np
import pytest

from mlvectordb_b200 import _capi, pack_bitmap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    with open(os.path.join(ROOT, "include", "mlv_index.h")) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(mlv_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    names = _declared_symbols()
    assert len(names) >= 20 and "mlv_index_search" in names and "mlv_merge_topk" in names
    lib = C.CDLL(_capi.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/mlv_index.h but not exported"
    assert set(names) == set(_capi.SIGNATURES), "ctypes binding and header disagree"
    assert _capi.lib().mlv_abi_version() == _capi.ABI_VERSION


def test_status_strings_and_null_handles():
    lib = _capi.lib()
    assert lib.mlv_status_string(0) == b"ok"
    assert b"no CPU fallback" in lib.mlv_status_string(_capi.MLV_E_NO_DEVICE)
    assert lib.mlv_index_destroy(None) == _capi.MLV_E_INVALID
    assert lib.mlv_index_info(None, None) == _capi.MLV_E_INVALID
    h = C.c_void_p()
    assert lib.mlv_index_create(0, 0, 0, 0, C.byref(h)) == _capi.MLV_E_INVALID      # dim 0
    assert lib.mlv_index_create(8, 7, 0, 0, C.byref(h)) == _capi.MLV_E_INVALID      # unknown metric


def test_no_gpu_means_loud_failure(has_gpu):
    if has_gpu:
        pytest.skip("a GPU is present")
    from mlvectordb_b200 import DeviceShard, GpuIndex
    from _refshim import Vector
    with pytest.raises(RuntimeError, match="no CUDA device"):
        DeviceShard(8, "l2")
    idx = GpuIndex(space="cosine")           # constructing is fine (no namespace yet) ...
    with pytest.raises(RuntimeError, match="no CUDA device"):
        idx.add([Vector([1.0, 2.0])], "ns")  # ... but nothing is ever served from the CPU
    assert idx.search(type("Q", (), {"values": [1.0, 2.0]})(), 1, "ns", "cosine") == []   # unknown namespace -> []


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "mlvectordb_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            tree = ast.parse(open(os.path.join(pkg, fn)).read())
            for node in ast.walk(tree):
                mods = []
                if isinstance(node, ast.Import):
                    mods = [a.name for a in node.names]
                elif isinstance(node, ast.ImportFrom):
                    mods = [node.module or ""]
                assert not any(m == "oracle" or m.startswith("oracle.") for m in mods), f"{fn} imports the oracle"
    for fn in os.listdir(os.path.join(pkg, "csrc")):
        assert "oracle" not in open(os.path.join(pkg, "csrc", fn)).read().replace("oracle/exact_scan.c", "").replace(
            "oracle/synthetic.py", "") or fn == "Makefile"


def test_pack_bitmap_layout():
    m = np.zeros(70, bool)
    m[[0, 31, 32, 69]] = True
    w = pack_bitmap(m)
    assert w.dtype == np.uint32 and w.tolist() == [0x80000001, 0x1, 0x20]
    assert pack_bitmap(np.ones(64, bool)).tolist() == [0xFFFFFFFF, 0xFFFFFFFF]
    assert pack_bitmap(np.zeros(0, bool)).shape == (0,)


def test_space_aliases():
    from mlvectordb_b200 import canonical_space
    assert canonical_space("euclidean") == "l2" and canonical_space("dot") == "ip" and canonical_space("cosine") == "cosine"
    with pytest.raises(ValueError):
        canonical_space("manhattan")


def test_float32_json_encoder_round_trips_without_a_gpu():
    """``mlv_format_f32_json`` (host-only helper of the response path): shortest text that round-trips every float32,
    non-finite values as Python's json module writes them, buffer-size contract."""
    import json
    rng = np.random.default_rng(0)
    vals = np.concatenate([rng.standard_normal(5000).astype(np.float32) * np.float32(10.0) ** rng.integers(-20, 20, 5000).astype(np.float32),
                           np.array([0.0, -0.0, 1.0, 3.0, 1e10, 1e-7, np.float32(1) / 3, np.finfo(np.float32).max,
                                     np.finfo(np.float32).tiny, 1e-45], dtype=np.float32)])
    text = _capi.format_f32_json(vals)
    back = np.array(json.loads(text), dtype=np.float32)
    assert np.array_equal(back, vals) and np.array_equal(np.signbit(back), np.signbit(vals))
    assert len(text) < len(json.dumps(vals.tolist())) * 0.7             # float32-shortest, not float64 repr
    assert _capi.format_f32_json(np.array([np.nan, np.inf, -np.inf], np.float32)) == b"[NaN,Infinity,-Infinity]"
    assert _capi.format_f32_json(np.empty(0, np.float32)) == b"[]"
    lib = _capi.lib()
    n = C.c_uint64()
    small = C.create_string_buffer(8)
    one = np.ones(4, np.float32)
    assert lib.mlv_format_f32_json(one.ctypes.data, 4, small, len(small), C.byref(n)) == _capi.MLV_E_INVALID


def test_every_tuning_key_is_documented_in_the_header():
    """mlv_index_set_tuning's keys live in one if-chain; the header is the only place a caller can learn them."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "mlvectordb_b200", "csrc", "mlv_index.cu")).read()
    hdr = open(os.path.join(root, "include", "mlv_index.h")).read()
    keys = sorted(set(re.findall(r'k == "([a-z0-9_]+)"', src)))
    assert len(keys) >= 20
    assert [k for k in keys if f'"{k}"' not in hdr] == []


def test_candidate_key_decoder_inverts_the_kernels_encoding():
    """key_parts is the inverse of f32_orderable (csrc/common.cuh): keys order as (distance, row) and decode bit-exactly,
    including +-0, +-inf, NaN, subnormals and negative values."""
    from mlvectordb_b200.shard import key_parts, make_keys
    tiny = np.float32(1.4e-45)
    vals = np.array([-np.inf, -3.4e38, -1.5, -tiny, -0.0, 0.0, tiny, 1e-40, 1.0, 3.4e38, np.inf, np.nan], np.float32)
    rows = np.arange(len(vals), dtype=np.uint32) * np.uint32(977)
    keys = make_keys(vals, rows)
    # f32_orderable: sign set -> all bits flipped, else the sign bit set
    hi = (keys >> np.uint64(32)).astype(np.uint32)
    assert hi[4] == 0x7FFFFFFF and hi[5] == 0x80000000 and hi[0] == 0x007FFFFF and hi[10] == 0xFF800000
    d, r = key_parts(keys)
    assert np.array_equal(d.view(np.uint32), vals.view(np.uint32)) and np.array_equal(r, rows)
    assert (np.diff(keys.astype(np.uint64)) > 0).all(), "key order is not the distance order"   # vals ascend, NaN last
    rng = np.random.default_rng(0)
    bits = rng.integers(0, 2 ** 32, 10_000, dtype=np.uint64).astype(np.uint32)
    rr = rng.integers(0, 2 ** 32, 10_000, dtype=np.uint64).astype(np.uint32)
    d, r = key_parts(make_keys(bits.view(np.float32), rr))
    assert np.array_equal(d.view(np.uint32), bits) and np.array_equal(r, rr)
    fin = ~np.isnan(bits.view(np.float32))
    k = make_keys(bits.view(np.float32)[fin], np.zeros(fin.sum(), np.uint32))
    o = np.argsort(k, kind="stable")
    assert (np.diff(bits.view(np.float32)[fin][o].astype(np.float64)) >= 0).all()
