"""CPU checks of the drop-in boundary: libqot_b200.so loads, exports every symbol that
include/qot_b200.h declares (and the ctypes table binds exactly those), the product package
never touches oracle/ or the reference, and it refuses to run without CUDA (no fallback)."""
import ctypes
import re
import subprocess
import sys
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
HEADER = ROOT / "include" / "qot_b200.h"
PKG = ROOT / "gnn_qot_estimation_b200"


def declared_symbols():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    return sorted(set(re.findall(r"\b(qot_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def lib_path():
    from gnn_qot_estimation_b200 import build
    return build.build()          # no-op when the stamp matches; nvcc cross-compiles without a GPU


def test_header_declares_the_documented_families():
    syms = declared_symbols()
    for fam in ("qot_collate", "qot_build_csr", "qot_tconv_fwd", "qot_tconv_bwd", "qot_nnconv_fwd",
                "qot_nnconv_bwd", "qot_gat_fwd", "qot_gat_bwd", "qot_bn_stats", "qot_bn_bwd_sparse",
                "qot_pool_mlp_fwd", "qot_pool_mlp_bwd", "qot_lut_head_fwd", "qot_lut_head_bwd",
                "qot_lightpath_infer_stream", "qot_lightpath_infer_wire_host", "qot_last_error"):
        assert fam in syms, fam


def test_library_exports_every_declared_symbol(lib_path):
    handle = ctypes.CDLL(str(lib_path))
    for name in declared_symbols():
        assert hasattr(handle, name), f"{name} declared in qot_b200.h but not exported"


def test_ctypes_table_matches_header(lib_path):
    from gnn_qot_estimation_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared_symbols()
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    for name, (_, argtypes) in _lib.SIGNATURES.items():
        m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
        assert m, name
        params = m.group(1).strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert n == len(argtypes), f"{name}: header has {n} parameters, ctypes table {len(argtypes)}"
    _lib.lib()                     # binds every symbol; raises AttributeError on a missing one


@pytest.mark.parametrize("struct,ctype,size", [("qot_sgd_hyper_t", "QotSgdHyper", 32),
                                               ("qot_param_seg_t", "QotParamSeg", 24),
                                               ("qot_lp_state_t", "QotLpState", 264),
                                               ("qot_lp_changes_t", "QotLpChanges", 72),
                                               ("qot_lp_demands_t", "QotLpDemands", 80)])
def test_ctypes_structs_match_header(struct, ctype, size):
    """Field names, order, offsets and size of the structs the kernels read from device memory, and of the network-state
    queries' argument structs."""
    from gnn_qot_estimation_b200 import _lib
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    body = re.search(r"typedef struct \{([^}]*)\}\s*" + struct + r"\s*;", text).group(1)
    names = [re.sub(r"\[\d+\]$", "", n.strip().lstrip("*")) for decl in body.split(";") if decl.strip()
             for n in decl.strip().removeprefix("const ").split(None, 1)[1].split(",")]
    cls = getattr(_lib, ctype)
    assert [f[0] for f in cls._fields_] == names
    assert ctypes.sizeof(cls) == size
    if struct == "qot_lp_state_t":
        assert cls._fields_[0][1] is _lib.QotLpGraphCfg and ctypes.sizeof(_lib.QotLpGraphCfg) == cls.S.offset == 184
    if struct == "qot_sgd_hyper_t":
        offs = {f[0]: getattr(cls, f[0]).offset for f in cls._fields_}
        assert offs == {"lr": 0, "momentum": 4, "dampening": 8, "weight_decay": 12, "nesterov": 16, "maximize": 20,
                        "one_minus_dampening": 24, "reserved": 28}
        assert getattr(cls, "one_minus_dampening").size == 4 and cls._fields_[6][1] is ctypes.c_float


def test_no_torch_types_in_the_abi():
    code = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)      # declarations only, no comments
    assert "torch" not in code.lower() and "at::" not in code and "Tensor" not in code
    assert re.findall(r"#include\s*<([^>]+)>", code) == ["stddef.h", "stdint.h"]


def test_library_is_sm100a_only(lib_path):
    out = subprocess.run(["cuobjdump", "--list-elf", str(lib_path)], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = set(re.findall(r"sm_\d+a?", out.stdout))
    assert archs == {"sm_100a"}, archs


def test_cpu_arguments_fail_through_the_abi(lib_path):
    """Argument validation works without a GPU: bad sizes return QOT_E_BADARG + a message."""
    from gnn_qot_estimation_b200 import _lib
    L = _lib.lib()
    assert L.qot_version() >= 101
    rc = L.qot_build_csr(None, -1, 4, 1, 0, None, None, None, None, None, 0, None)
    assert rc == -1 and b"negative" in L.qot_last_error()
    rc = L.qot_tconv_fwd(None, None, None, None, None, None, 10, 17, 1.0, None, None, None, None, None)
    assert rc == -1 and b"H must be" in L.qot_last_error()
    assert L.qot_csr_workspace_bytes(1000, 5000) > 0
    assert L.qot_lightpath_prepared_floats() >= 5 * 4 * 2 + 128 * 5 + 128 + 128 * 32 + 32 + 96 + 3


STATE_QUERIES = {"qot_lightpath_candidates": 2, "qot_lightpath_reconfigure": 2, "qot_lightpath_change_sets": 4,
                 "qot_lightpath_placements": 6, "qot_lightpath_provision": 8}      # name -> position of `prepared`


@pytest.mark.parametrize("name", sorted(STATE_QUERIES))
def test_state_query_arguments_fail_through_the_abi(lib_path, name):
    """The network-state queries validate their arguments before any CUDA call: with an empty query the call returns 0
    without a GPU, and a NULL descriptor, a negative count, a misaligned `prepared` or an `is_lut_index` out of range
    each returns QOT_E_BADARG with a message naming the entry point."""
    from gnn_qot_estimation_b200 import _lib
    L = _lib.lib()
    argtypes = _lib.SIGNATURES[name][1]
    query_cls, at = argtypes[1]._type_, STATE_QUERIES[name]
    assert argtypes[0] is ctypes.POINTER(_lib.QotLpState)
    assert query_cls in (_lib.QotLpChanges, _lib.QotLpDemands)
    assert argtypes[at:at + 3] == [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32]   # prepared, lut index, max_impact

    def call(state=True, query=True, S=0, count=0, prepared=1 << 20, lut=1):
        st = _lib.QotLpState(cfg=_lib.QotLpGraphCfg(F=8, L=4, Q=16), S=S)
        q = query_cls(**{query_cls._fields_[0][0]: count})                      # K or D
        args = [ctypes.byref(st) if state else None, ctypes.byref(q) if query else None]
        args += [0 if t in (ctypes.c_int32, ctypes.c_int64) else None for t in argtypes[2:]]
        args[at], args[at + 1] = prepared, lut
        return getattr(L, name)(*args)

    assert call() == 0
    for bad, why in ((dict(state=False), b"descriptor"), (dict(query=False), b"descriptor"), (dict(S=-1), b"bad size"),
                     (dict(count=-1), b"bad size"), (dict(prepared=(1 << 20) + 4), b"16-byte aligned"),
                     (dict(prepared=None), b"16-byte aligned"), (dict(lut=5), b"is_lut_index"),
                     (dict(lut=-1), b"is_lut_index")):
        assert call(**bad) == -1, bad
        msg = L.qot_last_error()
        assert msg.startswith(name.encode() + b":") and why in msg, (bad, msg)


def test_product_refuses_cpu_tensors():
    from gnn_qot_estimation_b200 import LightpathGNN, TopologicalGNN, ops, synthetic
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.build_csr(torch.zeros(2, 3, dtype=torch.int64), 4)
    hb = synthetic.lightpath_store(2, seed=0).host_batch(0, 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        LightpathGNN(5, 32, 3, is_lut_index=1).eval()(hb)
    tb = synthetic.nsfnet_store(2, seed=0).host_batch(0, 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        TopologicalGNN(14, 16, 3, edge_dim=4)(tb)


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    from gnn_qot_estimation_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", tmp_path / "libqot_b200.so")
    with pytest.raises(RuntimeError, match="no CPU or PyTorch fallback"):
        _lib.lib()


def test_product_never_imports_oracle_or_reference():
    """The oracle is test infrastructure: nothing under the product package may import, open or
    execute it (nor /root/reference)."""
    bad = []
    for p in list(PKG.rglob("*.py")) + list(PKG.rglob("*.cu")) + list(PKG.rglob("*.cuh")):
        t = p.read_text()
        if re.search(r"^\s*(from|import)\s+(oracle|torch_geometric)\b", t, flags=re.M) or "/root/reference" in t:
            bad.append(str(p))
    assert not bad, bad
    code = ("import sys; sys.path.insert(0, %r); import gnn_qot_estimation_b200 as g; "
            "from gnn_qot_estimation_b200 import ops, nn, batch, synthetic, pipeline; "
            "g.TopologicalGNN; g.LightpathGNN; "
            "assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules), 'oracle imported'" % str(ROOT))
    subprocess.run([sys.executable, "-c", code], check=True)


def test_no_triton_or_compile_in_product():
    for p in PKG.rglob("*.py"):
        t = p.read_text()
        assert "import triton" not in t and "torch.compile" not in t, p


@pytest.mark.parametrize("M,Nc,K,splits", [(128, 128, 32, 1), (300, 68, 96, 1), (1000, 256, 64, 1), (256, 384, 64, 1),
                                           (1024, 100, 128, 1), (10000, 2560, 256, 1), (4097, 1024, 256, 1),
                                           (256, 256, 80000, 37), (2560, 256, 10016, 64), (128, 384, 64, 3)])
def test_gemm_tile_pairs_cover_every_output_tile_once(lib_path, M, Nc, K, splits):
    """Host-only hook of csrc/gemm_tc.cu: the cluster kernel hands out PAIRS of tiles; whatever the tile counts
    (odd x odd: a partner off the matrix edge that computes but does not store; n-count odd and m-count even: pairs
    along m) every 128 x 128 output tile of every split-K slice must be stored by exactly one CTA, the two CTAs of a pair
    must share the operand block they multicast and walk the same k-blocks, and the slices must tile the reduction."""
    import numpy as np
    L = ctypes.CDLL(str(lib_path))
    fn = L.qot_debug_gemm_tiles
    fn.restype = ctypes.c_int64
    fn.argtypes = [ctypes.c_int64] * 5 + [ctypes.c_void_p, ctypes.c_int64]
    kb_total = K // 32
    kps = -(-kb_total // splits)
    n = fn(M, Nc, K, kps, splits, None, 0)
    assert n > 0 and n % 2 == 0
    out = np.zeros((n, 6), dtype=np.int64)
    assert fn(M, Nc, K, kps, splits, out.ctypes.data, n) == n
    tm, tn = -(-M // 128), -(-Nc // 128)
    seen = {}
    for p in range(0, n, 2):
        a, b = out[p], out[p + 1]
        assert a[4] == 1                                            # rank 0 always owns a real tile
        assert tuple(a[2:4]) == tuple(b[2:4]) and a[5] == b[5]      # same k-blocks: the pair runs in lockstep
        assert a[0] == b[0] or a[1] == b[1]                          # shared operand block: same A rows or same W rows
        for t in (a, b):
            assert 0 <= t[0] < tm * 128 and 0 <= t[1] < tn * 128 and t[0] % 128 == 0 and t[1] % 128 == 0
            if t[4]:
                key = (int(t[5]), int(t[0]), int(t[1]))
                assert key not in seen, key
                seen[key] = (int(t[2]), int(t[3]))
    assert len(seen) == splits * tm * tn
    for (z, m0, n0), (kb0, nkb) in seen.items():                     # slices tile [0, kb_total)
        assert kb0 == z * kps and nkb == max(0, min(kps, kb_total - kb0))
    assert sum(v[1] for k, v in seen.items() if k[1] == 0 and k[2] == 0) == kb_total
