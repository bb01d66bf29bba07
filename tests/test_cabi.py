"""CPU-side checks of the drop-in boundary: the C-ABI library builds, loads and exports every
symbol include/mlg_b200.h declares; argument validation works without a GPU; the product refuses
to compute on CPU tensors (no fallback)."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__
    __graft_entry__.build()
    from multilevel_gnn_b200 import _cabi
    return _cabi.lib()


def _declared():
    hdr = open(os.path.join(ROOT, "include", "mlg_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(mlg_[a-z0-9_]+)\s*\(", hdr)))


def test_header_symbols_exported(lib):
    from multilevel_gnn_b200 import _cabi
    names = _declared()
    assert len(names) >= 15
    raw = ctypes.CDLL(_cabi.LIB_PATH)
    for n in names:
        assert hasattr(raw, n), "libmlg_b200.so does not export %s" % n
    assert sorted(_cabi.exported_symbols()) == names, "ctypes table and header disagree"


def test_ctypes_signatures_match_header():
    """Every prototype of include/mlg_b200.h against the ctypes table: same argument count, pointers bound as c_void_p,
    int64_t / int / float / double as the matching scalar -- a drifted binding would push garbage into a kernel launch."""
    from multilevel_gnn_b200 import _cabi
    hdr = open(os.path.join(ROOT, "include", "mlg_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    hdr = re.sub(r"//[^\n]*", "", hdr)
    kinds = {ctypes.c_void_p: "ptr", ctypes.c_char_p: "ptr", ctypes.c_int64: "i64", ctypes.c_int: "int",
             ctypes.c_float: "f32", ctypes.c_double: "f64"}
    seen = 0
    for ret, name, args in re.findall(r"([A-Za-z_][A-Za-z0-9_ \*]*?)\b(mlg_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", hdr):
        res, argtypes = _cabi._SIGNATURES[name]
        params = [a.strip() for a in args.split(",") if a.strip() and a.strip() != "void"]
        want = []
        for prm in params:
            if "*" in prm:
                want.append("ptr")
            elif re.match(r"(const\s+)?(int64_t|uint64_t)\b", prm):
                want.append("i64")
            elif re.match(r"(const\s+)?int\b", prm):
                want.append("int")
            elif re.match(r"(const\s+)?float\b", prm):
                want.append("f32")
            elif re.match(r"(const\s+)?double\b", prm):
                want.append("f64")
            else:
                raise AssertionError("%s: unrecognised parameter %r" % (name, prm))
        got = [kinds[t] for t in argtypes]
        assert got == want, "%s: header %s vs ctypes %s" % (name, want, got)
        rk = "ptr" if "*" in ret else ("i64" if "int64_t" in ret else "int")
        assert kinds[res] == rk, "%s: return type %s vs ctypes %s" % (name, ret.strip(), kinds[res])
        seen += 1
    assert seen == len(_cabi._SIGNATURES), "parsed %d prototypes, table has %d" % (seen, len(_cabi._SIGNATURES))


def test_abi_version_and_errors(lib):
    from multilevel_gnn_b200 import _cabi
    assert lib.mlg_abi_version() == 2
    rc = lib.mlg_gen_aggr_fwd(None, None, None, None, None, 4, 8, 0, 1.0, None, 1.0, None, None, 1e-7, 0, None,
                              None, None, None, None)
    assert rc < 0 and "null" in _cabi.last_error()
    rc = lib.mlg_pool_fwd(None, None, None, None, None, None, 1, 1, 1, 1, 1, 99, 0, None, None)
    assert rc < 0
    assert lib.mlg_csr_build_workspace_bytes(1000, 100, 1) > 4 * 1100 * 4


def test_no_cpu_fallback(lib):
    import multilevel_gnn_b200 as m
    from multilevel_gnn_b200 import _cabi
    conv = m.GENConv(8, 8, aggr="softmax", encode_edge=False, norm="layer")
    with pytest.raises(_cabi.NativeLibraryError):
        conv(torch.randn(5, 8), torch.zeros(2, 6, dtype=torch.long), torch.randn(6, 8))
    with pytest.raises(_cabi.NativeLibraryError):
        m.knn_graph_matrix(torch.randn(20, 4), 3)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "multilevel-gnn_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "/root/reference" not in src.replace("(/root/reference", "").replace(" /root/reference/opt.py", ""), f


def test_state_dict_keys_match_reference_layout():
    import multilevel_gnn_b200 as m
    model = m.MultilevelGNN(m.configs.make_args("gbm"))
    keys = set(model.state_dict().keys())
    for k in ["node_embedding", "learnable_pca_params", "gnn_model.0.gconv.lin_l.weight", "gnn_model.0.gconv.lin_r.weight",
              "gnn_model.0.gconv.nn.0.weight", "gnn_model.0.gconv.nn.0.bias", "gnn_model.1.gconv.lin_r.weight",
              "conv_model.0.weight", "conv_model.2.bias", "head.0.weight", "head.3.bias"]:
        assert k in keys, k
    assert sum(p.numel() for p in model.parameters()) == 2833264          # SURVEY.md App. B.7
    g = m.GENConv(16, 16, aggr="softmax", learn_t=True, msg_norm=True, encode_edge=True, edge_feat_dim=16, norm="layer")
    assert set(g.state_dict()) == {"t", "feature_encoder.0.weight", "feature_encoder.0.bias", "feature_encoder.1.weight",
                                   "feature_encoder.1.bias", "feature_encoder.3.weight", "feature_encoder.3.bias",
                                   "msg_norm.msg_scale", "edge_encoder.weight", "edge_encoder.bias"}
