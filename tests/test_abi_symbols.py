"""CPU: libpsb_b200.so loads and exports every symbol include/psb.h declares (no compute)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "psb.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(psb_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    from prodsearch_b200 import _lib
    from prodsearch_b200.build import build_library
    build_library()
    names = _declared()
    assert len(names) >= 13
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), "missing export " + n
        assert n in _lib.SIGNATURES, "no ctypes signature for " + n
    assert sorted(_lib.SIGNATURES) == names
    assert _lib.load().psb_abi_version() == 1
    assert _lib.status_string(0) == "ok" and "aligned" in _lib.status_string(-4)


def test_contrib_struct_layout():
    from prodsearch_b200 import _lib
    assert ctypes.sizeof(_lib.Contrib) == 72          # psb_contrib_t: 8 x 8-byte fields + 2 x int32


def test_argument_validation_without_gpu():
    """Host-side argument checks return PSB_E_* before any CUDA call."""
    from prodsearch_b200 import _lib
    lib = _lib.load()
    assert lib.psb_gather_rows(None, 10, 128, None, 0, None, None, None) == -1          # null table
    assert lib.psb_gather_rows(16, 10, 130, None, 0, None, None, None) == -2            # d % 4 != 0
    assert lib.psb_gather_rows(8, 10, 128, None, 0, None, None, None) == -4             # misaligned
    assert lib.psb_gather_rows(16, 10, 128, None, 0, None, None, None) == 0             # n == 0: no launch
    assert lib.psb_scatter_reduce_workspace_bytes(1000, 50) > 16 * 1000
    assert lib.psb_catalog_topk_workspace_bytes(4, 100, 128, 10, 7) == -5               # bad mode
    # 3xTF32 GEMM entry: shape / alignment rules are checked on the host before any CUDA call
    assert lib.psb_debug_gemm3_tf32(1024, 100, 10, 100, 2048, 64, None, 4096, 64, None) == -5      # k % 64 != 0
    assert lib.psb_debug_gemm3_tf32(1024, 128, 10, 128, 2048, 96, None, 4096, 96, None) == -5      # j % 64 != 0
    assert lib.psb_debug_gemm3_tf32(1032, 128, 10, 128, 2048, 64, None, 4096, 64, None) == -5      # a not 16-byte aligned
    assert lib.psb_debug_gemm3_tf32(1024, 64, 10, 128, 2048, 64, None, 4096, 64, None) == -1       # lda < k
    assert lib.psb_debug_gemm3_tf32(1024, 128, 0, 128, 2048, 64, None, 4096, 64, None) == 0        # no rows: no launch
    assert lib.psb_launch_count() == 0


def test_no_oracle_or_reference_in_product():
    """The product path may not import the oracle or read /root/reference."""
    pkg = os.path.join(ROOT, "prodsearch_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f
                assert "/root/reference" not in src, f


def test_row_grad_sink_fork_plumbing_present():
    """The gradient sink forks its sort + reduce chain onto a side stream and joins it in one engine callback;
    both ends must exist (a missing join only shows up on a GPU box)."""
    from prodsearch_b200 import functional as F_
    assert callable(F_.run_forked) and callable(F_.RowGradSink._join_forked)
    assert callable(getattr(F_.RowGradSink, "_finalize_callback")) and callable(getattr(F_.RowGradSink, "finalize"))


def _prototypes():
    """name -> (return type, [parameter types]) parsed from include/psb.h (comments stripped)."""
    text = open(os.path.join(ROOT, "include", "psb.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"//[^\n]*", "", text)
    out = {}
    for ret, name, params in re.findall(r"([A-Za-z_][A-Za-z0-9_ ]*?[\s\*]+)\b(psb_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", text):
        plist = [] if params.strip() in ("", "void") else [p.strip() for p in params.split(",")]
        out[name] = (ret.strip(), [re.sub(r"\s*\b[A-Za-z_][A-Za-z0-9_]*$", "", p).strip() for p in plist])
    return out


def _ctype_class(t):
    """Coarse class of a C type as ctypes has to pass it."""
    t = t.replace("const", "").strip()
    if "*" in t or t in ("psb_stream_t",):
        return "ptr"
    return {"int": "i32", "int32_t": "i32", "int64_t": "i64", "float": "f32", "double": "f64", "uint64_t": "u64",
            "uint32_t": "u32"}[t]


def test_ctypes_signatures_match_the_header_prototypes():
    """A ctypes call with the wrong arity or integer width is silent undefined behaviour: every prototype of
    include/psb.h must agree, parameter by parameter, with the (restype, argtypes) entry _lib.py binds it with."""
    from prodsearch_b200 import _lib
    protos = _prototypes()
    assert sorted(protos) == _declared()
    by_ctype = {ctypes.c_void_p: "ptr", ctypes.c_char_p: "ptr", ctypes.c_int32: "i32", ctypes.c_int64: "i64",
                ctypes.c_float: "f32", ctypes.c_double: "f64", ctypes.c_uint64: "u64", ctypes.c_uint32: "u32",
                ctypes.c_int: "i32"}

    def cls(ct):
        if ct in by_ctype:
            return by_ctype[ct]
        assert issubclass(ct, (ctypes._Pointer, ctypes.Structure, ctypes.Array)) or hasattr(ct, "contents"), ct
        return "ptr" if not issubclass(ct, ctypes.Structure) else "struct"
    for name, (ret, params) in sorted(protos.items()):
        res, args = _lib.SIGNATURES[name]
        assert len(args) == len(params), "%s: header has %d parameters, ctypes binds %d" % (name, len(params), len(args))
        got = [cls(a) for a in args]
        want = []
        for p in params:
            base = p.replace("const", "").strip()
            want.append("struct" if (base.endswith("_t") and base.startswith("psb_") and "*" not in base
                                     and base != "psb_stream_t") else _ctype_class(p))
        assert got == want, "%s: header %s, ctypes %s" % (name, want, got)
        assert cls(res) == ("ptr" if "*" in ret else _ctype_class(ret)), "%s: return type" % name


def test_stage_diff_script_layout_matches_the_library():
    """profiles/diff_enc_tc.py restates encoder_common.cuh's saved_layout to name the regions it compares: its total has
    to be what psb_encoder_saved_bytes reports for the same configuration (a host-side size query, no GPU)."""
    import importlib.util
    from prodsearch_b200 import _lib
    spec = importlib.util.spec_from_file_location("diff_enc_tc", os.path.join(ROOT, "profiles", "diff_enc_tc.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    cfg = _lib.EncoderCfg()
    cfg.S, cfg.T, cfg.d, cfg.heads, cfg.ff, cfg.copies, cfg.out_pos = m.S, m.T, m.D, m.H, m.FF, m.C, 0
    cfg.ln_eps, cfg.p_drop = 1e-6, 0.0
    cfg.first = cfg.table = cfg.idx = 16            # non-null, aligned stand-ins: the query only validates them
    cfg.table_rows = 10
    total = sum(n for _, n in m.layout().values())
    assert _lib.load().psb_encoder_saved_bytes(ctypes.byref(cfg)) == 4 * total
