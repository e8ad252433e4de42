"""CPU-only: the C-ABI library loads and exports every symbol include/t3d.h declares."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "t3d.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(t3d_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_symbols():
    syms = _header_symbols()
    assert "t3d_loss_fwd_bwd" in syms and "t3d_version" in syms
    assert len(syms) >= 8


def test_library_exports_every_declared_symbol(lib_built):
    handle = ctypes.CDLL(lib_built.LIB_PATH)
    missing = [s for s in _header_symbols() if not hasattr(handle, s)]
    assert not missing, f"symbols declared in include/t3d.h but not exported: {missing}"
    handle.t3d_version.restype = ctypes.c_int
    header = open(os.path.join(ROOT, "include", "t3d.h")).read()
    assert handle.t3d_version() == int(re.search(r"#define T3D_ABI_VERSION (\d+)", header).group(1)) == lib_built.ABI_VERSION


def test_python_binding_lists_every_declared_symbol(lib_built):
    assert sorted(lib_built.declared_symbols()) == _header_symbols()
    lib_built.lib()     # argtypes/restype set for each; raises if one is absent


def test_single_entry_points_reject_bad_arguments_without_a_gpu(lib_built):
    lib = lib_built.lib()
    assert lib.t3d_loss_workspace_bytes(0, 4, 4, 0) == 0
    assert lib.t3d_loss_workspace_bytes(2, 384, 512, 1) > 0
    rc = lib.t3d_loss_fwd_bwd(*([None] * 4), 8, 8, None, None, 8, 8, None, None, 3, None, None, 0, *([None] * 4),
                              1, 8, 8, 0, 0.2, 0.5, 0.3, 0.4, 1.0, None, None, None, None, None, 0, None)
    assert rc == -1
    assert b"NULL" in lib.t3d_last_error()
    # the library checks its arguments before any CUDA call: dummy non-NULL pointers never get dereferenced
    p = 256
    rc = lib.t3d_loss_fwd_bwd(p, p, p, p, 8, 8, None, None, 8, 8, None, None, 0, None, None, 0, p, None, None, None,
                              1, 8, 8, 0, 0.2, 0.5, 0.3, 0.4, 1.0, p, p, None, None, p, 1 << 20, None)
    assert rc == -1                     # exactly one dpred NULL
    assert b"NULL" in lib.t3d_last_error()
    for stats_scales, phase, what in ((3, 0, b"stats_scales"), (1, 7, b"phase")):
        rc = lib.t3d_preprocess_train_u16(p, 1, 8, 8, 8, 8, p, 3, None, p, None, stats_scales, 0, p, 1 << 20, phase, None)
        assert rc == -1
        assert what in lib.t3d_last_error()
    rc = lib.t3d_depth_metrics(p, 1, 0, p, 8, 8, None, 1, 8, 8, 0, p, None, None, p, 1 << 20, None, 7, None)
    assert rc == -1
    assert b"phase" in lib.t3d_last_error()


def _runtime_strings(py_source):
    """String constants of a module that are not docstrings (citations of reference files live in docstrings / comments)."""
    import ast
    tree = ast.parse(py_source)
    doc = set()
    for node in ast.walk(tree):
        if isinstance(node, (ast.Module, ast.ClassDef, ast.FunctionDef, ast.AsyncFunctionDef)) and node.body and \
                isinstance(node.body[0], ast.Expr) and isinstance(node.body[0].value, ast.Constant):
            doc.add(id(node.body[0].value))
    return [n.value for n in ast.walk(tree) if isinstance(n, ast.Constant) and isinstance(n.value, str) and id(n) not in doc]


def test_product_does_not_import_oracle():
    """The product path must never route through oracle/ (or any CPU fallback), nor touch the reference tree at run
    time: /root/reference may only be CITED (docstrings, comments)."""
    pkg = os.path.join(ROOT, "thermal3d_vision_b200")
    seen = 0
    for top in (pkg, os.path.join(ROOT, "dropin")):
        for dirpath, _, files in os.walk(top):
            for f in files:
                if not f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                    continue
                src = open(os.path.join(dirpath, f)).read()
                seen += 1
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                if f.endswith(".py"):
                    bad = [v for v in _runtime_strings(src) if "/root/reference" in v or v.startswith("oracle")]
                else:
                    code = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
                    code = re.sub(r"//[^\n]*", "", code)
                    bad = ["/root/reference"] if "/root/reference" in code else []
                assert not bad, (f, bad)
    assert seen > 20
