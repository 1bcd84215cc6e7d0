"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/rs_b200.h declares, and the ctypes prototype table covers the whole header.
No compute calls are made (no GPU needed)."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "rs_b200.h")


def _declared():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rs_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_entry_points():
    names = _declared()
    for must in ("rs_embed_gather_fwd", "rs_embed_segsum_adam", "rs_route_ids", "rs_interacting_fwd",
                 "rs_interacting_bwd", "rs_din_fwd", "rs_din_bwd", "rs_gemm", "rs_logit_head_fwd_bwd"):
        assert must in names


def test_library_exports_every_declared_symbol_at_abi_v6():
    from recommendsystem_b200 import cabi
    if not cabi.LIB_PATH.exists():
        pytest.skip("library not built (run __graft_entry__.build())")
    lib = cabi.load()
    assert cabi.MISSING == []
    out = subprocess.run(["nm", "-D", "--defined-only", str(cabi.LIB_PATH)], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\bT (rs_[a-z0-9_]+)", out))
    declared = set(_declared())
    assert declared <= exported, sorted(declared - exported)
    assert lib.rs_abi_version() == 6 and lib.rs_built_for_sm100a() == 1


def test_prototype_table_matches_header():
    from recommendsystem_b200 import cabi
    assert sorted(cabi.PROTOTYPES) == _declared()


def test_prototype_arity_matches_header():
    """Argument counts in the ctypes table equal the parameter counts in the header."""
    from recommendsystem_b200 import cabi
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for name, (_, args) in cabi.PROTOTYPES.items():
        m = re.search(r"\b" + name + r"\s*\(([^;]*?)\)\s*;", text, flags=re.S)
        assert m, name
        params = m.group(1).strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert n == len(args), (name, n, len(args))


def test_no_cpu_fallback_for_host_tensors():
    import torch
    from recommendsystem_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.transpose2d(torch.zeros(4, 4))


def test_product_never_imports_the_oracle_or_the_reference():
    """oracle/ is test infrastructure: only tests/, __graft_entry__.smoke() and bench.py's CPU legs may use it, and
    nothing that runs on the GPU box may read /root/reference.  Enforced on the sources (AST import scan)."""
    import ast
    import pathlib
    root = pathlib.Path(__file__).resolve().parent.parent
    offenders = []
    for path in sorted((root / "recommendsystem_b200").rglob("*.py")):
        tree = ast.parse(path.read_text())
        for node in ast.walk(tree):
            names = []
            if isinstance(node, ast.Import):
                names = [a.name for a in node.names]
            elif isinstance(node, ast.ImportFrom):
                names = [node.module or ""]
            if any(n == "oracle" or n.startswith("oracle.") for n in names):
                offenders.append(f"{path.relative_to(root)}:{node.lineno}")
        if "/root/reference" in path.read_text():
            offenders.append(f"{path.relative_to(root)}: mentions /root/reference")
    assert not offenders, offenders
    # bench.py and __graft_entry__.py may import the oracle, but only inside the functions that are the CPU legs
    for fname, allowed in (("bench.py", {"cpu_autoint_samples_per_s", "run_reference"}), ("__graft_entry__.py", {"smoke", "build"})):
        tree = ast.parse((root / fname).read_text())
        for fn in [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef)]:
            for node in ast.walk(fn):
                mods = [a.name for a in node.names] if isinstance(node, ast.Import) else (
                    [node.module or ""] if isinstance(node, ast.ImportFrom) else [])
                if any(m == "oracle" or m.startswith("oracle.") for m in mods):
                    assert fn.name in allowed, f"{fname}:{node.lineno} imports oracle inside {fn.name}()"
        top = [n for n in tree.body if isinstance(n, (ast.Import, ast.ImportFrom))]
        for node in top:
            mods = [a.name for a in node.names] if isinstance(node, ast.Import) else [node.module or ""]
            assert not any(m == "oracle" or m.startswith("oracle.") for m in mods), f"{fname}: top-level oracle import"
        assert "/root/reference" not in (root / fname).read_text(), fname
