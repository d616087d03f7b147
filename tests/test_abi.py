"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol
include/bellman_b200.h declares, and refuses to run without a CUDA device (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

import bellman_b200 as bb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    names = set()
    for hdr in ("bellman_b200.h", "bellman_b200_diag.h"):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names |= set(re.findall(r"\b(bb_[a-z0-9_]+)\s*\(", text))
    return sorted(names)


def test_public_header_holds_no_diagnostics():
    text = open(os.path.join(ROOT, "include", "bellman_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    assert not re.search(r"\bbb_(selftest|synth|diag)_", text)


def test_library_is_built_in_tree():
    assert os.path.exists(bb.LIB_PATH), "run __graft_entry__.build() first"
    assert os.path.dirname(bb.LIB_PATH) == os.path.join(ROOT, "bellman_b200")


def test_every_declared_symbol_is_exported():
    lib = bb.load_library()
    names = declared_symbols()
    assert len(names) >= 25
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/bellman_b200.h but not exported"


def test_rust_sys_crate_binds_every_public_symbol():
    """rust/bellman-b200-sys/src/lib.rs (source only: no Rust toolchain here) declares every function of the
    public header with the same number of parameters."""
    def params(text, name):
        m = re.search(r"\b%s\s*\(" % name, text)
        assert m, name
        depth, i = 0, m.end() - 1
        for j in range(i, len(text)):
            depth += text[j] == "("
            depth -= text[j] == ")"
            if depth == 0:
                inner = text[i + 1:j].strip()
                break
        if inner in ("", "void"):
            return 0
        return len([x for x in re.sub(r"\[[^\]]*\]", "", inner).split(",") if x.strip()])
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "bellman_b200.h")).read(), flags=re.S)
    rs = re.sub(r"//[^\n]*", "", open(os.path.join(ROOT, "rust", "bellman-b200-sys", "src", "lib.rs")).read())
    names = sorted(set(re.findall(r"\b(bb_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 30
    for name in names:
        assert re.search(r"pub fn %s\s*\(" % name, rs), f"{name} missing from the -sys crate"
        assert params(hdr, name) == params(rs[rs.index("pub fn " + name):], name), name


def test_header_is_plain_c():
    """the boundary is a C ABI: the header must compile as C99 (no C++ or torch types)"""
    import subprocess, tempfile
    src = "#include \"bellman_b200_diag.h\"\nint main(void) { bb_witness w; bb_crs_desc d; (void)w; (void)d; return BB_PARTIALS_BYTES == 960 ? 0 : 1; }\n"
    with tempfile.NamedTemporaryFile("w", suffix=".c", delete=False) as f:
        f.write(src)
    res = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                          "-fsyntax-only", f.name], capture_output=True, text=True)
    os.unlink(f.name)
    assert res.returncode == 0, res.stderr


def test_no_cpu_fallback_without_device():
    """in a process that sees no CUDA device (none is made visible, so this runs on a GPU machine too)"""
    code = ("import bellman_b200 as bb\n"
            "try:\n    bb.Worker()\n"
            "except bb.BackendError as e:\n    print(e)\n"
            "else:\n    raise SystemExit('a Worker was created without a CUDA device')\n")
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "no CPU fallback" in res.stdout or "18" in res.stdout


def test_density_packing_matches_bitvec_lsb0():
    words, n = bb.pack_density([1, 0, 0, 1] + [0] * 60 + [1])
    assert n == 65 and int(words[0]) == 0b1001 and int(words[1]) == 1
    words, n = bb.pack_density([])
    assert n == 0 and words.shape[0] >= 1


def test_product_does_not_reference_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py may import, link or execute oracle/."""
    bad = re.compile(r"#include[^\n]*oracle|import\s+oracle|from\s+oracle|oracle/|liboracle|o1_[a-z]", re.I)
    for dirpath, _, files in os.walk(os.path.join(ROOT, "bellman_b200")):
        if "build" in dirpath.split(os.sep):
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")) or f == "Makefile":
                src = open(os.path.join(dirpath, f), errors="replace").read()
                assert not bad.search(src), (dirpath, f, bad.search(src).group(0))
