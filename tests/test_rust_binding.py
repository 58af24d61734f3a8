"""The Rust -sys crate (rust/shimmer-b200-sys, sources only: no rustc in this image) must declare exactly what
include/shimmer_b200.h declares: same symbols, same arity, same struct fields in the same order, same constants."""
import os
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
HEADER = (ROOT / "include" / "shimmer_b200.h").read_text()
RUST = (ROOT / "rust" / "shimmer-b200-sys" / "src" / "lib.rs").read_text()


def _strip_c_comments(s):
    return re.sub(r"/\*.*?\*/", " ", s, flags=re.S)


def _c_functions():
    src = _strip_c_comments(HEADER)
    out = {}
    for m in re.finditer(r"\b(shim_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args in ("", "void") else len(args.split(","))
    return out


def _rust_functions():
    block = RUST[RUST.index('extern "C" {'):]
    out = {}
    for m in re.finditer(r"pub fn (shim_[a-z0-9_]+)\s*\((.*?)\)\s*(?:->\s*[^;]+)?;", block, flags=re.S):
        args = [a for a in m.group(2).replace("\n", " ").split(",") if a.strip()]
        out[m.group(1)] = len(args)
    return out


def test_every_header_symbol_is_declared_with_the_same_arity():
    c, r = _c_functions(), _rust_functions()
    assert len(c) >= 40
    assert set(c) == set(r), (sorted(set(c) - set(r)), sorted(set(r) - set(c)))
    assert {k: (c[k], r[k]) for k in c if c[k] != r[k]} == {}


def _c_struct_fields(name):
    src = _strip_c_comments(HEADER)
    body = re.search(r"typedef struct %s\s*\{(.*?)\}\s*%s\s*;" % (name, name), src, flags=re.S).group(1)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        names = decl.split(None, 1)[1]
        fields += [re.sub(r"\[.*?\]", "", n).strip() for n in names.split(",")]
    return fields


def _rust_struct_fields(name):
    body = re.search(r"pub struct %s\s*\{(.*?)\n\}" % name, RUST, flags=re.S).group(1)
    return re.findall(r"pub ([a-z0-9_]+)\s*:", body)


def test_pod_structs_have_the_headers_fields_in_order():
    for name in ("shim_camera", "shim_render_params", "shim_stats"):
        assert _c_struct_fields(name) == _rust_struct_fields(name), name


def test_constants_agree():
    src = _strip_c_comments(HEADER)
    c = {k: int(v) for k, v in re.findall(r"\b(SHIM_[A-Z0-9_]+)\s*=\s*(-?\d+)", src)}
    r = {k: int(v) for k, v in re.findall(r"pub const (SHIM_[A-Z0-9_]+)\s*:\s*\w+\s*=\s*(-?\d+)\s*;", RUST)}
    assert c and c == r


def test_library_exports_what_the_rust_crate_links_against():
    from raytracinginoneweekendinrust_b200 import capi
    lib = capi.load_library()
    for name in _rust_functions():
        assert hasattr(lib, name), name


PATCH = ROOT / "rust" / "shimmer-patch" / "shimmer-b200.patch"
# the reference crate's files the patch changes, as far as the patch and make_patch.py record them
# (tests/golden/make_reference_excerpt.py); SHIMMER_REFERENCE_DIR may name a full checkout instead
REFERENCE = Path(os.environ.get("SHIMMER_REFERENCE_DIR") or ROOT / "tests" / "golden" / "reference_excerpt")


def test_reference_patch_applies_cleanly(tmp_path):
    """rust/shimmer-patch/shimmer-b200.patch (the `record` method of every implementor, Bvh upload, Camera POD, the new
    body of Renderer::render, src/backend.rs) applies to the reference crate without fuzz and is what make_patch.py
    generates from it.  The Rust code is applied, not compiled."""
    import shutil
    import subprocess
    import sys
    ref = REFERENCE.resolve()
    work = tmp_path / "shimmer"
    work.mkdir()
    shutil.copy(ref / "Cargo.toml", work / "Cargo.toml")
    shutil.copytree(ref / "src", work / "src")
    out = subprocess.run(["patch", "-p1", "--no-backup-if-mismatch", "-i", str(PATCH)], cwd=work, capture_output=True, text=True)
    assert out.returncode == 0 and "FAILED" not in out.stdout and "fuzz" not in out.stdout, out.stdout + out.stderr
    assert (work / "src" / "backend.rs").read_text() == (ROOT / "rust" / "shimmer-patch" / "backend.rs").read_text()
    # every implementor the crate ships overrides `record`: 4 textures, 5 materials, 12 hittables
    n = sum(p.read_text().count("fn record(&self, r: &mut crate::backend::Recorder)") for p in (work / "src").rglob("*.rs"))
    assert n == 4 + 5 + 12, n
    assert "crate::backend::render_on_device(" in (work / "src" / "renderer.rs").read_text()
    # the committed patch is what the generator produces today
    regen = tmp_path / "regenerated.patch"
    gen = subprocess.run([sys.executable, str(ROOT / "rust" / "shimmer-patch" / "make_patch.py"), str(ref), str(regen)],
                         capture_output=True, text=True)
    assert gen.returncode == 0, gen.stderr
    assert regen.read_bytes() == PATCH.read_bytes()
