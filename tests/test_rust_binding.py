"""CPU tier: the Rust side of the boundary exists as files and stays in lock step with include/pna_cuda.h.

No Rust toolchain is in this image, so the crate (rust/pna-cuda-sys) cannot be compiled here; this test parses its source
instead: the `extern "C"` block must declare exactly the header's functions with matching arity, the #[repr(C)] structs must
have the header's field order and the sizes the ctypes binding (checked against the built library elsewhere) has, and the
seam patches must apply to the three reference files they name."""
import ctypes as C
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CRATE = os.path.join(ROOT, "rust", "pna-cuda-sys")

RUST_SIZES = {"u8": 1, "i32": 4, "u32": 4, "u64": 8, "f32": 4, "c_int": 4}


def _header_functions():
    hdr = open(os.path.join(ROOT, "include", "pna_cuda.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    out = {}
    for name, params in re.findall(r"\b(pna_cuda_\w+)\s*\(([^;{]*?)\)\s*;", hdr, flags=re.S):
        ps = [p for p in (x.strip() for x in params.split(",")) if p and p != "void"]
        out[name] = len(ps)
    return hdr, out


def _rust_source():
    return open(os.path.join(CRATE, "src", "lib.rs")).read()


def test_crate_files_exist():
    for f in ("Cargo.toml", "build.rs", os.path.join("src", "lib.rs")):
        assert os.path.getsize(os.path.join(CRATE, f)) > 200, f
    cargo = open(os.path.join(CRATE, "Cargo.toml")).read()
    assert 'name = "pna-cuda-sys"' in cargo and 'links = "pna_cuda"' in cargo
    build = open(os.path.join(CRATE, "build.rs")).read()
    assert "compute_100a" in build and "abi.cu" in build and ".cuda(true)" in build


def test_extern_block_matches_header():
    _, want = _header_functions()
    src = _rust_source()
    ext = src[src.index('extern "C" {'):]
    ext = ext[:ext.index("\n}\n")]
    got = {}
    for name, params in re.findall(r"pub fn (pna_cuda_\w+)\(([^;]*?)\)\s*(?:->\s*[^;]+)?;", ext, flags=re.S):
        got[name] = len([p for p in params.split(",") if p.strip()])
    assert set(got) == set(want), (sorted(set(want) - set(got)), sorted(set(got) - set(want)))
    assert got == want, {k: (got[k], want[k]) for k in want if got[k] != want[k]}
    assert len(want) >= 40


def _rust_struct(src, name):
    m = re.search(r"#\[repr\(C\)\]\s*(?:#\[derive\([^)]*\)\]\s*)?pub struct " + name + r" \{(.*?)\n\}", src, flags=re.S)
    assert m, name
    return [(f.strip(), t.strip()) for f, t in re.findall(r"pub (\w+):\s*([^,\n]+),", m.group(1))]


def _layout(fields):
    """size of a #[repr(C)] struct of scalars / pointers / byte arrays / nested spans on a 64-bit target"""
    off, align = 0, 1
    for _, t in fields:
        if t.startswith("*"):
            sz, al = 8, 8
        elif t.startswith("["):
            m = re.match(r"\[u8;\s*(\d+)\]", t)
            sz, al = int(m.group(1)), 1
        elif t == "pna_span":
            sz, al = 16, 8
        else:
            sz = al = RUST_SIZES[t]
        off = (off + al - 1) // al * al
        off += sz
        align = max(align, al)
    return (off + align - 1) // align * align


def test_repr_c_structs_match_header_and_ctypes(pna):
    import importlib
    ffi = importlib.import_module("portable-network-archive_b200._ffi")
    hdr, _ = _header_functions()
    src = _rust_source()
    pairs = {"pna_span": ffi.Span, "pna_buf": ffi.Buf, "pna_decode_desc": ffi.DecodeDesc, "pna_encode_desc": ffi.EncodeDesc}
    for name, ct in pairs.items():
        rf = _rust_struct(src, name)
        assert [f for f, _ in rf] == [f for f, *_ in ct._fields_], name             # same field order as the ctypes mirror
        assert _layout(rf) == C.sizeof(ct), (name, _layout(rf), C.sizeof(ct))       # same size
        m = re.search(r"typedef struct \{([^}]*)\}\s*" + name + r"\s*;", hdr, flags=re.S)   # and as the C header
        assert m, name
        c_fields = re.findall(r"(\w+)\s*(?:\[\d+\])?\s*[;,]", re.sub(r"/\*.*?\*/", "", m.group(1), flags=re.S))
        assert c_fields == [f for f, _ in rf], (name, c_fields)
    # the status / code constants
    for k, v in re.findall(r"\b(PNA_[A-Z_]+)\s*=\s*(\d+)", hdr):
        m = re.search(r"pub const " + k + r": \w+ = (\d+);", src)
        assert m and m.group(1) == v, k


def test_seam_patches_apply_to_the_reference(tmp_path):
    """tests/golden/reference_src holds, for every reference file (v0.37.0) a patch changes, the lines the patch's hunks
    replace and keep as context, hunk after hunk in file order.  The patches must apply to them without fuzz, so an edit
    to a patch that no longer matches the reference's code fails here."""
    pdir = os.path.join(ROOT, "rust", "patches")
    ref = os.path.join(ROOT, "tests", "golden", "reference_src")
    patches = sorted(f for f in os.listdir(pdir) if f.endswith(".patch"))
    assert [p[:4] for p in patches] == ["0001", "0002", "0003"]
    touched = set()
    for p in patches:
        text = open(os.path.join(pdir, p)).read()
        touched |= set(re.findall(r"^\+\+\+ b/(\S+)", text, flags=re.M))
    assert {"lib/src/format/chunk.rs", "lib/src/entry/read.rs", "lib/src/entry/write.rs"} <= touched
    # dry-run against a copy of the files
    for rel in touched:
        dst = tmp_path / rel
        dst.parent.mkdir(parents=True, exist_ok=True)
        dst.write_bytes(open(os.path.join(ref, rel), "rb").read())
    for p in patches:
        r = subprocess.run(["patch", "-p1", "--dry-run", "--fuzz=0", "-i", os.path.join(pdir, p)], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0, (p, r.stdout, r.stderr)
