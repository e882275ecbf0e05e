"""The Rust side of the drop-in (rust/gpu.rs + rust/patches/) cannot be compiled here — no cargo / rustc in the image — so
it is held to what CAN be checked mechanically:

* every `#[repr(C)]` struct and every `extern "C"` prototype of gpu.rs is the transcription of include/rayrs_b200.h:
  same fields in the same order with the same scalar types / array lengths / pointer-ness, same constants;
* the patches are purely additive (main.rs too: the call goes in front of the rayon tile loop, which stays, compiled out),
  well-formed for `patch -p1` (headers, hunk line counts, offsets), leave the patched files' delimiters balanced, and
  put their context lines where the upstream lines this repository records (SURVEY.md) are;
* everything gpu.rs uses from the patched modules (`BvhCursor`, `FlatGeom`, `FlatMaterial`, `Hittable::flatten`, ...) is
  defined by the patches.
"""
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
HEADER = (ROOT / "include" / "rayrs_b200.h").read_text()
GPU_RS = (ROOT / "rust" / "gpu.rs").read_text()
PATCHES = sorted((ROOT / "rust" / "patches").glob("*.patch"))

C_SCALAR = {"uint32_t": "u32", "int32_t": "i32", "uint64_t": "u64", "int64_t": "i64", "double": "f64", "float": "f32",
            "int": "c_int", "char": "c_char", "uint8_t": "u8", "size_t": "usize", "void": "c_void"}


def _strip_c_comments(s):
    return re.sub(r"/\*.*?\*/", "", s, flags=re.S)


def _c_structs():
    """name -> [(field, rust-style type string)] for every `typedef struct X { ... } X;` of the header"""
    out = {}
    for m in re.finditer(r"typedef struct (\w+) \{(.*?)\} \1;", _strip_c_comments(HEADER), flags=re.S):
        fields = []
        for decl in m.group(2).split(";"):
            decl = " ".join(decl.split())
            if not decl:
                continue
            is_ptr = "*" in decl
            decl_np = decl.replace("*", " ").replace("const ", "")
            parts = decl_np.split()
            ctype, names = parts[0], " ".join(parts[1:])
            for name in names.split(","):
                name = name.strip()
                arr = re.match(r"(\w+)\[(\d+)\]$", name)
                base = C_SCALAR.get(ctype, ctype)
                if is_ptr:
                    fields.append((name, "ptr " + base))
                elif arr:
                    fields.append((arr.group(1), f"[{base}; {arr.group(2)}]"))
                else:
                    fields.append((name, base))
        out[m.group(1)] = fields
    return out


def _rust_structs():
    out = {}
    for m in re.finditer(r"#\[repr\(C\)\]\s*(?:#\[derive\([^\]]*\)\]\s*)?pub struct (\w+) \{(.*?)\n\}", GPU_RS, flags=re.S):
        fields = []
        for line in m.group(2).splitlines():
            line = line.split("//")[0].strip().rstrip(",")
            fm = re.match(r"(?:pub )?(\w+): (.+)$", line)
            if not fm:
                continue
            name, typ = fm.group(1), fm.group(2).strip()
            if typ.startswith("*const ") or typ.startswith("*mut "):
                typ = "ptr " + typ.split(" ", 1)[1]
            fields.append((name.rstrip("_"), typ))
        out[m.group(1)] = fields
    return out


def test_repr_c_structs_are_the_headers():
    c, r = _c_structs(), _rust_structs()
    checked = 0
    for name, rf in r.items():
        if name in ("RrsScene", "RrsComm"):  # opaque handles: `typedef struct X X;` in the header
            assert re.search(rf"typedef struct {name} {name};", HEADER)
            continue
        assert name in c, f"gpu.rs declares {name}, the header does not"
        assert rf == c[name], f"{name}: gpu.rs {rf} != header {c[name]}"
        checked += 1
    # the structs that cross the FFI on the render path must all be there
    for need in ("RrsPrim", "RrsMaterial", "RrsEmission", "RrsNode", "RrsNodeF64", "RrsSceneDesc", "RrsCamera", "RrsRenderParams",
                 "RrsStats"):
        assert need in r, need
    assert checked >= 9


def _c_prototypes():
    out = {}
    text = _strip_c_comments(HEADER)
    for m in re.finditer(r"^(int|void|const char\*) (rrs_\w+)\((.*?)\);", text, flags=re.S | re.M):
        ret, name, args = m.group(1), m.group(2), " ".join(m.group(3).split())
        params = []
        if args != "void":
            for a in args.split(","):
                a = a.strip()
                stars = a.count("*")
                toks = a.replace("*", " ").replace("const ", "").split()
                base = C_SCALAR.get(toks[0], toks[0])
                params.append("ptr" * 0 + ("*" * stars) + base)
        out[name] = ({"int": "c_int", "void": "", "const char*": "*c_char"}[ret], params)
    return out


def _rust_prototypes():
    out = {}
    block = re.search(r'extern "C" \{(.*?)\n\}', GPU_RS, flags=re.S).group(1)
    for m in re.finditer(r"fn (rrs_\w+)\((.*?)\)\s*(?:->\s*([^;]+))?;", block, flags=re.S):
        name, args, ret = m.group(1), " ".join(m.group(2).split()), (m.group(3) or "").strip()
        params = []
        for a in filter(None, (x.strip() for x in args.split(","))):
            typ = a.split(":", 1)[1].strip()
            stars = typ.count("*")
            base = typ.replace("*const", "").replace("*mut", "").strip()
            params.append("*" * stars + base)
        ret = ret.replace("*const ", "*").replace("*mut ", "*")
        out[name] = (ret, params)
    return out


def test_extern_block_matches_the_header_prototypes():
    c, r = _c_prototypes(), _rust_prototypes()
    assert len(r) >= 10
    for name, (ret, params) in r.items():
        assert name in c, f"gpu.rs binds {name}, which the header does not declare"
        assert ret == c[name][0], (name, ret, c[name][0])
        assert params == c[name][1], (name, params, c[name][1])
    # the render path: scene creation (one and several GPUs), both render calls, the communicator, stats, errors
    for need in ("rrs_scene_create", "rrs_scene_create_multi", "rrs_scene_destroy", "rrs_render", "rrs_render_multi",
                 "rrs_comm_init_all", "rrs_comm_destroy", "rrs_stats", "rrs_last_error", "rrs_device_count"):
        assert need in r, need


def test_constants_match_the_header():
    def c_define(name):
        m = re.search(rf"#define {name} (0x[0-9A-Fa-f]+|\d+)u?", HEADER)
        assert m, name
        return int(m.group(1), 0)

    def rust_const(name):
        m = re.search(rf"pub const {name}: u32 = ([0-9A-Fa-fx_]+);", GPU_RS)
        assert m, name
        return int(m.group(1).replace("_", ""), 0)

    for name in ("RRS_ABI_VERSION", "RRS_REF_LEAF", "RRS_REF_EMPTY"):
        assert rust_const(name) == c_define(name), name
    # material tags travel as the declaration order of `enum Material` (material.rs:57-68) == RrsMaterialTag
    tags = re.search(r"typedef enum RrsMaterialTag \{(.*?)\}", HEADER, flags=re.S).group(1)
    order = [t.split("=")[0].strip() for t in tags.split(",") if t.strip()]
    assert [int(t.split("=")[1]) for t in tags.split(",") if t.strip()] == list(range(len(order)))
    assert order[0] == "RRS_MAT_LAMBERTIAN" and order[-1] == "RRS_MAT_NO_REFLECT" and len(order) == 9


def test_patches_only_add_lines():
    assert len(PATCHES) == 5
    for p in PATCHES:
        removed = [l for l in p.read_text().splitlines() if l.startswith("-") and not l.startswith("---")]
        assert not removed, (p.name, removed[:3])  # main.rs.patch too: the CPU tile loop stays, compiled out


# The upstream file each patch applies to.  The upstream sources are not part of this repository, so what follows holds
# the patches to what `patch -p1` needs of them and to the few upstream lines this repository records (SURVEY.md).
UPSTREAM = {"lib.rs.patch": "rayrs-lib/src/lib.rs", "geometry.rs.patch": "rayrs-lib/src/geometry.rs",
            "material.rs.patch": "rayrs-lib/src/material.rs", "bvh.rs.patch": "rayrs-lib/src/bvh.rs",
            "main.rs.patch": "rayrs/src/main.rs"}
# rayrs/src/main.rs as SURVEY.md records it: the tile loop (`into_par_iter` over 16x16 tiles) spans lines 61-94,
# between `Image::blocks` (57) and `Image::from_blocks` (101)
MAIN_RS_LINES = {57: "Image::blocks(", 101: "Image::from_blocks("}
TILE_LOOP = (61, 94)


def _hunks(patch):
    """[(old_start, old_len, new_start, new_len, [(old line number the line sits at or before, line)])] of a unified diff"""
    lines = patch.read_text().splitlines()
    out = []
    for ln in lines[2:]:
        m = re.fullmatch(r"@@ -(\d+),(\d+) \+(\d+),(\d+) @@.*", ln)
        if m:
            out.append(tuple(map(int, m.groups())) + ([],))
            old = out[-1][0]
            continue
        assert out, (patch.name, ln)
        out[-1][4].append((old, ln))
        old += ln[:1] == " "
    return out


def test_patches_are_well_formed_unified_diffs():
    """a/ and b/ headers naming the upstream file; hunk headers whose line counts are those of their bodies; hunks in
    order without overlap, each new-file offset the old one shifted by the lines earlier hunks add."""
    assert sorted(p.name for p in PATCHES) == sorted(UPSTREAM)
    for p in PATCHES:
        head = [ln.split("\t")[0] for ln in p.read_text().splitlines()[:2]]   # a timestamp may follow a tab
        assert head == [f"--- a/{UPSTREAM[p.name]}", f"+++ b/{UPSTREAM[p.name]}"], (p.name, head)
        hunks = _hunks(p)
        assert hunks, p.name
        shift, old_end = 0, 0
        for o0, ol, n0, nl, body in hunks:
            kinds = [ln[:1] for _, ln in body]
            assert set(kinds) <= {" ", "+"}, (p.name, o0, set(kinds))
            assert (ol, nl) == (kinds.count(" "), len(kinds)), (p.name, o0, ol, nl)
            assert o0 > old_end and n0 == o0 + shift, (p.name, o0, n0, shift)
            old_end, shift = o0 + ol - 1, shift + kinds.count("+")


def test_patched_sources_keep_their_delimiters_balanced():
    """The patches only add lines to sources that compile, so a patched file balances its braces and parentheses
    exactly when the lines its patch adds do."""
    for p in PATCHES:
        text = _code_only("\n".join(ln[1:] for _, ln in sum((h[4] for h in _hunks(p)), []) if ln[:1] == "+"))
        for a, b in ("{}", "()", "[]"):
            assert text.count(a) == text.count(b), (p.name, a, text.count(a), text.count(b))


def test_lib_rs_declares_the_module_and_main_rs_compiles_out_the_tile_loop():
    lib = [ln[1:].strip() for _, ln in _hunks(ROOT / "rust" / "patches" / "lib.rs.patch")[0][4] if ln[:1] == "+"]
    assert "pub mod gpu;" in lib
    body = sum((h[4] for h in _hunks(ROOT / "rust" / "patches" / "main.rs.patch")), [])
    # the context lines sit where the recorded upstream file has them
    for at, text in MAIN_RS_LINES.items():
        assert any(old == at and ln[:1] == " " and text in ln for old, ln in body), (at, text)
    added = [(old, ln[1:].strip()) for old, ln in body if ln[:1] == "+"]
    code = [ln for _, ln in added]
    at = {ln: k for k, ln in enumerate(code)}
    # the GPU call, then `#[cfg(any())] let image = {` (never true) in front of the tile loop, and its `};` after it
    call = next(k for k, ln in enumerate(code) if "render_gpu(" in ln)
    assert call < at["#[cfg(any())]"] == at["let image = {"] - 1 < at["};"]
    assert added[at["let image = {"]][0] <= TILE_LOOP[0] and added[at["};"]][0] > TILE_LOOP[1]


def test_gpu_rs_uses_only_what_the_patches_define():
    added = "\n".join(l[1:] for p in PATCHES for l in p.read_text().splitlines() if l.startswith("+") and not l.startswith("+++"))
    for item in ("BvhCursor", "FlatGeom", "FlatMaterial"):
        assert re.search(rf"(struct|enum) {item}\b", added), f"{item} is imported by gpu.rs and defined by no patch"
    assert "pub mod gpu;" in added
    for method in ("fn cursor", "fn flatten", "fn flat"):
        assert method in added, method
    # every method gpu.rs calls on a cursor exists on BvhCursor
    cursor_impl = added[added.index("impl<'a> BvhCursor<'a>"):]
    defined = set(re.findall(r"pub\(crate\) fn (\w+)", cursor_impl))
    used = set(re.findall(r"\b(?:cursor|node|child|c|root)\.(\w+)\(", GPU_RS)) & {"bbox", "children", "object", "is_leaf", "len"}
    assert used <= defined | {"len"}, (used, defined)


def _code_only(rust):
    """Rust source without comments, string and char literals (a cheap stand-in for the compiler that is not here)"""
    text = re.sub(r"//.*", "", rust)
    text = re.sub(r'"(?:\\.|[^"\\])*"', '""', text)
    return re.sub(r"'(?:\\.|[^'\\])'", "' '", text)


def test_gpu_rs_balances_its_delimiters():
    text = _code_only(GPU_RS)
    for a, b in ("{}", "()", "[]"):
        assert text.count(a) == text.count(b), (a, text.count(a), text.count(b))
