"""Host mesh loaders (rayrs_b200/host/mesh_io.cpp): the PLY loader that completes the reference's
commented-out `ply` crate (header grammar, state machine and error messages of ply/src/lib.rs:31-317) and
the OBJ loader of wavefront_obj.rs:15-44.  The checker is an independent numpy/struct restatement."""
import struct

import numpy as np
import pytest

from rayrs_b200 import mesh, scenes

TYPES = {"char": "b", "uchar": "B", "short": "h", "ushort": "H", "int": "i", "uint": "I", "float": "f", "double": "d"}


def make_ply(fmt, verts, faces, vtype="float", ltype="uchar", itype="int", extra_vertex_props=(), comments=(),
             extra_element=None, index_name="vertex_indices"):
    """bytes of a PLY file built with struct, independent of the C++ writer."""
    hdr = ["ply", f"format {fmt} 1.0"] + [f"comment {c}" for c in comments]
    hdr += [f"element vertex {len(verts)}"] + [f"property {vtype} {n}" for n in "xyz"]
    hdr += [f"property {t} {n}" for t, n in extra_vertex_props]
    if extra_element:
        hdr += [f"element {extra_element[0]} {len(extra_element[2])}", f"property {extra_element[1]} value"]
    hdr += [f"element face {len(faces)}", f"property list {ltype} {itype} {index_name}", "end_header"]
    out = ("\n".join(hdr) + "\n").encode()
    if fmt == "ascii":
        body = []
        for v in verts:
            body.append(" ".join(repr(float(x)) for x in v) + "".join(f" {i + 1}" for i, _ in enumerate(extra_vertex_props)))
        if extra_element:
            body += [str(x) for x in extra_element[2]]
        for f in faces:
            body.append(" ".join(str(x) for x in [len(f)] + list(f)))
        return out + ("\n".join(body) + "\n").encode()
    e = "<" if fmt == "binary_little_endian" else ">"
    for v in verts:
        out += struct.pack(e + 3 * TYPES[vtype], *[float(x) for x in v])
        for i, (t, _) in enumerate(extra_vertex_props):
            out += struct.pack(e + TYPES[t], i + 1)
    if extra_element:
        for x in extra_element[2]:
            out += struct.pack(e + TYPES[extra_element[1]], x)
    for f in faces:
        out += struct.pack(e + TYPES[ltype], len(f)) + struct.pack(e + len(f) * TYPES[itype], *f)
    return out


VERTS = np.array([[0, 0, 0], [1, 0, 0.5], [1, 1, 0.25], [0, 1, -0.125], [0.5, 0.5, 2]], dtype=np.float64)
FACES = [[0, 1, 2], [0, 2, 3], [0, 1, 2, 3], [4, 3, 2, 1, 0]]  # triangles, a quad, a pentagon


def fan(verts, faces):
    out = []
    for f in faces:
        for k in range(1, len(f) - 1):
            out.append([verts[f[0]], verts[f[k]], verts[f[k + 1]]])
    return np.array(out, dtype=np.float64)


@pytest.mark.parametrize("fmt", ["ascii", "binary_little_endian", "binary_big_endian"])
@pytest.mark.parametrize("vtype,ltype,itype", [("float", "uchar", "int"), ("double", "ushort", "uint"), ("float", "int", "short")])
def test_ply_formats_types_and_polygons(tmp_path, native_built, fmt, vtype, ltype, itype):
    data = make_ply(fmt, VERTS, FACES, vtype, ltype, itype, extra_vertex_props=[("uchar", "red"), ("short", "quality")],
                    comments=["made by the test", "second"], extra_element=("weights", "double", [0.5, 1.5, 2.5]))
    path = tmp_path / "m.ply"
    path.write_bytes(data)
    tris = mesh.load_ply_file(path)
    assert tris.shape == (1 + 1 + 2 + 3, 3, 3)
    assert np.array_equal(tris, fan(VERTS, FACES))  # every test coordinate is exact in float32
    desc = mesh.ply_describe(data)
    assert desc[0] == f"format {fmt} 1.0"
    assert desc[1:3] == ["comment made by the test", "comment second"]
    assert "element vertex 5" in desc and "element weights 3" in desc and "element face 4" in desc
    assert any(l.startswith("list ") and l.endswith("vertex_indices") for l in desc)


def test_ply_vertex_index_alias_and_crlf(tmp_path, native_built):
    data = make_ply("ascii", VERTS, FACES[:2], index_name="vertex_index").replace(b"\n", b"\r\n")
    path = tmp_path / "crlf.ply"
    path.write_bytes(data)
    assert np.array_equal(mesh.load_ply_file(path), fan(VERTS, FACES[:2]))


@pytest.mark.parametrize("fmt", ["ascii", "binary_little_endian", "binary_big_endian"])
def test_ply_writer_roundtrip(tmp_path, native_built, fmt):
    verts, faces = scenes.torus_mesh(24, 12)
    path = tmp_path / "torus.ply"
    mesh.write_ply(path, verts, faces, fmt)
    tris = mesh.load_ply_file(path)
    assert np.array_equal(tris, scenes.mesh_triangles(verts, faces))  # %.9g round-trips float32
    raw = path.read_bytes()
    assert raw.startswith(b"ply\nformat " + fmt.encode() + b" 1.0\n")
    if fmt != "ascii":  # float32 xyz + (uchar count, 3 x int32) per face after the header
        body = raw[raw.index(b"end_header\n") + 11:]
        assert len(body) == verts.shape[0] * 12 + faces.shape[0] * 13
        e = "<" if fmt == "binary_little_endian" else ">"
        assert np.array_equal(np.frombuffer(body[: verts.size * 4], dtype=e + "f4").reshape(-1, 3), verts)


def test_mesh_scene_goes_through_the_ply_loader(native_built, tmp_path, monkeypatch):
    import tempfile
    monkeypatch.setattr(tempfile, "tempdir", str(tmp_path))
    spec = scenes.copper_torus(20, 10, 64, 48)
    verts, faces = scenes.torus_mesh(20, 10)
    tri_rows = spec.tables().objs
    tri_rows = tri_rows[tri_rows[:, 0] == 2][:, 3:12].reshape(-1, 3, 3)
    assert np.array_equal(tri_rows, scenes.mesh_triangles(verts, faces))
    # the PLY file lived in a directory of its own, gone with it: nothing shared with other users is left behind
    assert list(tmp_path.iterdir()) == []


HEAD = "ply\nformat ascii 1.0\nelement vertex 1\nproperty float x\nproperty float y\nproperty float z\n"
TAIL = "element face 0\nproperty list uchar int vertex_indices\nend_header\n0 0 0\n"


@pytest.mark.parametrize("text,message", [
    ("plyx\n", "unknown ply keyword: plyx"),                                   # from_line, lib.rs:60-65
    ("format ascii 1.0\n", "expected 'ply' identifier"),                       # Start state, lib.rs:235-241
    ("ply\nelement vertex 1\n", "expected format specification"),              # Format state
    ("ply\nformat ascii\n", "invalid format specifier"),                       # parse_format
    ("ply\nformat ascii 2.0\n", "invalid version: 2.0, valid versions: 1.0"),
    ("ply\nformat text 1.0\n", "invalid format: text"),                        # PlyFormat::from_string
    ("ply\nformat ascii 1.0\nproperty float x\n", "expected 'element' keyword"),  # StartElement state
    ("ply\nformat ascii 1.0\nelement vertex\n", "invalid element"),            # parse_element
    ("ply\nformat ascii 1.0\nelement vertex ten\n", "invalid digit found in string"),
    ("ply\nformat ascii 1.0\nelement vertex 1\nelement face 1\n", "expected 'property' keyword"),  # NewElement state
    ("ply\nformat ascii 1.0\nelement vertex 1\nproperty float\n", "invalid property"),            # parse_property
    ("ply\nformat ascii 1.0\nelement vertex 1\nproperty list uchar x\n", "invalid property"),
    ("ply\nformat ascii 1.0\nelement vertex 1\nproperty half x\n", "invalid property type: half"),
    (HEAD + "ply\n", "expected properties or new element"),                    # InElement state
    (HEAD, "unexpected EOF"),                                                  # Ply::load, lib.rs:340-346
    (HEAD + TAIL.replace("0 0 0\n", "0 0\n"), "unexpected EOF"),               # truncated body
    (HEAD + TAIL.replace("0 0 0\n", "0 zero 0\n"), "invalid value in element data"),
    ("ply\nformat ascii 1.0\n\nelement vertex 1\n", "unknown ply keyword: "),  # an empty line is not a keyword
])
def test_ply_header_errors(native_built, text, message):
    with pytest.raises(mesh.MeshError) as e:
        mesh.ply_describe(text.encode())
    assert str(e.value) == message


def test_ply_semantic_errors(tmp_path, native_built):
    p = tmp_path / "bad.ply"
    p.write_bytes(make_ply("ascii", VERTS, [[0, 1, 9]]))
    with pytest.raises(mesh.MeshError, match="face index out of range"):
        mesh.load_ply_file(p)
    p.write_bytes(b"ply\nformat ascii 1.0\nelement vertex 1\nproperty float x\nend_header\n0\n")
    with pytest.raises(mesh.MeshError, match="no vertex/face elements"):
        mesh.load_ply_file(p)
    with pytest.raises(mesh.MeshError, match="No such file"):
        mesh.load_ply_file(tmp_path / "missing.ply")
    # an empty mesh is not an error
    p.write_bytes(make_ply("binary_little_endian", VERTS[:0], []))
    assert mesh.load_ply_file(p).shape == (0, 3, 3)


def test_obj_loader_matches_reference_rules(tmp_path, native_built):
    """wavefront_obj.rs:15-44: split on single spaces, 'v' and 'f' lines only, 1-based indices."""
    p = tmp_path / "m.obj"
    p.write_text("# comment\no thing\nv 0 0 0\nv 1 0 0.5\nv 1 1 0.25\nvn 0 0 1\nv 0 1 -0.125\nf 1 2 3\nf 1 3 4\ns off\n")
    tris = mesh.load_obj_file(p)
    assert np.array_equal(tris, fan(VERTS, FACES[:2]))
    p.write_text("v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1/1 2/2 3/3\n")  # the reference unwrap()s a ParseIntError here
    with pytest.raises(mesh.MeshError, match="ParseIntError"):
        mesh.load_obj_file(p)
    p.write_text("v 0 0 0\nf 1 2 3\n")
    with pytest.raises(mesh.MeshError, match="index out of bounds"):
        mesh.load_obj_file(p)
    p.write_text("v  0 0 0\n")  # double space -> empty field -> ParseFloatError in the reference
    with pytest.raises(mesh.MeshError, match="ParseFloatError"):
        mesh.load_obj_file(p)


def test_obj_spheres_loader(tmp_path, native_built):
    """wavefront_obj.rs:46-66: a sphere per 'v' line; faces and everything else ignored."""
    from rayrs_b200.api import Material, Object, build_tables
    p = tmp_path / "pts.obj"
    p.write_text("v 0 0 0\nv 1 0 0.5\nf 1 2 1\nvn 0 0 1\nv -2 3 4\n")
    c = mesh.load_obj_file_spheres(p)
    assert np.array_equal(c, [[0, 0, 0], [1, 0, 0.5], [-2, 3, 4]])
    rows = build_tables([Object.from_spheres(c, 0.25, Material.no_reflect())]).objs   # Object::from_spheres lib.rs:423-431
    assert rows.shape[0] == 3 and (rows[:, 0] == 0).all() and (rows[:, 3] == 0.25).all() and np.array_equal(rows[:, 4:7], c)
    p.write_text("v 0 0\n")
    with pytest.raises(mesh.MeshError, match="index out of bounds"):
        mesh.load_obj_file_spheres(p)
