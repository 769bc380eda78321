#!/usr/bin/env python
"""Writes tests/golden/reference_excerpt.tar.xz: the part of SebLague/Ray-Tracing's Unity project that the scene reader consumes,
cut down so that the tests which read the original scenes run from this repository alone.

    python tests/golden/make_reference_excerpt.py <checkout of SebLague/Ray-Tracing>

What the archive holds (paths as in the original project):
  Assets/Scenes/<scene>.unity      the five shipped scenes with only the documents the reader uses (GameObject, Transform, Camera,
                                   MeshFilter, MonoBehaviour); materials, renderers, colliders, lights and render settings are dropped.
  Assets/Graphics/<mesh>.meta      the assets' .meta files unchanged (guids, normal import settings).
  Assets/Graphics/<mesh>           the meshes, cut down: an .obj is decimated by vertex clustering (same silhouette, a few thousand
                                   triangles); an .fbx keeps its first polygons of every geometry plus the polygons that hold each axis' smallest
                                   and largest vertex, so that the mesh's bounding box is the original's.  cube_rounded2.obj is kept whole.
The full meshes are 57 MB; Dragon_80K.obj alone has 87,130 triangles and Water.fbx 656,796.
"""
from __future__ import annotations

import io
import os
import re
import struct
import sys
import tarfile
import zlib

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)
from ray_tracing_b200 import fbx_mesh  # noqa: E402

OUT = os.path.join(REPO, "tests", "golden", "reference_excerpt.tar.xz")
SCENES = ["Glass Balls", "Glass Dragon", "Sphere Refract", "Splash", "Text"]
KEEP_CLASSES = {1, 4, 20, 33, 114}          # GameObject, Transform, Camera, MeshFilter, MonoBehaviour
OBJ_CELLS = {"Dragon_80K.obj": 24, "Icosphere.obj": 16, "cube_rounded2.obj": None}
FBX_POLYGONS = {"Text.fbx": 60, "Water.fbx": 1500}


def trim_scene(text: str) -> str:
    head = text[:text.index("--- !u!")]
    docs = re.finditer(r"^--- !u!(\d+) &-?\d+(?: stripped)?\n.*?(?=^--- !u!|\Z)", text, flags=re.S | re.M)
    return head + "".join(m.group(0) for m in docs if int(m.group(1)) in KEEP_CLASSES)


def decimate_obj(text: str, cells: int | None) -> str:
    """Vertex clustering on a grid of `cells` cells along the longest side: every vertex moves to the mean of its cell, its normal
    to the normalized sum of the corner normals there; triangles that collapse or repeat are dropped.  Keeps the silhouette."""
    if cells is None:
        return text
    v, vn, faces = [], [], []
    for ln in text.splitlines():
        if ln.startswith("v "):
            v.append([float(x) for x in ln.split()[1:4]])
        elif ln.startswith("vn "):
            vn.append([float(x) for x in ln.split()[1:4]])
        elif ln.startswith("f "):
            faces.append([(int(c.split("/")[0]) - 1, int(c.split("/")[2]) - 1) for c in ln.split()[1:]])
    v, vn = np.array(v), np.array(vn)
    lo = v.min(0)
    cell = (v.max(0) - lo).max() / cells
    _, cluster = np.unique(np.floor((v - lo) / cell).astype(np.int64), axis=0, return_inverse=True)
    cluster = cluster.reshape(-1)
    k = int(cluster.max()) + 1
    pos = np.zeros((k, 3))
    np.add.at(pos, cluster, v)
    pos /= np.bincount(cluster, minlength=k)[:, None]
    nrm = np.zeros((k, 3))
    seen, tris = set(), []
    for f in faces:
        for (a, na), (b, nb), (c, nc) in ((f[0], f[i], f[i + 1]) for i in range(1, len(f) - 1)):
            for vi, ni in ((a, na), (b, nb), (c, nc)):
                nrm[cluster[vi]] += vn[ni]
            t = (int(cluster[a]), int(cluster[b]), int(cluster[c]))
            if len(set(t)) == 3 and tuple(sorted(t)) not in seen:
                seen.add(tuple(sorted(t)))
                tris.append(t)
    nrm /= np.maximum(np.linalg.norm(nrm, axis=1, keepdims=True), 1e-30)
    used = sorted({c for t in tris for c in t})
    new = {c: i + 1 for i, c in enumerate(used)}
    return "\n".join([f"# decimated: vertex clustering on a {cells}-cell grid, {len(tris)} triangles"] +
                     [f"v {pos[c][0]:.6f} {pos[c][1]:.6f} {pos[c][2]:.6f}" for c in used] +
                     [f"vn {nrm[c][0]:.4f} {nrm[c][1]:.4f} {nrm[c][2]:.4f}" for c in used] +
                     ["f " + " ".join(f"{new[c]}//{new[c]}" for c in t) for t in tris]) + "\n"


# ---- binary FBX: read with the package's parser, cut every geometry, write back (32-bit offsets, version 7400) ----------------

def _prop(p) -> bytes:
    if isinstance(p, np.ndarray):
        code = {"<f4": "f", "<f8": "d", "<i8": "l", "<i4": "i", "|u1": "b"}[p.dtype.str]
        raw = zlib.compress(np.ascontiguousarray(p).tobytes())
        return code.encode() + struct.pack("<III", p.size, 1, len(raw)) + raw
    if isinstance(p, bytes):
        return b"R" + struct.pack("<I", len(p)) + p
    if isinstance(p, str):
        b = p.encode("utf-8")
        return b"S" + struct.pack("<I", len(b)) + b
    if isinstance(p, bool):
        return b"C" + struct.pack("<?", p)
    if isinstance(p, int):
        return b"L" + struct.pack("<q", p)
    if isinstance(p, float):
        return b"D" + struct.pack("<d", p)
    raise TypeError(type(p))


def _write_fbx(nodes) -> bytes:
    out = bytearray(b"Kaydara FBX Binary  \x00\x1a\x00" + struct.pack("<I", 7400))

    def emit(node):
        name, props, children = node
        start = len(out)
        pb = b"".join(_prop(p) for p in props)
        out.extend(b"\x00" * 12); out.append(len(name)); out.extend(name.encode()); out.extend(pb)
        for c in children:
            emit(c)
        if children:
            out.extend(b"\x00" * 13)
        struct.pack_into("<III", out, start, len(out), len(props), len(pb))
    for n in nodes:
        emit(n)
    out.extend(b"\x00" * 13 + b"\x00" * 160)
    return bytes(out)


def _cut_geometry(geom, polygons: int):
    verts = np.asarray(fbx_mesh._child(geom, "Vertices")[1][0], dtype=np.float64).reshape(-1, 3)
    pvi = np.asarray(fbx_mesh._child(geom, "PolygonVertexIndex")[1][0], dtype=np.int64)
    corner_vertex = np.where(pvi < 0, ~pvi, pvi)
    stop = np.flatnonzero(pvi < 0)
    start = np.concatenate([[0], stop[:-1] + 1])
    poly_of_corner = np.repeat(np.arange(len(stop)), stop - start + 1)
    keep = set(range(min(polygons, len(stop))))
    used = np.unique(corner_vertex)
    for axis in range(3):                                          # the polygons holding each axis' extreme vertices: same bounds
        for v in (used[np.argmin(verts[used, axis])], used[np.argmax(verts[used, axis])]):
            keep.add(int(poly_of_corner[np.flatnonzero(corner_vertex == v)[0]]))
    keep = sorted(keep)
    corners = np.concatenate([np.arange(start[p], stop[p] + 1) for p in keep])
    normals = fbx_mesh._layer_normals(geom, corner_vertex)
    new_of_old = {int(v): k for k, v in enumerate(dict.fromkeys(corner_vertex[corners].tolist()))}
    new_pvi = np.array([new_of_old[int(v)] for v in corner_vertex[corners]], dtype=np.int32)
    ends = pvi[corners] < 0
    new_pvi[ends] = ~new_pvi[ends]
    new_verts = verts[list(new_of_old)].reshape(-1)
    children = [("Vertices", [new_verts], []), ("PolygonVertexIndex", [new_pvi], [])]
    if normals is not None:
        children.append(("LayerElementNormal", [0], [("MappingInformationType", ["ByPolygonVertex"], []),
                                                     ("ReferenceInformationType", ["Direct"], []),
                                                     ("Normals", [np.ascontiguousarray(normals[corners]).reshape(-1)], [])]))
    return (geom[0], list(geom[1][:3]), children)


def cut_fbx(path: str, polygons: int) -> bytes:
    _, nodes = fbx_mesh.parse_fbx(path)
    objects = next(n for n in nodes if n[0] == "Objects")
    conns = next(n for n in nodes if n[0] == "Connections")
    kept = []
    for o in objects[2]:
        if o[0] == "Geometry" and len(o[1]) >= 3 and o[1][2] == "Mesh":
            kept.append(_cut_geometry(o, polygons))
        elif o[0] == "Model":
            kept.append((o[0], list(o[1][:3]), []))
    return _write_fbx([("Objects", [], kept), conns])


def main(ref: str) -> None:
    files = {}
    for s in SCENES:
        files[f"Assets/Scenes/{s}.unity"] = trim_scene(open(os.path.join(ref, "Assets", "Scenes", s + ".unity"), encoding="utf-8").read()).encode()
    gdir = os.path.join(ref, "Assets", "Graphics")
    for name, cells in OBJ_CELLS.items():
        files[f"Assets/Graphics/{name}"] = decimate_obj(open(os.path.join(gdir, name)).read(), cells).encode()
    for name, polys in FBX_POLYGONS.items():
        files[f"Assets/Graphics/{name}"] = cut_fbx(os.path.join(gdir, name), polys)
    for name in list(OBJ_CELLS) + list(FBX_POLYGONS):
        files[f"Assets/Graphics/{name}.meta"] = open(os.path.join(gdir, name + ".meta"), "rb").read()
    with tarfile.open(OUT, "w:xz", format=tarfile.USTAR_FORMAT) as tar:
        for rel in sorted(files):
            info = tarfile.TarInfo(rel)
            info.size, info.mtime, info.mode = len(files[rel]), 0, 0o644
            tar.addfile(info, io.BytesIO(files[rel]))
    print(f"{OUT}: {os.path.getsize(OUT)} bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
