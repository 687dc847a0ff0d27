"""Triangle meshes from scalar grids (NeRF.extract_mesh): the marching-tetrahedra kernel of the library
(knerf_isosurface_count / knerf_isosurface_emit, include/knerf.h) and binary PLY files."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from .. import _lib


def _vec3(x, name) -> np.ndarray:
    a = np.broadcast_to(np.asarray(x, dtype=np.float32), (3,)).copy()
    if not np.isfinite(a).all():
        raise ValueError(f"{name} must be finite, got {x!r}")
    return a


def marching_tetrahedra(field: torch.Tensor, iso: float, origin=(0.0, 0.0, 0.0), spacing=(1.0, 1.0, 1.0),
                        normals: bool = True):
    """field [nx,ny,nz] (CUDA float32, x slowest) -> (vertices [V,3], normals [V,3] or None, faces [T,3] int32), all
    CUDA tensors.  A point is inside where field > iso; vertex i sits at origin + spacing * (grid coordinate); faces are
    counter-clockwise seen from outside (towards smaller values), normals point there too.  Deterministic: the same
    field gives the same bytes.  One device -> host read (the vertex and triangle counts)."""
    if field.dim() != 3:
        raise ValueError(f"field must be [nx, ny, nz], got shape {tuple(field.shape)}")
    field = field.contiguous()
    nx, ny, nz = (int(s) for s in field.shape)
    lib = _lib.load()
    ws_bytes = lib.knerf_isosurface_workspace_bytes(nx, ny, nz)
    if ws_bytes < 0:
        raise _lib.KnerfError("knerf_isosurface_workspace_bytes: " + lib.knerf_last_error().decode())
    dev = field.device
    org, sp = _vec3(origin, "origin"), _vec3(spacing, "spacing")
    with torch.cuda.device(dev):
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        counts = torch.empty(2, dtype=torch.int64, device=dev)
        _lib.call("knerf_isosurface_count", _lib.ptr(field), nx, ny, nz, float(iso), _lib.ptr(counts, torch.int64),
                  ws.data_ptr(), ws_bytes, _lib.stream())
        V, T = (int(c) for c in counts.cpu())
        if V >= 2 ** 31:
            raise _lib.KnerfError(f"isosurface of {V} vertices: int32 face indices hold at most 2^31 - 1")
        verts = torch.empty((V, 3), dtype=torch.float32, device=dev)
        norms = torch.empty((V, 3), dtype=torch.float32, device=dev) if normals else None
        faces = torch.empty((T, 3), dtype=torch.int32, device=dev)
        _lib.call("knerf_isosurface_emit", _lib.ptr(field), nx, ny, nz, float(iso),
                  org.ctypes.data_as(C.c_void_p), sp.ctypes.data_as(C.c_void_p), _lib.ptr(verts), _lib.ptr(norms),
                  _lib.ptr(faces, torch.int32), V, T, ws.data_ptr(), ws_bytes, _lib.stream())
    return verts, norms, faces


# ---- PLY (binary little endian) -----------------------------------------------------------------------------------
def write_ply(path, vertices, faces, normals=None, colors=None) -> str:
    """Binary little-endian PLY: per vertex float x y z [float nx ny nz] [uchar red green blue], per face
    `list uchar int vertex_indices`.  colors are floats in [0, 1] (rounded to 0..255) or uint8.  Tensors or arrays."""
    host = lambda a: None if a is None else (a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a))  # noqa
    v, f, n, c = host(vertices), host(faces), host(normals), host(colors)
    V, T = len(v), len(f)
    fields = [("x", "<f4"), ("y", "<f4"), ("z", "<f4")]
    if n is not None:
        fields += [("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4")]
    if c is not None:
        fields += [("red", "u1"), ("green", "u1"), ("blue", "u1")]
    vert = np.empty(V, dtype=fields)
    for k, name in enumerate("xyz"):
        vert[name] = v[:, k]
    if n is not None:
        for k, name in enumerate(("nx", "ny", "nz")):
            vert[name] = n[:, k]
    if c is not None:
        c8 = c if c.dtype == np.uint8 else np.clip(np.rint(c.astype(np.float64) * 255.0), 0, 255).astype(np.uint8)
        for k, name in enumerate(("red", "green", "blue")):
            vert[name] = c8[:, k]
    face = np.empty(T, dtype=[("n", "u1"), ("i", "<i4", (3,))])
    face["n"] = 3
    face["i"] = f
    header = ["ply", "format binary_little_endian 1.0", f"element vertex {V}"]
    header += [f"property float {name}" for name, _ in fields[:3 + (3 if n is not None else 0)]]
    if c is not None:
        header += ["property uchar red", "property uchar green", "property uchar blue"]
    header += [f"element face {T}", "property list uchar int vertex_indices", "end_header"]
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "wb") as fh:
        fh.write(("\n".join(header) + "\n").encode("ascii"))
        fh.write(vert.tobytes())
        fh.write(face.tobytes())
    return path


_PLY_TYPES = {"char": "i1", "uchar": "u1", "short": "<i2", "ushort": "<u2", "int": "<i4", "uint": "<u4",
              "float": "<f4", "double": "<f8", "int8": "i1", "uint8": "u1", "int16": "<i2", "uint16": "<u2",
              "int32": "<i4", "uint32": "<u4", "float32": "<f4", "float64": "<f8"}


def read_ply(path) -> dict:
    """Reads what write_ply writes (binary little endian, triangle faces): dict of numpy arrays `vertices` [V,3],
    `normals` [V,3] or None, `colors` [V,3] uint8 or None, `faces` [T,3] int32."""
    with open(path, "rb") as fh:
        data = fh.read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    lines = data[:end].decode("ascii").splitlines()
    if lines[0] != "ply" or lines[1] != "format binary_little_endian 1.0":
        raise ValueError(f"{path}: not a binary little-endian PLY file")
    elements, cur = [], None
    for ln in lines[2:-1]:
        tok = ln.split()
        if tok[0] == "element":
            cur = [tok[1], int(tok[2]), []]
            elements.append(cur)
        elif tok[0] == "property":
            cur[2].append((tok[-1], tuple(tok[2:4]) if tok[1] == "list" else _PLY_TYPES[tok[1]]))
    off, out = end, {}
    for name, count, props in elements:
        if name == "vertex":
            dt = np.dtype([(p, t) for p, t in props])
            vert = np.frombuffer(data, dtype=dt, count=count, offset=off)
            off += dt.itemsize * count
            names = dt.names
            out["vertices"] = np.stack([vert[k] for k in "xyz"], -1)
            out["normals"] = np.stack([vert[k] for k in ("nx", "ny", "nz")], -1) if "nx" in names else None
            out["colors"] = np.stack([vert[k] for k in ("red", "green", "blue")], -1) if "red" in names else None
        elif name == "face":
            (pname, (ct, it)), = props
            dt = np.dtype([("n", _PLY_TYPES[ct]), ("i", _PLY_TYPES[it], (3,))])
            face = np.frombuffer(data, dtype=dt, count=count, offset=off)
            if count and not (face["n"] == 3).all():
                raise ValueError(f"{path}: only triangle faces are supported")
            off += dt.itemsize * count
            out["faces"] = face["i"].astype(np.int32)
        else:
            raise ValueError(f"{path}: unexpected element {name!r}")
    if off != len(data):
        raise ValueError(f"{path}: {len(data) - off} trailing bytes after the last element")
    return out
