"""PLY reader of auto_pose/meshrenderer/gl_utils/inout.py:8-160 (``load_ply``), vectorised with numpy.

Reads ``ascii`` and ``binary_little_endian`` files with triangular faces.  Returns the same dictionary as the reference:
'pts' [n, 3], 'normals' [n, 3], optional 'colors' [n, 3] and 'texture_uv' [n, 2] (float64), 'faces' [m, 3] (int64).
Unlike the reference, which prints and exits (or fails later with a KeyError), malformed input raises ValueError:
non-triangular faces, a model without normals, a truncated file, an unknown format or property type."""
import numpy as np

_TYPES = {"char": "i1", "int8": "i1", "uchar": "u1", "uint8": "u1", "short": "i2", "int16": "i2", "ushort": "u2", "uint16": "u2",
          "int": "i4", "int32": "i4", "uint": "u4", "uint32": "u4", "float": "f4", "float32": "f4", "double": "f8", "float64": "f8"}


def _type(name, path):
    if name not in _TYPES:
        raise ValueError("%s: unsupported PLY property type %r" % (path, name))
    return _TYPES[name]


def _header(data, path):
    end = data.find(b"end_header")
    if not data.startswith(b"ply") or end < 0:
        raise ValueError("%s: not a PLY file (no 'ply' magic or no end_header)" % path)
    nl = data.find(b"\n", end)
    body = len(data) if nl < 0 else nl + 1
    fmt = None
    elements = []          # [name, count, [(prop name, dtype, list count dtype or None)]]
    for raw in data[:end].decode("ascii", "replace").splitlines():
        tok = raw.split()
        if not tok:
            continue
        if tok[0] == "format":
            fmt = tok[1]
        elif tok[0] == "element":
            elements.append([tok[1], int(tok[2]), []])
        elif tok[0] == "property" and elements:
            if tok[1] == "list":
                elements[-1][2].append((tok[4], _type(tok[3], path), _type(tok[2], path)))
            else:
                elements[-1][2].append((tok[2], _type(tok[1], path), None))
    if fmt not in ("ascii", "binary_little_endian"):
        raise ValueError("%s: unsupported PLY format %r" % (path, fmt))
    return fmt, elements, body


def _face_layout(props, path):
    """index of the vertex_indices list among the face properties; every other property must be a scalar"""
    lists = [i for i, p in enumerate(props) if p[2] is not None]
    names = [props[i][0] for i in lists]
    if names.count("vertex_indices") + names.count("vertex_index") != 1 or len(lists) != 1:
        raise ValueError("%s: a face needs exactly one list property, vertex_indices" % path)
    return lists[0]


def load_ply(path):
    with open(path, "rb") as f:
        data = f.read()
    fmt, elements, pos = _header(data, path)
    vert = face = None
    if fmt == "ascii":
        lines = data[pos:].splitlines()
        li = 0
        for name, count, props in elements:
            rows = lines[li:li + count]
            li += count
            if len(rows) < count:
                raise ValueError("%s: truncated (element %s has %d of %d lines)" % (path, name, len(rows), count))
            if name == "vertex":
                vals = np.array(b" ".join(rows).split(), dtype=np.float64)
                if vals.size != count * len(props):
                    raise ValueError("%s: vertex lines do not have %d values each" % (path, len(props)))
                vert = {p[0]: vals.reshape(count, len(props))[:, i] for i, p in enumerate(props)}
            elif name == "face":
                k = _face_layout(props, path)
                toks = [r.split() for r in rows]
                if any(len(t) != len(props) + 3 for t in toks) or any(int(t[k]) != 3 for t in toks):
                    raise ValueError("%s: only triangular faces are supported" % path)
                face = np.array([t[k + 1:k + 4] for t in toks], dtype=np.int64).reshape(count, 3)
    else:
        for name, count, props in elements:
            if name == "face":
                k = _face_layout(props, path)
                fields = []
                for i, (pname, dt, ct) in enumerate(props):
                    if i == k:
                        fields += [("n", "<" + ct), ("idx", "<" + dt, (3,))]
                    else:
                        fields.append(("p%d" % i, "<" + dt))
                dtype = np.dtype(fields)
            elif any(p[2] is not None for p in props):
                raise ValueError("%s: list property in binary element %s is not supported" % (path, name))
            else:
                dtype = np.dtype([(p[0], "<" + p[1]) for p in props])
            if pos + count * dtype.itemsize > len(data):
                raise ValueError("%s: truncated (element %s needs %d bytes, %d left)" % (path, name, count * dtype.itemsize, len(data) - pos))
            rec = np.frombuffer(data, dtype=dtype, count=count, offset=pos)
            if name == "face" and count and np.any(rec["n"] != 3):
                raise ValueError("%s: only triangular faces are supported" % path)   # the first non-triangle is read at its true offset
            pos += count * dtype.itemsize
            if name == "vertex":
                vert = {p[0]: rec[p[0]].astype(np.float64) for p in props}
            elif name == "face":
                face = rec["idx"].astype(np.int64)
    if vert is None:
        raise ValueError("%s: no vertex element" % path)
    for key in ("x", "y", "z"):
        if key not in vert:
            raise ValueError("%s: vertex property %s is missing" % (path, key))
    if not {"nx", "ny", "nz"}.issubset(vert):
        raise ValueError("%s: the model has no vertex normals (nx, ny, nz)" % path)
    model = {"pts": np.stack([vert["x"], vert["y"], vert["z"]], 1),
             "normals": np.stack([vert["nx"], vert["ny"], vert["nz"]], 1)}
    if {"red", "green", "blue"}.issubset(vert):
        model["colors"] = np.stack([vert["red"], vert["green"], vert["blue"]], 1)
    if {"texture_u", "texture_v"}.issubset(vert):
        model["texture_uv"] = np.stack([vert["texture_u"], vert["texture_v"]], 1)
    if face is not None and len(face):
        if face.min() < 0 or face.max() >= len(model["pts"]):
            raise ValueError("%s: a face refers to a vertex that does not exist" % path)
        model["faces"] = face
    return model


def mesh_attributes(model, vertex_scale=1.0):
    """Vertex attributes and indices as the reference uploads them (meshrenderer_phong.py:41-55 after geometry.py:17-41):
    float32 [n, 9] = hstack(pts * vertex_scale, normals, colours / 255) with colour 160 where the file has none; int32 [m, 3]."""
    pts = model["pts"].astype(np.float32)
    normals = model["normals"].astype(np.float32)
    if "colors" in model:
        colors = model["colors"].astype(np.uint32) / 255.0
    else:
        colors = np.ones_like(pts) * 160.0 / 255.0
    if "faces" not in model:
        raise ValueError("the model has no faces")
    verts = np.hstack((pts * vertex_scale, normals, colors)).astype(np.float32)
    return np.ascontiguousarray(verts), np.ascontiguousarray(model["faces"].astype(np.int32))
