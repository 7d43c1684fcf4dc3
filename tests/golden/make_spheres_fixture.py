"""Generates tests/golden/spheres_mesh.npz from the reference's two-spheres example mesh (examples/spheres/mesh/spheres.msh:
14,362 curved cubic tetrahedra, Gmsh 2.2 binary, 3.4 MB).  Usage:  python tests/golden/make_spheres_fixture.py <reference checkout>

The fixture stores the mesh compactly, and tests/test_spheres_golden.py rebuilds the element nodes from it (load_fixture below):
  * the corner vertices, the corner connectivity as stored (orientation kept), the boundary triangles and their attributes;
  * the cubic lattice nodes that are NOT the affine image of the element's corners, once per mesh entity: the two nodes of each
    curved edge (the one nearer the lower vertex id first) and the centre node of each curved face (sorted vertex triple).
Every other lattice node is the affine combination of the corners; it sits within 3e-16 (relative to the mesh extent) of the
position stored in the .msh file."""
import os
import sys
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from palace_b200.host import gmsh  # noqa: E402

ORDER = 3
PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "spheres_mesh.npz")


def lattice_barycentric(order=ORDER):
    """[Nn][4] integer barycentric weights (times order) of the lattice nodes of gmsh.load_tets' element node layout."""
    lat = np.array([(a, b, c) for c in range(order + 1) for b in range(order + 1 - c) for a in range(order + 1 - b - c)])
    return np.concatenate([order - lat.sum(axis=1, keepdims=True), lat], axis=1)


def _entity_slots(elems, order=ORDER):
    """Edge-node and face-node slots of every element with their global keys: (slot, vertex a, vertex b, first) for the
    nodes on edges (a < b; first: the node nearer a) and (slot, a, b, c) for the face-centre nodes (a < b < c)."""
    bary = lattice_barycentric(order)
    edge, face = [], []
    for s, w in enumerate(bary):
        nz = np.nonzero(w)[0]
        if nz.size == 2:
            va, vb = elems[:, nz[0]], elems[:, nz[1]]
            lo = np.minimum(va, vb)
            edge.append((s, lo, np.maximum(va, vb), np.where(va == lo, w[nz[0]], w[nz[1]]) == order - 1))
        elif nz.size == 3:
            v = np.sort(elems[:, nz], axis=1)
            face.append((s, v[:, 0], v[:, 1], v[:, 2]))
    return edge, face


def load_fixture(path=PATH):
    """gmsh.HighOrderTetMesh of the stored mesh."""
    F = np.load(path)
    verts, elems = F["verts"], F["elems"].astype(np.int64)
    nv = verts.shape[0]
    X = np.einsum("nk,ekc->enc", lattice_barycentric() / ORDER, verts[elems])      # affine images [ne][Nn][3]
    edge, face = _entity_slots(elems)
    ekey = F["curved_edges"][:, 0].astype(np.int64) * nv + F["curved_edges"][:, 1]
    for s, a, b, first in edge:
        i = np.searchsorted(ekey, a * nv + b)
        hit = (i < ekey.size) & (ekey[np.minimum(i, ekey.size - 1)] == a * nv + b)
        X[hit, s] = F["curved_edge_nodes"][i[hit], np.where(first[hit], 0, 1)]
    fk = F["curved_faces"].astype(np.int64)
    fkey = (fk[:, 0] * nv + fk[:, 1]) * nv + fk[:, 2]
    for s, a, b, c in face:
        k = (a * nv + b) * nv + c
        i = np.searchsorted(fkey, k)
        hit = (i < fkey.size) & (fkey[np.minimum(i, fkey.size - 1)] == k)
        X[hit, s] = F["curved_face_nodes"][i[hit]]
    return gmsh.HighOrderTetMesh(ORDER, verts, elems, np.ones(elems.shape[0], dtype=np.int32), np.ascontiguousarray(np.transpose(X, (0, 2, 1))),
                                 F["bdr_attr"].astype(np.int32), F["bdr_verts"].astype(np.int64))


def main(ref):
    m = gmsh.load_tets(os.path.join(ref, "examples/spheres/mesh/spheres.msh"))
    assert m.order == ORDER and (m.attr == 1).all() and m.verts.shape[0] < 2 ** 16
    X = np.transpose(m.xe, (0, 2, 1))
    aff = np.einsum("nk,ekc->enc", lattice_barycentric() / ORDER, m.verts[m.elems])
    curved = np.abs(X - aff).max(axis=2) > 1e-9 * np.abs(m.verts).max()
    edge, face = _entity_slots(m.elems)
    ce = {}
    for s, a, b, first in edge:
        for e in np.nonzero(curved[:, s])[0]:
            ce.setdefault((int(a[e]), int(b[e])), [None, None])[0 if first[e] else 1] = X[e, s]
    cf = {}
    for s, a, b, c in face:
        for e in np.nonzero(curved[:, s])[0]:
            cf[(int(a[e]), int(b[e]), int(c[e]))] = X[e, s]
    assert all(x is not None for v in ce.values() for x in v)
    ek, fk = sorted(ce), sorted(cf)
    arrays = dict(verts=m.verts, elems=m.elems.astype(np.uint16), bdr_attr=m.bdr_attr.astype(np.uint8), bdr_verts=m.bdr_verts.astype(np.uint16),
                  curved_edges=np.array(ek, dtype=np.uint16), curved_edge_nodes=np.array([ce[k] for k in ek]),
                  curved_faces=np.array(fk, dtype=np.uint16), curved_face_nodes=np.array([cf[k] for k in fk]))
    # LZMA members (np.load reads any zip compression): a third smaller than np.savez_compressed's deflate
    with zipfile.ZipFile(PATH, "w", compression=zipfile.ZIP_LZMA) as z:
        for k, v in arrays.items():
            with z.open(k + ".npy", "w") as f:
                np.lib.format.write_array(f, np.ascontiguousarray(v))
    r = load_fixture()
    err = np.abs(r.xe - m.xe).max() / np.abs(m.verts).max()
    assert err < 1e-15 and (r.elems == m.elems).all() and (r.bdr_verts == m.bdr_verts).all()
    print("wrote", PATH, os.path.getsize(PATH), "bytes;", m.ne, "tets,", len(ek), "curved edges,", len(fk), "curved faces; "
          f"element nodes within {err:.1e} of the .msh file")


if __name__ == "__main__":
    main(sys.argv[1])
