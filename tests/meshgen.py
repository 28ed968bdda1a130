"""Seeded meshes with high-valence vertices, Jacobian rows longer than 64 entries and split fans.

The shipped meshes have no vertex with more than 8 incident cells, so the branches of the kernels that depend on the valence
(the fan tree's wider steps, the SpMV tail loop past 64 entries, the assembly fallbacks) need meshes of their own.  Every
generator goes through Mesh.from_arrays; boundary lines carry tag 10 (Neumann) on the side x > 0 (wheel, bow-tie) or x = 1
(Delaunay) and tag 0 elsewhere.
"""
import copy

import numpy as np

NEUMANN = 10
# Dirichlet calls and inlet data for these meshes: every tag-0 line carries the inlet profile (non-zero data)
CALLS = [{0: True}]
INLET = dict(u_m=1.5, H=4.0, y0=-2.0)


def _boundary_lines(cells):
    e = np.sort(cells[:, [0, 1, 1, 2, 2, 0]].reshape(-1, 2), axis=1)
    u, cnt = np.unique(e, axis=0, return_counts=True)
    return u[cnt == 1]


def _mesh(pkg, xy, cells, neumann_side):
    lines = _boundary_lines(cells)
    mid = 0.5 * (xy[lines[:, 0]] + xy[lines[:, 1]])
    tag = np.where(neumann_side(mid), NEUMANN, 0).astype(np.int32)
    return pkg.Mesh.from_arrays(xy, cells.astype(np.int32), lines.astype(np.int32), tag)


def wheel(pkg, k, rings=2):
    """A centre vertex of valence k inside `rings` rings of k vertices each (radius j / rings).  Ring j is turned by half a
    step against ring j - 1, so the strip between two rings is the cyclic sequence of its vertices sorted by angle, every
    three consecutive ones a cell: ring vertices have valence 5 (first ring), 6 (inner rings) or 3 (outer ring)."""
    xy = [np.zeros((1, 2))]
    ang = []
    for j in range(1, rings + 1):
        a = 2 * np.pi * (np.arange(k) + 0.5 * ((j - 1) % 2)) / k
        ang.append(a)
        xy.append(j / rings * np.stack([np.cos(a), np.sin(a)], axis=1))
    xy = np.concatenate(xy)
    first = [1 + j * k for j in range(rings)]
    cells = [[0, first[0] + i, first[0] + (i + 1) % k] for i in range(k)]
    for j in range(rings - 1):
        ids = np.concatenate([first[j] + np.arange(k), first[j + 1] + np.arange(k)])
        order = ids[np.argsort(np.concatenate([ang[j], ang[j + 1]]) % (2 * np.pi), kind="stable")]
        cells += [[order[m], order[(m + 1) % (2 * k)], order[(m + 2) % (2 * k)]] for m in range(2 * k)]
    return _mesh(pkg, xy, np.array(cells), lambda mid: mid[:, 0] > 0)


def delaunay(pkg, n, seed=0):
    """scipy's Delaunay triangulation of n seeded uniform points in the unit square plus its four corners; the boundary is
    the hull (the four sides, one edge each: the cells along the sides are slivers)."""
    from scipy.spatial import Delaunay
    rng = np.random.default_rng(seed)
    xy = np.concatenate([np.array([[0.0, 0.0], [1.0, 0.0], [1.0, 1.0], [0.0, 1.0]]), rng.random((n, 2))])
    tri = Delaunay(xy)
    return _mesh(pkg, xy, tri.simplices, lambda mid: mid[:, 0] > 1 - 1e-12)


def bowtie(pkg, m=12):
    """Two half-disc fans of m cells each that meet only at the origin: one vertex (valence 2 m) whose cells form two open
    fans."""
    xy = [np.zeros((1, 2))]
    cells = []
    for s in range(2):
        a = np.pi * s + np.linspace(0.1, np.pi - 0.1, m + 1)
        base = 1 + s * (m + 1)
        xy.append(np.stack([np.cos(a), np.sin(a)], axis=1))
        cells += [[0, base + i, base + i + 1] for i in range(m)]
    return _mesh(pkg, np.concatenate(xy), np.array(cells), lambda mid: mid[:, 0] > 0)


# local orientation reversed (vertices 1 <-> 2): the 15 cell dofs are (u, v, p) of vertices 0, 1, 2, then (u, v) of the edges
# (v0 v1), (v1 v2), (v2 v0); face f of a cell is the edge (v_f, v_f+1)
FLIP_VERTICES = [0, 2, 1]
FLIP_DOFS = [0, 1, 2, 6, 7, 8, 3, 4, 5, 13, 14, 11, 12, 9, 10]
FLIP_FACE = np.array([2, 1, 0], np.int32)


def flipped(part, which):
    """Shallow copy of a Part whose cells `which` (mask or indices) are listed clockwise.  The global operator is the same,
    so the oracle on `part` stays the reference."""
    sel = np.zeros(part.n_cells, bool)
    sel[which] = True
    out = copy.copy(part)
    cv = np.array(part.cell_vertices).reshape(-1, 3)
    cd = np.array(part.cell_dofs).reshape(-1, 15)
    cv[sel] = cv[sel][:, FLIP_VERTICES]
    cd[sel] = cd[sel][:, FLIP_DOFS]
    bf = np.array(part.bface_face)
    on = sel[np.asarray(part.bface_cell)]
    bf[on] = FLIP_FACE[bf[on]]
    out.cell_vertices, out.cell_dofs, out.bface_face = cv.reshape(-1), cd.reshape(-1), bf
    return out


def valence(mesh):
    return np.bincount(np.asarray(mesh.cells).ravel(), minlength=mesh.n_vertices)


def row_lengths(part):
    return np.diff(np.asarray(part.jac_rowptr))
