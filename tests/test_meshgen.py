"""The generated meshes of tests/meshgen.py (CPU only): each one has the property the GPU tests rely on, and the host layout of
the one-CTA triangular solves holds on their velocity blocks."""
import numpy as np
import pytest
import scipy.sparse as sp

import meshgen as mg
from test_tri_layout import MEDIUM, PRODUCTION, helper, run  # noqa: F401  (helper: fixture)


def part_of(pkg, m):
    return pkg.Part(pkg.Dofs(m), 0)


def velocity_block_of(part):
    """Pattern of the velocity block of a one-rank Part's Jacobian with diagonally dominant random values (the construction of
    test_tri_layout.velocity_block)."""
    n = part.n_own_u
    rp, cl = np.asarray(part.jac_rowptr), np.asarray(part.jac_col)
    A = sp.csr_matrix((np.ones(rp[n]), cl[: rp[n]], rp[: n + 1]), shape=(n, part.n_own))[:, :n].tocsr()
    A.sort_indices()
    rng = np.random.default_rng(5)
    A.data = rng.uniform(-1.0, 1.0, A.nnz)
    A.setdiag(8.0 + rng.random(n) + np.asarray(abs(A).sum(axis=1)).ravel())
    A.sort_indices()
    return A.tocsr()


@pytest.mark.parametrize("k", [9, 16, 31, 32, 33, 34, 35, 65])
def test_wheel_valence(pkg, k):
    """Centre of valence k; first ring 5, inner rings 6, outer ring 3; the centre's rows (7 k + 3 entries) pass 64 entries."""
    rings = 6
    m = mg.wheel(pkg, k, rings)
    v = mg.valence(m)
    assert m.n_vertices == 1 + rings * k and m.n_cells == k * (2 * rings - 1)
    assert v[0] == k
    assert (v[1:k + 1] == 5).all() and (v[k + 1:(rings - 1) * k + 1] == 6).all() and (v[(rings - 1) * k + 1:] == 3).all()
    L = mg.row_lengths(part_of(pkg, m))
    assert L.max() == 7 * k + 3 and (L > 64).sum() >= 3
    c, f, t = m.boundary_faces()
    assert len(t) == k and set(t) == {0, mg.NEUMANN}


@pytest.mark.parametrize("n,big", [(3000, False), (8000, True)])
def test_delaunay_sizes_and_rows(pkg, n, big):
    m = mg.delaunay(pkg, n)
    d = pkg.Dofs(m)
    L = mg.row_lengths(pkg.Part(d, 0))
    assert m.n_vertices == n + 4 and m.n_boundary_edges == 4 and m.n_inverted == 0
    assert mg.valence(m).max() >= 12 and (L > 64).sum() > 300 and L.max() > 90
    assert (d.n > 65536) == big
    # seeded: the same mesh every time
    assert np.array_equal(mg.delaunay(pkg, n).cells, m.cells)


def test_bowtie_has_two_open_fans(pkg):
    """The centre's 24 cells split into two fans, each open (a first and a last cell), that share no edge."""
    m = mg.bowtie(pkg)
    cells = np.asarray(m.cells)
    v = mg.valence(m)
    assert v[0] == 24 and v[1:].max() <= 2
    inc = cells[(cells == 0).any(axis=1)]
    # the two other vertices of each incident cell: cells are adjacent in a fan when they share one of them
    others = [set(c) - {0} for c in inc.tolist()]
    parent = list(range(len(others)))

    def find(i):
        while parent[i] != i:
            i = parent[i]
        return i
    for i in range(len(others)):
        for j in range(i):
            if others[i] & others[j]:
                parent[find(i)] = find(j)
    fans = {}
    for i in range(len(others)):
        fans.setdefault(find(i), []).append(i)
    assert sorted(len(f) for f in fans.values()) == [12, 12]
    for f in fans.values():   # open fan: two of its outer vertices are in one cell only
        cnt = np.bincount(np.concatenate([list(others[i]) for i in f]))
        assert (cnt == 1).sum() == 2
    assert part_of(pkg, m).n_own == pkg.Dofs(m).n


def test_flipped_copy(pkg):
    """Reversing a cell's orientation keeps its vertex set, its dof set, the dofs of each vertex and edge and the vertices
    of each boundary face."""
    part = part_of(pkg, mg.delaunay(pkg, 200))
    sel = np.random.default_rng(1).random(part.n_cells) < 0.5
    fl = mg.flipped(part, sel)
    cv0, cv1 = np.asarray(part.cell_vertices).reshape(-1, 3), fl.cell_vertices.reshape(-1, 3)
    cd0, cd1 = np.asarray(part.cell_dofs).reshape(-1, 15), fl.cell_dofs.reshape(-1, 15)
    assert np.array_equal(cv1[~sel], cv0[~sel]) and np.array_equal(cv1[sel], cv0[sel][:, [0, 2, 1]])
    xy = np.asarray(part.xy).reshape(-1, 2)

    def area(cv):
        a, b, c = xy[cv[:, 0]], xy[cv[:, 1]], xy[cv[:, 2]]
        return (b[:, 0] - a[:, 0]) * (c[:, 1] - a[:, 1]) - (c[:, 0] - a[:, 0]) * (b[:, 1] - a[:, 1])
    assert (area(cv0) > 0).all() and ((area(cv1) < 0) == sel).all()
    # vertex k's (u, v, p) and edge (v_k, v_k+1)'s (u, v) follow the vertices
    for c in np.flatnonzero(sel)[:50]:
        vmap0 = {cv0[c, k]: tuple(cd0[c, 3 * k:3 * k + 3]) for k in range(3)}
        vmap1 = {cv1[c, k]: tuple(cd1[c, 3 * k:3 * k + 3]) for k in range(3)}
        emap0 = {frozenset((cv0[c, k], cv0[c, (k + 1) % 3])): tuple(cd0[c, 9 + 2 * k:11 + 2 * k]) for k in range(3)}
        emap1 = {frozenset((cv1[c, k], cv1[c, (k + 1) % 3])): tuple(cd1[c, 9 + 2 * k:11 + 2 * k]) for k in range(3)}
        assert vmap0 == vmap1 and emap0 == emap1
    bc, bf0, bf1 = np.asarray(part.bface_cell), np.asarray(part.bface_face), fl.bface_face
    for c, f0, f1 in zip(bc, bf0, bf1):
        assert {cv0[c, f0], cv0[c, (f0 + 1) % 3]} == {cv1[c, f1], cv1[c, (f1 + 1) % 3]}


@pytest.mark.parametrize("name", ["wheel32", "delaunay3000"])
@pytest.mark.parametrize("limits", ["production", "medium"])
def test_layout_walk_long_rows(pkg, helper, name, limits):  # noqa: F811
    """Velocity rows of up to 227 entries (wheel) and hundreds of rows past 64 entries (Delaunay) through the one-CTA layout."""
    m = mg.wheel(pkg, 32, 6) if name == "wheel32" else mg.delaunay(pkg, 3000)
    A = velocity_block_of(part_of(pkg, m))
    assert np.diff(A.indptr).max() > 64
    run(helper, A, PRODUCTION if limits == "production" else MEDIUM)


def test_layout_walk_refuses_delaunay_20000(pkg, helper):  # noqa: F811
    """A level wider than window / 4 rows: the layout refuses (the kernel's precondition), build_block then picks another solve."""
    A = velocity_block_of(part_of(pkg, mg.delaunay(pkg, 20000)))
    y, stats = np.zeros(A.shape[0]), np.zeros(8, np.int64)
    L = PRODUCTION
    rc = helper.tri_layout_check(A.shape[0], A.indptr.astype(np.int64), A.indices.astype(np.int32), np.ascontiguousarray(A.data), y.copy(), y,
                                 L["window"], L["ring_slots"], L["ring_rows"], L["depth"], L["flush"], stats)
    assert rc == -3
