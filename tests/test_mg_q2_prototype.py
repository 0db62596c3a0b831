"""Executable record of the design argument behind the solver type "cg.mg2" (dune_hdd_b200/csrc/multigrid.cu): a scipy
restatement of the polOrder-2 preconditioner on oracle-assembled Q2 matrices.

  M^-1 r = D_9^-1 r + P V_P(P^T r) [+ H V_H(H^T r)]

D_9 are the 9 x 9 cell blocks, P the bilinear interpolation of the conforming Q1 vertex space into Q2-DG (node a + 3 b of
a cell gets w(i, a) w(j, b) of its vertex i + 2 j, w(0, a) = 1 - a / 2, w(1, a) = a / 2), H the hourglass family: cell c
gets s[v0(c)] g with v0(c) the cell's lower-left vertex and g = (2/3, -1/3, 2/3) x (2/3, -1/3, 2/3).  The Q2 volume term of
a constant factor is integrated with the 2 x 2 Gauss rule, under which the cell function (x^2 - 1/3)(y^2 - 1/3) has a zero
gradient at every quadrature point; it is continuous across faces, so a field of that shape with a smoothly varying
amplitude has almost no energy, and neither the conforming Q1 space nor the cell blocks represent it.  Without H the CG
iteration count grows with 1/h; with H it stays flat.  V_P and V_H are one geometric V(1,1)-cycle each (the helpers of
tests/test_mg_prototype.py).  The CUDA path is compared with direct solves in tests/test_gpu_mg2.py."""
import warnings

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle import oracle as o
from tests.test_mg_prototype import _hierarchy, _vcycle

warnings.filterwarnings("ignore")

G1 = np.array([2.0 / 3.0, -1.0 / 3.0, 2.0 / 3.0])
HOURGLASS = np.outer(G1, G1).ravel()  # node a + 3 b


def _w(i, a):
    return 1.0 - a / 2.0 if i == 0 else a / 2.0


def _operators(m):
    """P (conforming Q1 -> Q2-DG) and H (hourglass family indexed by the lower-left vertex) as sparse matrices"""
    N, nv, nc = m.n_dofs, m.nv, m.nc
    cv = m.cv.reshape(-1, 4)
    rows, cols, vals = [], [], []
    for c in range(nc):
        for b in range(3):
            for a in range(3):
                for j in range(2):
                    for i in range(2):
                        w = _w(i, a) * _w(j, b)
                        if w:
                            rows.append(9 * c + a + 3 * b); cols.append(cv[c, i + 2 * j]); vals.append(w)
    P = sp.csr_matrix((vals, (rows, cols)), shape=(N, nv))
    H = sp.csr_matrix((np.tile(HOURGLASS, nc), (np.arange(N), np.repeat(cv[:, 0], 9))), shape=(N, nv))
    return P, H


def _hourglass_operator(A, H):
    """H^T A H; the rows of the top vertex row and the right vertex column are empty (no cell has its lower-left vertex
    there) and get the mean diagonal"""
    Ah = (H.T @ A @ H).tolil()
    d = Ah.diagonal()
    mean = d[d > 0].mean()
    for v in np.flatnonzero(d == 0):
        Ah[v, v] = mean
    return Ah.tocsr()


def _iterations(n, variant, tensor=None):
    m = o.mesh_cube(n, n, -1.0, 1.0, -1.0, 1.0).with_polorder(2)
    rp, col = o.pattern(m)
    A = o.to_scipy(rp, col, o.assemble_lhs(m, o.const(1.0), tensor, rp, col)).tocsr()
    b = o.assemble_rhs(m, o.esv2007_force())
    N, nv = m.n_dofs, m.nv
    P, H = _operators(m)
    Ap, Ah = (P.T @ A @ P).tocsr(), _hourglass_operator(A, H)
    # both auxiliary operators are 9-point vertex stencils: nothing at index distance 2 (A_P: jumps of continuous
    # functions cancel; A_H: only cells sharing a face couple, and their lower-left vertices are lattice neighbours)
    ix, iy = np.arange(nv) % (n + 1), np.arange(nv) // (n + 1)
    for S in (Ap, Ah):
        coo = S.tocoo()
        far = (np.abs(ix[coo.row] - ix[coo.col]) > 1) | (np.abs(iy[coo.row] - iy[coo.col]) > 1)
        assert np.abs(coo.data[far]).max(initial=0.0) <= 1e-12 * np.abs(coo.data).max()
    lvp, lvh = _hierarchy(Ap, n), _hierarchy(Ah, n)
    D = sp.block_diag([sp.csr_matrix(np.linalg.inv(A[9 * c:9 * c + 9, 9 * c:9 * c + 9].toarray())) for c in range(m.nc)],
                      format="csr")

    def prec(r):
        z = D @ r + P @ _vcycle(lvp, 0, P.T @ r)
        if variant == "hourglass":
            z = z + H @ _vcycle(lvh, 0, H.T @ r)
        return z

    it = [0]
    x, info = spla.cg(A, b, rtol=1e-10, maxiter=2000, M=spla.LinearOperator((N, N), matvec=prec),
                      callback=lambda xk: it.__setitem__(0, it[0] + 1))
    assert info == 0
    assert np.linalg.norm(A @ x - b) <= 1e-8 * np.linalg.norm(b)
    return it[0]


def test_hourglass_family_restores_mesh_independent_convergence():
    counts = {n: {v: _iterations(n, v) for v in ("plain", "hourglass")} for n in (8, 16, 32)}
    # the conforming Q1 space alone misses the hourglass family: the count grows with 1/h
    assert counts[16]["plain"] >= counts[8]["plain"] + 10
    assert counts[32]["plain"] >= counts[16]["plain"] + 20
    # with it the count is flat
    hg = [counts[n]["hourglass"] for n in (8, 16, 32)]
    assert max(hg) <= 45 and max(hg) - min(hg) <= 5, counts
    assert counts[32]["hourglass"] < counts[32]["plain"] / 2


def test_hourglass_family_with_a_heterogeneous_cellwise_tensor():
    """a random 100:1 cell-wise diffusion tensor (the SPE10 kind of data; a cell-wise *factor* is no test case here: the
    reference's SWIPDG matrix is indefinite for such a factor, already on Q1): H still removes the growth with 1/h"""
    counts = {}
    for n in (16, 32):
        k = 10.0 ** np.random.default_rng(1).uniform(0.0, 2.0, n * n)
        tensor = np.zeros((n * n, 4))
        tensor[:, 0] = tensor[:, 3] = k
        counts[n] = {v: _iterations(n, v, tensor) for v in ("plain", "hourglass")}
    assert counts[32]["plain"] >= 2 * counts[16]["plain"] - 10, counts
    assert counts[32]["hourglass"] <= 80 and counts[32]["hourglass"] <= counts[16]["hourglass"] + 15, counts
    assert counts[32]["hourglass"] < counts[32]["plain"] / 3, counts
