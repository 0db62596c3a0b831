"""Executable record of the design argument behind the solver type "cg.mg" (dune_hdd_b200/csrc/multigrid.cu): a scipy
restatement of the preconditioner on oracle-assembled matrices.

  M^-1 r = D_blk^-1 r + P V(P^T r) [+ P C V_C(C P^T r)]

With the reference's midpoint-rule volume term the conforming auxiliary operator A_c = P^T A P has a second family of
low-energy modes (checkerboard x smooth).  A plain multigrid hierarchy does not see it - the CG iteration count grows
with 1/h - while the additional checkerboard-twisted hierarchy brings it back to the count of an exact coarse solve.
The CUDA path is compared with direct solves in tests/test_gpu_parity.py and operator by operator with the restatement
in tests/mg_reference.py in tests/test_gpu_preconditioners.py; this file pins the algorithm itself on CPU."""
import warnings

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from oracle import oracle as o
from tests.mg_reference import hierarchy, vcycle

warnings.filterwarnings("ignore")


def _iterations(n, variant):
    m = o.mesh_cube(n, n, -1.0, 1.0, -1.0, 1.0)
    rp, col = o.pattern(m)
    A = o.to_scipy(rp, col, o.assemble_lhs(m, o.const(1.0), None, rp, col)).tocsr()
    b = o.assemble_rhs(m, o.esv2007_force())
    N, nv = m.n_dofs, m.nv
    P = sp.csr_matrix((np.ones(N), (np.arange(N), m.cv.reshape(-1))), shape=(N, nv))
    Ac = (P.T @ A @ P).tocsr()
    # P^T A P is a 9-point vertex stencil: everything at index distance 2 cancels (jumps of continuous functions)
    ix, iy = np.arange(nv) % (n + 1), np.arange(nv) // (n + 1)
    coo = Ac.tocoo()
    far = (np.abs(ix[coo.row] - ix[coo.col]) > 1) | (np.abs(iy[coo.row] - iy[coo.col]) > 1)
    assert np.abs(coo.data[far]).max(initial=0.0) <= 1e-12 * np.abs(coo.data).max()
    C = sp.diags((-1.0) ** (ix + iy))
    # the prototype coarsens down to 3 x 3 vertices (the device stops at 400)
    lv, lvC = hierarchy(Ac, n, n, max_coarse=9), hierarchy((C @ Ac @ C).tocsr(), n, n, max_coarse=9)
    lu = spla.splu(Ac.tocsc())
    D = sp.block_diag([sp.csr_matrix(np.linalg.inv(A[4 * c:4 * c + 4, 4 * c:4 * c + 4].toarray())) for c in range(m.nc)], format="csr")

    def prec(r):
        z, rc = D @ r, P.T @ r
        if variant == "exact":
            return z + P @ lu.solve(rc)
        z = z + P @ vcycle(lv, rc)
        if variant == "twisted":
            z = z + P @ (C @ vcycle(lvC, C @ rc))
        return z

    it = [0]
    x, info = spla.cg(A, b, rtol=1e-10, maxiter=2000, M=spla.LinearOperator((N, N), matvec=prec),
                      callback=lambda xk: it.__setitem__(0, it[0] + 1))
    assert info == 0
    assert np.linalg.norm(A @ x - b) <= 1e-8 * np.linalg.norm(b)
    return it[0]


def test_twisted_hierarchy_restores_mesh_independent_convergence():
    counts = {n: {v: _iterations(n, v) for v in ("exact", "plain", "twisted")} for n in (16, 32)}
    for n in (16, 32):
        assert counts[n]["exact"] <= 40 and counts[n]["twisted"] <= 50
    # plain multigrid misses the checkerboard family and degrades with 1/h; the twisted pair does not
    assert counts[32]["plain"] >= counts[16]["plain"] + 15
    assert counts[32]["twisted"] <= counts[16]["twisted"] + 10
    assert counts[32]["twisted"] < counts[32]["plain"]
