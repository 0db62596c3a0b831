"""The preconditioner of the solver type "cg.mg2.simplex" (dune_hdd_b200/csrc/multigrid.cu, DESIGN.md 6) restated in
float64 scipy on top of tests/mg_reference.py, for the CPU prototype (tests/test_mg_p2_prototype.py) and the
operator-by-operator GPU comparison (tests/test_gpu_mg2_simplex.py).

  P2 on lattice simplices      M^-1 r = D_6^-1 r + P V(P^T r)

D_6: the 6 x 6 cell blocks of A.  P: the interpolation of the conforming P1 space on the (nx+1) x (ny+1) vertex lattice
into P2-DG.  The P2 nodes of a triangle (v0, v1, v2) are in the DoF order of oracle.reference_nodes(SIMPLEX, 2):
(0,0), (1/2,0), (1,0), (0,1/2), (1/2,1/2), (0,1), so node 0 = v0, node 2 = v1, node 5 = v2 and the edge midpoints
1 = (v0+v1)/2, 3 = (v0+v2)/2, 4 = (v1+v2)/2.  One hierarchy: the P2 volume rule is exact, there is no hourglass family.
V: one V(1,1)-cycle of tests/mg_reference.py on the level-0 operator P^T A P, a 9-point vertex stencil."""
import numpy as np
import scipy.sparse as sp

from tests.mg_reference import MAX_COARSE, Multigrid, block_inverses, from_stencil, hierarchy, to_stencil

# NODE_WEIGHTS[n][j]: weight of vertex j of the cell at P2 node n
NODE_WEIGHTS = np.array([[1.0, 0.0, 0.0], [0.5, 0.5, 0.0], [0.0, 1.0, 0.0],
                         [0.5, 0.0, 0.5], [0.0, 0.5, 0.5], [0.0, 0.0, 1.0]])


def transfer(cell_verts, n_verts):
    """P: DG DoFs (6 per cell, cell-major) x lattice vertices"""
    cv = np.asarray(cell_verts)
    nc = cv.shape[0]
    n, j = np.nonzero(NODE_WEIGHTS)
    rows = (6 * np.arange(nc)[:, None] + n[None, :]).ravel()
    cols = cv[:, j].ravel()
    vals = np.tile(NODE_WEIGHTS[n, j], nc)
    return sp.csr_matrix((vals, (rows, cols)), shape=(6 * nc, n_verts))


class MultigridP2(Multigrid):
    """Multigrid of tests/mg_reference.py for P2 on a lattice-structured triangle grid: n_loc = 6, one hierarchy.  A: the
    frozen system matrix, or level0: the level-0 stencil S (9, nv) as given (then A may be None)."""

    def __init__(self, cell_verts, nx, ny, A=None, level0=None, max_coarse=MAX_COARSE):
        self.kind, self.nx, self.ny, self.nl = "p2", nx, ny, 6
        self.Pi = [transfer(cell_verts, (nx + 1) * (ny + 1))]
        if level0 is None:
            A = sp.csr_matrix(A)
            level0 = [to_stencil(self.Pi[0].T @ A @ self.Pi[0], nx, ny)]
        self.level0 = level0
        self.levels = [hierarchy(from_stencil(level0[0], nx, ny), nx, ny, max_coarse)]
        if A is not None:
            self.D, self.Dinv = block_inverses(A, self.nl)
