"""Executable record of the design argument behind the solver type "cg.mg2.simplex" (dune_hdd_b200/csrc/multigrid.cu):
a scipy restatement of the polOrder-2 preconditioner on lattice-structured triangle grids, on oracle-assembled matrices.

  M^-1 r = D_6^-1 r [+ P V(P^T r)]

D_6 are the 6 x 6 cell blocks, P the interpolation of the conforming P1 space on the vertex lattice into P2-DG
(tests/mg_reference_p2.py).  The P2 volume term is integrated exactly, so unlike Q2 on cubes (tests/test_mg_q2_prototype.py)
there is no hourglass family and no second hierarchy: block Jacobi alone grows with 1/h, one V(1,1)-cycle on the
conforming P1 space keeps the CG iteration count flat, also for the OS2014 factor at mu = 0.1.  ESV2007 on
grids.simplex(s) (the ALU ladder, 8 s^2 triangles on [-1, 1]^2), CG to 1e-10.  The CUDA path is compared with direct
solves and operator by operator with this restatement in tests/test_gpu_mg2_simplex.py."""
import warnings

import numpy as np
import scipy.sparse.linalg as spla

from dune_hdd_b200 import grids
from oracle import oracle as o
from tests.helpers import oracle_mesh
from tests.mg_reference_p2 import MultigridP2

warnings.filterwarnings("ignore")


def _iterations(s, factor, multigrid):
    g = grids.simplex(s)
    m = oracle_mesh(g).with_polorder(2)
    rp, col = o.pattern(m)
    A = o.to_scipy(rp, col, o.assemble_lhs(m, factor, None, rp, col)).tocsr()
    b = o.assemble_rhs(m, o.esv2007_force())
    # the prototype coarsens down to 3 x 3 vertices (the device stops at 400); MultigridP2 asserts through to_stencil
    # that P^T A P is a 9-point stencil
    mg = MultigridP2(g.cell_verts, 2 * s, 2 * s, A=A, max_coarse=9)
    N = A.shape[0]
    prec = mg if multigrid else mg.block_jacobi
    it = [0]
    x, info = spla.cg(A, b, rtol=1e-10, maxiter=5000, M=spla.LinearOperator((N, N), matvec=prec),
                      callback=lambda xk: it.__setitem__(0, it[0] + 1))
    assert info == 0
    assert np.linalg.norm(A @ x - b) <= 1e-8 * np.linalg.norm(b)
    return it[0]


def test_conforming_p1_vcycle_keeps_p2_iterations_flat():
    sizes = (4, 8, 16)
    bj = {s: _iterations(s, o.const(1.0), False) for s in sizes}
    mg = {s: _iterations(s, o.const(1.0), True) for s in sizes}
    # block Jacobi alone grows with 1/h (59, 95, 126 when this was written)
    assert bj[16] >= bj[4] + 50, bj
    # one V(1,1)-cycle on the conforming P1 lattice: flat (35, 35, 34)
    assert max(mg.values()) <= 40 and max(mg.values()) - min(mg.values()) <= 3, mg


def test_conforming_p1_vcycle_with_the_os2014_factor():
    f = o.os2014_factor(0.1)
    bj = {s: _iterations(s, f, False) for s in (4, 16)}
    mg = {s: _iterations(s, f, True) for s in (4, 8, 16)}
    # 136 -> 528 with block Jacobi; 41, 40, 40 with the V-cycle
    assert bj[16] >= 3 * bj[4], bj
    assert max(mg.values()) <= 45, mg
