"""Solver type "cg.mg2": CG with the polOrder-2 multigrid preconditioner on structured Q2 grids
(block Jacobi + conforming Q1 + hourglass family, one V(1,1)-cycle per hierarchy; tests/test_mg_q2_prototype.py states
the argument on the CPU).  Against sparse direct solves of the oracle-assembled systems."""
import numpy as np
import pytest

import dune_hdd_b200 as hdd
from dune_hdd_b200 import grids, problems
from oracle import oracle as o
from tests.helpers import direct_solve, oracle_mesh, rel

pytestmark = pytest.mark.gpu

SOL_TOL = 1e-8


def _q2_system(g, factor=None, tensor=None):
    m = oracle_mesh(g).with_polorder(2)
    rp, col = o.pattern(m)
    A = o.assemble_lhs(m, factor or o.const(1.0), tensor, rp, col)
    return m, rp, col, A, o.assemble_rhs(m, o.esv2007_force())


def _iterations(d, typ, precision=1e-10, max_iter=5000, **kw):
    _, info = d.solve({"type": typ, "precision": precision, "max_iter": max_iter}, return_info=True, **kw)
    assert info["converged"], (typ, info)
    return info["iterations"]


@pytest.mark.parametrize("n,parts", [(8, (1, 1)), (16, (2, 2)), (32, (1, 1)), (48, (4, 4)), (64, (1, 1))])
def test_cg_mg2_matches_direct_solve(gpu, n, parts):
    g = grids.cube(n, partitions=parts)  # the partitioned grids have subdomain-major cell numbering
    d = hdd.SWIPDG(g, problems.ESV2007(), polorder=2)
    d.init()
    types = d.solver_types()
    assert "cg.mg2" in types and types[0] == "cg.diagonal"
    m, rp, col, A, b = _q2_system(g)
    u, info = d.solve({"type": "cg.mg2", "precision": 1e-13, "max_iter": 500}, return_info=True)
    assert info["converged"] and rel(u, direct_solve(rp, col, A, b)) <= SOL_TOL
    it = _iterations(d, "cg.mg2")
    assert it <= 50, it
    if n >= 32:
        ib = _iterations(d, "cg.blockdiagonal", max_iter=50000)
        assert it < ib / 2, (it, ib)


def test_cg_mg2_iterations_flat_in_h(gpu):
    counts = {}
    for n in (16, 64):
        d = hdd.SWIPDG(grids.cube(n), problems.ESV2007(), polorder=2)
        d.init()
        counts[n] = _iterations(d, "cg.mg2")
        assert _iterations(d, "cg.multigrid2") == counts[n]  # the alias
    assert abs(counts[64] - counts[16]) <= 5, counts


def test_cg_mg2_spe10_shape(gpu):
    g = grids.cube(100, 20, (0.0, 0.0), (5.0, 1.0))
    prob = problems.Spe10Model1(g)
    d = hdd.SWIPDG(g, prob, polorder=2)
    d.init()
    m = oracle_mesh(g).with_polorder(2)
    rp, col = o.pattern(m)
    A = o.assemble_lhs(m, o.const(1.0), prob.diffusion_tensor, rp, col)
    assert rel(d.system_matrix().affine_part(), A) <= 1e-12
    b = d.rhs().affine_part()
    u, info = d.solve({"type": "cg.mg2", "precision": 1e-12, "max_iter": 5000}, return_info=True)
    assert info["converged"], info
    assert np.linalg.norm(o.spmv(rp, col, A, u) - b) <= 1e-9 * np.linalg.norm(b), info


def test_cg_mg2_parametric_and_expression_factors(gpu):
    # parametric operator: both hierarchies are rebuilt for every frozen A(mu)
    g = grids.cube(32)
    fac = problems.AffinelyDecomposable(problems.Constant(1.0), [problems.Expression("x[0]*x[0]+0.1", 2)], ["mu"])
    p = problems.Problem(fac, problems.ESV2007().force, parameter_name="mu", parameter_size=1)
    d = hdd.SWIPDG(g, p, polorder=2)
    d.init()
    for mu in (0.1, 10.0):
        um, im = d.solve({"type": "cg.mg2", "precision": 1e-13, "max_iter": 1000}, mu=mu, return_info=True)
        ud = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 200000}, mu=mu)
        assert im["converged"] and rel(um, ud) <= SOL_TOL, (mu, im)
    # an order-2 expression factor: the volume rule is 3 x 3, the hourglass family is not energy-free there and H is
    # redundant, but it must not hurt
    pe = problems.Problem(problems.AffinelyDecomposable(problems.Expression("2+x[0]*x[1]", 2, "diffusion_factor")),
                          problems.ESV2007().force)
    de = hdd.SWIPDG(g, pe, polorder=2)
    de.init()
    m, rp, col, A, b = _q2_system(g, o.fn([(2.0, o.FN_ONE), (1.0, o.FN_XY)], 2))
    u, info = de.solve({"type": "cg.mg2", "precision": 1e-13, "max_iter": 500}, return_info=True)
    assert info["converged"] and rel(u, direct_solve(rp, col, A, b)) <= SOL_TOL
    it = _iterations(de, "cg.mg2")
    assert it <= 50 and it < _iterations(de, "cg.blockdiagonal", max_iter=50000) / 2, it


def test_cg_mg2_nonzero_dirichlet_and_neumann_data(gpu):
    g = grids.cube(16)
    cen = g.centers()
    bt = np.ones((g.n_cells, g.n_loc), np.uint8)
    bt[(cen[:, 0] < 0)[:, None] & (g.cell_neigh < 0)] = 2
    prob = problems.ESV2007()
    prob.neumann = problems.AffinelyDecomposable(problems.Expression("0.5+x[0]*x[1]-2*x[1]", 2, "neumann"))
    prob.dirichlet = problems.AffinelyDecomposable(problems.Expression("1+x[0]*x[1]", 2, "dirichlet"))
    d = hdd.SWIPDG(g, prob, boundary_info=bt, polorder=2)
    d.init()
    m = oracle_mesh(g).with_polorder(2)
    rp, col = o.pattern(m)
    gn = o.fn([(0.5, o.FN_ONE), (1.0, o.FN_XY), (-2.0, o.FN_Y)], 2)
    gd = o.fn([(1.0, o.FN_ONE), (1.0, o.FN_XY)], 2)
    b = o.assemble_rhs(m, o.esv2007_force(), o.const(1.0), gd, neumann=gn, bnd_type=bt)
    A = o.assemble_lhs(m, o.const(1.0), None, rp, col, bnd_dirichlet=(bt == 1))
    u, info = d.solve({"type": "cg.mg2", "precision": 1e-13, "max_iter": 500}, return_info=True)
    assert info["converged"] and rel(u, direct_solve(rp, col, A, b)) <= SOL_TOL
    assert _iterations(d, "cg.mg2") <= 50


def test_cg_mg2_requirements(gpu):
    # polOrder 1: the Q1 multigrid is "cg.mg"
    d1 = hdd.SWIPDG(grids.cube(8), problems.ESV2007())
    d1.init()
    with pytest.raises(hdd.discretizations.requirements_not_met, match="cg.mg"):
        d1.solve({"type": "cg.mg2", "precision": 1e-10, "max_iter": 100})
    # P2 on triangles
    ds = hdd.SWIPDG(grids.simplex(4), problems.ESV2007(), polorder=2)
    ds.init()
    with pytest.raises(hdd.discretizations.requirements_not_met, match="cg.blockdiagonal"):
        ds.solve({"type": "cg.mg2", "precision": 1e-10, "max_iter": 100})
    # Q2 on a cube grid whose vertices are not numbered as a lattice
    g = grids.cube(8)
    perm = np.random.default_rng(3).permutation(g.n_verts).astype(np.int32)
    xy = np.empty_like(g.xy)
    xy[perm] = g.xy
    dp = hdd.SWIPDG(grids.Grid(g.kind, xy, perm[g.cell_verts], g.cell_neigh), problems.ESV2007(), polorder=2)
    dp.init()
    with pytest.raises(hdd.discretizations.requirements_not_met, match="cg.blockdiagonal"):
        dp.solve({"type": "cg.mg2", "precision": 1e-10, "max_iter": 100})
    # the same discretization still solves with block Jacobi
    u, info = dp.solve({"type": "cg.blockdiagonal", "precision": 1e-10, "max_iter": 5000}, return_info=True)
    assert info["converged"]
