"""Solver type "cg.mg2.simplex": CG with the polOrder-2 multigrid preconditioner on lattice-structured triangle grids
(block Jacobi with the 6 x 6 cell blocks + the conforming P1 space on the vertex lattice, one V(1,1)-cycle;
tests/test_mg_p2_prototype.py states the argument on the CPU).  Solutions against sparse direct solves of the
oracle-assembled systems, and the preconditioner operator by operator against the float64 restatement in
tests/mg_reference_p2.py, with the bars of tests/test_gpu_preconditioners.py."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import dune_hdd_b200 as hdd
from dune_hdd_b200 import capi, grids, problems
from oracle import oracle as o
from tests.helpers import direct_solve, oracle_mesh, rel
from tests.mg_reference_p2 import MultigridP2
from tests.test_gpu_preconditioners import (FACTOR_XY, OP_TOL, RZ_TOL, SYM_TOL, Z_TOL, _max_rel, _mixed_boundary, _pcg,
                                            check_block_jacobi, check_operators, check_symmetry, check_vertex,
                                            device_shapes, level_operator, precondition, right_hand_sides)

pytestmark = pytest.mark.gpu

TYPE = "cg.mg2.simplex"
SOL_TOL = 1e-8
ESV = problems.ESV2007
REFUSED = hdd.discretizations.requirements_not_met


def _iterations(d, typ=TYPE, precision=1e-10, max_iter=5000, **kw):
    _, info = d.solve({"type": typ, "precision": precision, "max_iter": max_iter}, return_info=True, **kw)
    assert info["converged"], (typ, info)
    return info["iterations"]


def _p2(g, prob=None, bt=None):
    d = hdd.SWIPDG(g, prob or ESV(), boundary_info=bt, polorder=2)
    d.init()
    return d


def _oracle(g, factor=None, bt=None):
    m = oracle_mesh(g).with_polorder(2)
    rp, col = o.pattern(m)
    A = o.assemble_lhs(m, factor or o.const(1.0), None, rp, col, bnd_dirichlet=None if bt is None else (bt == 1))
    return m, rp, col, A


def _solve_against_direct(d, g, factor=None, bt=None, b=None, mu=None):
    m, rp, col, A = _oracle(g, factor, bt)
    b = o.assemble_rhs(m, o.esv2007_force()) if b is None else b
    u, info = d.solve({"type": TYPE, "precision": 1e-13, "max_iter": 500}, mu=mu, return_info=True)
    assert info["converged"], info
    assert rel(u, direct_solve(rp, col, A, b)) <= SOL_TOL, (mu, rel(u, direct_solve(rp, col, A, b)))
    return u


# ---- solutions -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("s", [4, 8, 16, 32])
def test_cg_mg2_simplex_matches_direct_solve(gpu, s):
    g = grids.simplex(s)
    d = _p2(g)
    types = d.solver_types()
    assert types[-1] == TYPE and types[0] == "cg.diagonal"
    _solve_against_direct(d, g)
    it = _iterations(d)
    assert it <= 45, it
    if s == 32:
        assert it < _iterations(d, "cg.blockdiagonal", max_iter=50000) / 2


def test_cg_mg2_simplex_iterations_flat_in_h(gpu):
    counts = {}
    for s in (8, 32):
        d = _p2(grids.simplex(s))
        counts[s] = _iterations(d)
        assert _iterations(d, "cg.multigrid2.simplex") == counts[s]  # the alias
    assert max(counts.values()) <= 45 and abs(counts[32] - counts[8]) <= 5, counts


def test_cg_mg2_simplex_partitioned_and_block_swipdg(gpu):
    # subdomain-major cell numbering
    g = grids.simplex(12, partitions=(2, 3))
    _solve_against_direct(_p2(g), g)
    # BlockSWIPDG on 4 and 16 subdomains is the same system as SWIPDG on the same grid
    opts = {"type": TYPE, "precision": 1e-13, "max_iter": 500}
    for parts in ((2, 2), (4, 4)):
        g = grids.simplex(16, partitions=parts)
        db = hdd.BlockSWIPDG(g, ESV(), polorder=2)
        db.init()
        ub = db.solve(opts)
        us = _solve_against_direct(_p2(g), g)
        assert rel(ub, us) <= SOL_TOL, parts


def test_cg_mg2_simplex_os2014_parametric(gpu):
    g = grids.simplex(16)
    d = _p2(g, problems.OS2014ParametricESV2007())
    b = d.rhs().affine_part()
    for mu in (0.1, 1.0):
        _solve_against_direct(d, g, o.os2014_factor(mu), b=b, mu=mu)
        assert _iterations(d, mu=mu) <= 45, mu


def test_cg_mg2_simplex_expression_factor(gpu):
    g = grids.simplex(16)
    prob = problems.Problem(problems.AffinelyDecomposable(problems.Expression("2+x[0]*x[1]", 2, "diffusion_factor")),
                            ESV().force)
    d = _p2(g, prob)
    _solve_against_direct(d, g, FACTOR_XY)
    assert _iterations(d) <= 45


def test_cg_mg2_simplex_mixed_boundary(gpu):
    g = grids.simplex(8)
    bt = _mixed_boundary(g)
    d = _p2(g, bt=bt)
    _solve_against_direct(d, g, bt=bt)
    assert _iterations(d) <= 45


def test_cg_mg2_simplex_nonzero_dirichlet_and_neumann_data(gpu):
    g = grids.simplex(8)
    bt = _mixed_boundary(g)
    prob = ESV()
    prob.neumann = problems.AffinelyDecomposable(problems.Expression("0.5+x[0]*x[1]-2*x[1]", 2, "neumann"))
    prob.dirichlet = problems.AffinelyDecomposable(problems.Expression("1+x[0]*x[1]", 2, "dirichlet"))
    d = _p2(g, prob, bt)
    m = oracle_mesh(g).with_polorder(2)
    gn = o.fn([(0.5, o.FN_ONE), (1.0, o.FN_XY), (-2.0, o.FN_Y)], 2)
    gd = o.fn([(1.0, o.FN_ONE), (1.0, o.FN_XY)], 2)
    b = o.assemble_rhs(m, o.esv2007_force(), o.const(1.0), gd, neumann=gn, bnd_type=bt)
    _solve_against_direct(d, g, bt=bt, b=b)
    assert _iterations(d) <= 45


def test_cg_mg2_simplex_requirements(gpu):
    # polOrder 1 on the same lattice: "cg.mg"
    d1 = hdd.SWIPDG(grids.simplex(4), ESV())
    d1.init()
    with pytest.raises(REFUSED, match="use 'cg.mg' for polOrder 1"):
        d1.solve({"type": TYPE, "precision": 1e-10, "max_iter": 100})
    # cube grids: "cg.mg" / "cg.mg2"
    for p in (1, 2):
        dc = hdd.SWIPDG(grids.cube(8), ESV(), polorder=p)
        dc.init()
        with pytest.raises(REFUSED, match=r"use 'cg.mg' \(polOrder 1\) or 'cg.mg2' \(polOrder 2\)"):
            dc.solve({"type": TYPE, "precision": 1e-10, "max_iter": 100})
    # a triangle grid whose vertices are not numbered as a lattice: "cg.blockdiagonal", which still solves it
    g = grids.simplex(4)
    perm = np.random.default_rng(3).permutation(g.n_verts).astype(np.int32)
    xy = np.empty_like(g.xy)
    xy[perm] = g.xy
    dp = _p2(grids.Grid(g.kind, xy, perm[g.cell_verts], g.cell_neigh))
    with pytest.raises(REFUSED, match="use 'cg.blockdiagonal'"):
        dp.solve({"type": TYPE, "precision": 1e-10, "max_iter": 100})
    assert dp.solve({"type": "cg.blockdiagonal", "precision": 1e-10, "max_iter": 5000}, return_info=True)[1]["converged"]
    # s = 21: the 42 x 42 lattice halves to 21 x 21 (484 vertices > 400, odd)
    with pytest.raises(REFUSED, match="stuck at 21 x 21"):
        _p2(grids.simplex(21)).solve({"type": TYPE, "precision": 1e-10, "max_iter": 100})
    # a negative diffusion factor: the coarsest operator is negative definite
    neg = problems.Problem(problems.AffinelyDecomposable(problems.Constant(-1.0)), ESV().force)
    with pytest.raises(REFUSED, match="not positive definite"):
        _p2(grids.simplex(4), neg).solve({"type": TYPE, "precision": 1e-10, "max_iter": 100})
    # P2 triangles: the refusals of "cg.mg" and "cg.mg2" name the new type
    dt = _p2(grids.simplex(4))
    for typ in ("cg.mg", "cg.mg2"):
        with pytest.raises(REFUSED, match="or 'cg.mg2.simplex'"):
            dt.solve({"type": typ, "precision": 1e-10, "max_iter": 100})


# ---- the preconditioner, operator by operator ----------------------------------------------------------------------------
def build_case(spec):
    """(discretization, grid, [(mu, A(mu))], assembled rhs, nx) of a named case "s[,parts=AxB][,problem=...]" """
    size, *rest = spec.split(",")
    args = dict(a.split("=") for a in rest)
    s = int(size)
    g = grids.simplex(s, partitions=tuple(map(int, args.get("parts", "1x1").split("x"))))
    bt, factors, prob = None, [(None, o.const(1.0))], ESV()
    pb = args.get("problem", "esv")
    if pb == "mixed":
        bt = _mixed_boundary(g)
    elif pb == "os2014":
        prob = problems.OS2014ParametricESV2007()
        factors = [(mu, o.os2014_factor(mu)) for mu in (0.1, 1.0)]
    elif pb == "expr":
        prob = problems.Problem(problems.AffinelyDecomposable(problems.Expression("2+x[0]*x[1]", 2, "diffusion_factor")),
                                ESV().force)
        factors = [(None, FACTOR_XY)]
    d = _p2(g, prob, bt)
    mats = []
    for mu, f in factors:
        m, rp, col, A = _oracle(g, f, bt)
        mats.append((mu, o.to_scipy(rp, col, A).tocsr()))
    return d, g, mats, o.assemble_rhs(m, o.esv2007_force()), 2 * s


def check_case(d, g, A, b, nx, mu=None, what=""):
    mg = MultigridP2(g.cell_verts, nx, nx, A=A)
    rhs = right_hand_sides(g, 6, b)
    for name, r in rhs.items():
        tag = (what, mu, name)
        zb = precondition(d, "cg.blockdiagonal", r, mu)[0]
        check_block_jacobi(mg.D, zb, r, tag)
        z, rz, v = precondition(d, TYPE, r, mu, (nx + 1) ** 2)
        if name == "normal":
            check_operators(d, mg, tag)
        check_vertex(mg, v.reshape(1, -1), r, tag)
        z_ref = mg(r)
        assert _max_rel(z, z_ref) <= Z_TOL, (tag, _max_rel(z, z_ref))
        assert _max_rel(z - zb, mg.correction(r)) <= Z_TOL, tag
        assert abs(rz - r @ z_ref) <= RZ_TOL * np.linalg.norm(r) * np.linalg.norm(z_ref), (tag, rz, r @ z_ref)
    check_symmetry(lambda x: precondition(d, TYPE, x, mu)[0], rhs["normal"], rhs["rhs"], (what, mu))


def run_case(spec):
    d, g, mats, b, nx = build_case(spec)
    for mu, A in mats:
        check_case(d, g, A, b, nx, mu, spec)
    return d


# one level (9^2 vertices), one level at the 400-vertex cap (19^2), two levels (33^2 -> 17^2), partitioned numbering
# (25^2 -> 13^2), the OS2014 factor at two parameters (the hierarchy rebuilt in place), mixed boundary, an expression factor
CASES = {"4": 1, "9": 1, "16": 2, "12,parts=2x3": 2, "16,problem=os2014": 2, "8,problem=mixed": 1, "8,problem=expr": 1}


@pytest.mark.parametrize("spec", list(CASES))
def test_mg2_simplex_preconditioner_matches_the_reference(gpu, spec):
    d = run_case(spec)
    assert len(device_shapes(d)) == CASES[spec]


def test_mg2_simplex_gauss_jordan_coarsest_inverse(gpu):
    """HDD_MG_COARSE_GJ=1 is read once per process: the Tier A cases in a child process"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, HDD_MG_COARSE_GJ="1")
    p = subprocess.run([sys.executable, "-m", "tests.test_gpu_mg2_simplex", "9", "16"], cwd=root, env=env,
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert p.stdout.count("ok") == 2


def test_mg2_simplex_preconditioner_on_a_large_grid(gpu):
    """simplex(208): 346 112 owned triangles (the grid-stride loop of k_dg_prolong_dot_p2 runs more than once), 417^2
    vertices, six levels down to 14^2; the level-0 operator comes from the device"""
    s, nx = 208, 416
    g = grids.simplex(s)
    d = _p2(g)
    r = np.random.default_rng(11).standard_normal(g.n_cells * 6)
    z, rz, v = precondition(d, TYPE, r, n_vertex=(nx + 1) ** 2)
    mg = MultigridP2(g.cell_verts, nx, nx, level0=[level_operator(d, 0, 0)[2]])
    shapes = device_shapes(d)
    assert shapes == [(L["nx"], L["ny"]) for L in mg.levels[0]] and len(shapes) == 6 and shapes[-1] == (13, 13)
    for l, S_ref in enumerate(mg.stencils(0)[1:], start=1):
        err = (np.abs(level_operator(d, l, 0)[2] - S_ref) / np.abs(S_ref[4])).max()
        assert err <= OP_TOL, (l, err)
    check_vertex(mg, v.reshape(1, -1), r)
    zb = precondition(d, "cg.blockdiagonal", r)[0]
    assert np.abs(z - zb - mg.correction(r)).max() <= Z_TOL * np.abs(z).max()
    assert abs(rz - r @ z) <= RZ_TOL * np.linalg.norm(r) * np.linalg.norm(z)
    s2 = np.random.default_rng(12).standard_normal(r.size)
    zs = precondition(d, TYPE, s2)[0]
    assert r @ z > 0.0 and s2 @ zs > 0.0
    assert abs(s2 @ z - r @ zs) <= SYM_TOL * np.sqrt((r @ z) * (s2 @ zs))


def test_mg2_simplex_cg_iterates_follow_the_reference_pcg(gpu):
    """max_iter 20, 3, 1, 12 on one handle: the first call launches directly, the later ones replay the cached
    two-iteration graph, and the done latch falls in the middle of a batch"""
    d, g, ((_, A),), b, nx = build_case("16")
    mg = MultigridP2(g.cell_verts, nx, nx, A=A)
    for maxit in (20, 3, 1, 12):
        with pytest.raises(hdd.discretizations.linear_solver_failed):
            d.uncached_solve({"type": TYPE, "precision": 1e-30, "max_iter": maxit})
        p = C.POINTER(C.c_double)()
        capi.check(capi.lib().hdd_solution_dev(d._h, C.byref(p)))
        x = np.empty(A.shape[0])
        capi.check(capi.lib().hdd_copy_to_host(d._h, capi.ptr(x), p, C.c_size_t(x.nbytes)))
        x_ref = _pcg(A, b, mg, maxit)
        assert rel(x, x_ref) <= 1e-10, (maxit, rel(x, x_ref))


if __name__ == "__main__":
    # the named operator cases in this process (test_mg2_simplex_gauss_jordan_coarsest_inverse runs it with
    # HDD_MG_COARSE_GJ=1)
    for case in sys.argv[1:]:
        run_case(case)
        print("ok", case)
