"""GPU parity: the CUDA path (through the C-ABI) against the CPU oracle on identical grids and inputs.

Bars (BASELINE.json north_star): pattern and DoF map bit-exact, assembled entries 1e-12 relative, solution /
norms / indicators 1e-8 relative, goldens to their 3 printed digits."""
import os

import numpy as np
import pytest

import dune_hdd_b200 as hdd
from dune_hdd_b200 import grids, problems
from oracle import oracle as o
from tests.helpers import direct_solve, golden, oracle_mesh, oracle_system, rel

pytestmark = pytest.mark.gpu

ENTRY_TOL = 1e-12
SOL_TOL = 1e-8


def _grid(kind, n, partitions=(1, 1)):
    return grids.simplex(n, partitions=partitions) if kind == "alu" else grids.cube(n, partitions=partitions)


@pytest.mark.parametrize("kind,n", [("alu", 4), ("alu", 8), ("sgrid", 8), ("sgrid", 16), ("sgrid", 1), ("alu", 1)])
def test_esv2007_pattern_and_entries(gpu, kind, n):
    g = _grid(kind, n)
    d = hdd.SWIPDG(g, problems.ESV2007())
    d.init()
    d.init()  # idempotent
    m, rp, col, A, b = oracle_system(g, o.const(1.0), o.esv2007_force())
    rp_g, col_g = d.pattern()
    assert np.array_equal(rp_g, rp) and np.array_equal(col_g, col)  # bit-exact pattern + DoF map
    M = d.system_matrix()
    assert M.num_components() == 0 and M.has_affine_part()
    assert rel(M.affine_part(), A) <= ENTRY_TOL
    R = d.rhs()
    assert R.num_components() == 0 and R.has_affine_part()
    assert rel(R.affine_part(), b) <= ENTRY_TOL


@pytest.mark.parametrize("kind,n", [("alu", 4), ("alu", 16), ("sgrid", 8), ("sgrid", 32)])
def test_esv2007_solve_matches_direct_solve(gpu, kind, n):
    g = _grid(kind, n)
    d = hdd.SWIPDG(g, problems.ESV2007())
    d.init()
    m, rp, col, A, b = oracle_system(g, o.const(1.0), o.esv2007_force())
    u_ref = direct_solve(rp, col, A, b)
    for typ in ("cg.diagonal", "cg.identity", "cg.blockdiagonal"):
        u, info = d.solve({"type": typ, "precision": 1e-13, "max_iter": 20000}, return_info=True)
        assert info["converged"]
        assert rel(u, u_ref) <= SOL_TOL
    # operator application
    x = np.random.default_rng(0).standard_normal(g.n_dofs)
    assert rel(d.apply(x), o.spmv(rp, col, A, x)) <= 1e-13


def test_cg_iterates_follow_the_oracle_cg(gpu):
    g = grids.cube(16)
    d = hdd.SWIPDG(g, problems.ESV2007())
    d.init()
    m, rp, col, A, b = oracle_system(g, o.const(1.0), o.esv2007_force())
    for maxit in (1, 2, 5, 20):
        x_ref, it, rr = o.cg(rp, col, A, b, precond=1, rtol=1e-30, maxit=maxit)
        with pytest.raises(hdd.discretizations.linear_solver_failed):
            d.uncached_solve({"type": "cg.diagonal", "precision": 1e-30, "max_iter": maxit})
        x = np.empty(g.n_dofs)
        import ctypes as C
        p = C.POINTER(C.c_double)()
        hdd.capi.check(hdd.capi.lib().hdd_solution_dev(d._h, C.byref(p)))
        hdd.capi.check(hdd.capi.lib().hdd_copy_to_host(d._h, hdd.capi.ptr(x), p, C.c_size_t(x.nbytes)))
        assert rel(x, x_ref) <= 1e-11


_ALU_STEM = "linearelliptic-swipdg-expectations_esv2007_2daluconform"
GOLDEN_ALU = {k: golden(_ALU_STEM, k) for k in ("L2", "H1_semi", "energy", "eta_NC_ESV2007", "eta_R_ESV2007",
                                                  "eta_DF_ESV2007", "eta_ESV2007", "eta_ESV2007_alt")}


def _digits3(x, gold):
    return abs(x - gold) <= 0.006 * abs(gold)


@pytest.mark.parametrize("level", [0, 1, 2])
def test_esv2007_estimators_and_goldens(gpu, level):
    g = grids.simplex(4 * 2 ** level)
    d = hdd.SWIPDG(g, problems.ESV2007())
    d.init()
    u = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 50000})
    m = oracle_mesh(g)
    ind_ref = o.indicators(m, u, o.esv2007_force(), o.const(1.0))
    ind = d.indicators(u)
    for k in ("nc2", "res2", "r2", "df2", "dfstar2", "rstar2", "resstar2"):
        assert np.abs(ind[k] - ind_ref[k]).max() <= SOL_TOL * np.abs(ind_ref[k]).max(), k
    assert rel(ind["amin"], ind_ref["amin"]) <= 1e-14
    est = hdd.estimators.SWIPDG
    assert est.available(d) == hdd.estimators.ESV2007_TYPES
    for typ in est.available(d):
        eta = est.estimate(d, u, typ)
        if typ in GOLDEN_ALU:
            assert _digits3(eta, GOLDEN_ALU[typ][level]), (typ, eta)
    eta_ref = np.sqrt((ind_ref["nc2"] + (np.sqrt(ind_ref["r2"]) + np.sqrt(ind_ref["df2"])) ** 2).sum())
    assert abs(est.estimate(d, u, "eta_ESV2007") - eta_ref) <= SOL_TOL * eta_ref
    loc = est.estimate_local(d, u, "eta_ESV2007")
    assert loc.shape == (g.n_cells,) and abs(loc.sum() - 1.0) < 1e-12
    loc = est.estimate_local(d, u, "eta_ESV2007_alt")
    assert loc.shape == (g.n_cells,)
    err = o.error_norms(m, u, o.esv2007_exact())
    assert _digits3(err["L2"], GOLDEN_ALU["L2"][level]) and _digits3(err["H1_semi"], GOLDEN_ALU["H1_semi"][level])


def test_os2014_parametric_parts_and_sweep(gpu):
    g = grids.simplex(4, partitions=(4, 4))
    prob = problems.OS2014ParametricESV2007()
    d = hdd.BlockSWIPDG(g, prob)
    d.init()
    m = oracle_mesh(g)
    rp, col = o.pattern(m)
    M = d.system_matrix()
    assert M.num_components() == 1 and M.has_affine_part() and M.coefficient(0) == "mu"
    assert rel(M.affine_part(), o.assemble_lhs(m, o.os2014_affine(), None, rp, col)) <= ENTRY_TOL
    assert rel(M.component(0), o.assemble_lhs(m, o.os2014_component(), None, rp, col)) <= ENTRY_TOL
    R = d.rhs()
    assert R.num_components() == 1 and R.coefficient(0) == "mu"  # the (zero) dirichlet x factor-component vector
    assert np.all(R.component(0) == 0.0)
    b = o.assemble_rhs(m, o.esv2007_force())
    assert rel(R.affine_part(), b) <= ENTRY_TOL
    with pytest.raises(hdd.discretizations.wrong_parameter_type):
        d.solve(mu=None)
    with pytest.raises(hdd.discretizations.wrong_parameter_type):
        d.solve(mu=[0.1, 0.2])
    for mu in (0.1, 0.5, 1.0):
        A = o.assemble_lhs(m, o.os2014_factor(mu), None, rp, col)
        assert rel(M.freeze_parameter(mu), A) <= ENTRY_TOL
        u_ref = direct_solve(rp, col, A, b)
        u = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 50000}, mu=mu)
        assert rel(u, u_ref) <= SOL_TOL
        for mu_hat in (0.1, 1.0):
            prm = {"mu": mu, "mu_bar": mu, "mu_hat": mu_hat, "parameter_range_min": 0.1, "parameter_range_max": 1.0}
            ind_ref = o.indicators(m, u, o.esv2007_force(), o.os2014_factor(mu), a_hat=o.os2014_factor(mu_hat),
                                   a_bar=o.os2014_factor(mu), a_min=o.os2014_factor(0.1), a_max=o.os2014_factor(1.0))
            ind = d.indicators(u, prm)
            for k in ("nc2", "res2", "df2", "dfstar2", "resstar2", "amin"):
                assert np.abs(ind[k] - ind_ref[k]).max() <= SOL_TOL * np.abs(ind_ref[k]).max(), (k, mu, mu_hat)


GOLDEN_OS2014_MU1 = {  # test/linearelliptic-block-swipdg-expectations_os2014_2daluconform.cxx:170-212, [4 4 1]
    (1.0, 1.0): {"eta_DF_OS2014": [3.55e-1, 1.76e-1], "eta_OS2014": [7.74e-01, 3.82e-01]},
    (1.0, 0.1): {"eta_DF_OS2014": [1.36, 1.33], "eta_DF_OS2014_*": [4.13e-01, 2.05e-01]},
}


@pytest.mark.parametrize("level", [0, 1])
def test_os2014_goldens_mu1(gpu, level):
    g = grids.simplex(4 * 2 ** level, partitions=(4, 4))
    d = hdd.BlockSWIPDG(g, problems.OS2014ParametricESV2007())
    d.init()
    u = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 50000}, mu=1.0)
    est = hdd.estimators.BlockSWIPDG
    assert est.available(d) == hdd.estimators.OS2014_TYPES
    for (mu, mu_hat), gold in GOLDEN_OS2014_MU1.items():
        prm = {"mu": mu, "mu_bar": mu, "mu_hat": mu_hat, "parameter_range_min": 0.1, "parameter_range_max": 1.0}
        for typ, vals in gold.items():
            eta = est.estimate(d, u, typ, prm)
            assert abs(eta - vals[level]) <= 0.012 * vals[level], (typ, mu, mu_hat, eta)
    with pytest.raises(hdd.discretizations.wrong_input_given):
        est.estimate(d, u, "eta_OS2014", {"mu": 1.0, "mu_bar": 1.0})  # missing mu_hat
    loc = est.estimate_local(d, u, "eta_OS2014", {"mu": 1.0, "mu_bar": 1.0, "mu_hat": 1.0,
                                                  "parameter_range_min": 0.1, "parameter_range_max": 1.0})
    assert loc.shape == (16,)


GOLDEN_BLOCK_ESV = {  # test/linearelliptic-block-swipdg-expectations_esv2007_2daluconform.cxx:35-134, level 0 and 1
    (1, 1): {"eta_R_OS2014": [5.79e-01, 2.90e-01], "eta_OS2014": [1.10e+00, 5.45e-01]},
    (2, 2): {"eta_R_OS2014": [2.89e-01, 1.45e-01], "eta_OS2014": [8.10e-01, 4.00e-01]},
    (4, 4): {"eta_R_OS2014": [1.45e-01, 7.26e-02], "eta_OS2014": [6.65e-01, 3.27e-01]},
    (8, 8): {"eta_R_OS2014": [7.23e-02, 3.63e-02], "eta_OS2014": [5.93e-01, 2.91e-01]},
}


@pytest.mark.parametrize("parts", [(1, 1), (2, 2), (4, 4), (8, 8)])
def test_block_swipdg_esv2007(gpu, parts):
    for level in (0, 1):
        g = grids.simplex(4 * 2 ** level, partitions=parts)
        d = hdd.BlockSWIPDG(g, problems.ESV2007())
        d.init()
        assert d.num_subdomains() == parts[0] * parts[1]
        u = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 50000})
        m = oracle_mesh(g)
        err = o.error_norms(m, u, o.esv2007_exact())
        assert _digits3(err["L2"], GOLDEN_ALU["L2"][level])  # block == non-block norms
        for typ, vals in GOLDEN_BLOCK_ESV[parts].items():
            eta = hdd.estimators.BlockSWIPDG.estimate(d, u, typ)
            assert _digits3(eta, vals[level]), (parts, typ, eta)
        assert _digits3(hdd.estimators.BlockSWIPDG.estimate(d, u, "eta_NC_OS2014"), GOLDEN_ALU["eta_NC_ESV2007"][level])
        assert _digits3(hdd.estimators.BlockSWIPDG.estimate(d, u, "eta_DF_OS2014_*"), GOLDEN_ALU["eta_DF_ESV2007"][level])


def test_block_views_are_sub_blocks_of_the_global_matrix(gpu):
    g = grids.simplex(4, partitions=(2, 2))
    d = hdd.BlockSWIPDG(g, problems.ESV2007())
    d.init()
    rp, col = d.pattern()
    S = o.to_scipy(rp, col, d.system_matrix().affine_part()).tocsr()
    off = d.subdomain_offsets()
    assert off[-1] == g.n_dofs
    for ss in range(4):
        nbs = d.neighbouring_subdomains(ss)
        assert ss not in nbs and len(nbs) >= 2
        L = d.get_local_operator(ss)
        assert abs(L - S[off[ss]:off[ss + 1], off[ss]:off[ss + 1]]).max() == 0.0
        for nn in nbs:
            Cn = d.get_coupling_operator(ss, nn)
            assert abs(Cn - S[off[ss]:off[ss + 1], off[nn]:off[nn + 1]]).max() == 0.0
            assert Cn.nnz > 0
    with pytest.raises(hdd.discretizations.index_out_of_range):
        d.neighbouring_subdomains(4)
    far = [s for s in range(4) if s != 0 and s not in d.neighbouring_subdomains(0)]
    for nn in far:
        with pytest.raises(hdd.discretizations.wrong_input_given):
            d.get_coupling_operator(0, nn)
    u = np.arange(g.n_dofs, dtype=float)
    assert np.array_equal(d.globalize_vectors([d.localize_vector(u, s) for s in range(4)]), u)


def test_spe10_shaped_sgrid_with_cellwise_tensor(gpu):
    g = grids.cube(100, 20, (0.0, 0.0), (5.0, 1.0))
    prob = problems.Spe10Model1(g)
    d = hdd.SWIPDG(g, prob)
    d.init()
    m = oracle_mesh(g)
    rp, col = o.pattern(m)
    A = o.assemble_lhs(m, o.const(1.0), prob.diffusion_tensor, rp, col)
    b = o.assemble_rhs(m, o.cellwise(prob.force.affine.cell_values))
    assert np.array_equal(d.pattern()[1], col)
    assert rel(d.system_matrix().affine_part(), A) <= ENTRY_TOL
    assert rel(d.rhs().affine_part(), b) <= ENTRY_TOL
    u = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 200000})
    assert rel(u, direct_solve(rp, col, A, b)) <= SOL_TOL
    assert d.available_estimators() == []  # estimators exist for ALU simplices only (estimators/swipdg.hh:71)
    with pytest.raises(hdd.discretizations.you_are_using_this_wrong):
        d.estimate(u, "eta_ESV2007")


def test_error_behaviour(gpu):
    g = grids.simplex(4)
    d = hdd.SWIPDG(g, problems.ESV2007())
    with pytest.raises(hdd.discretizations.you_are_using_this_wrong):
        d.pattern()  # init() not called (discretizations/base.hh:370-377)
    with pytest.raises(hdd.discretizations.you_are_using_this_wrong):
        d.solve()
    d.init()
    with pytest.raises(hdd.discretizations.wrong_input_given):
        d.uncached_solve({"type": "bicgstab.ilut"})
    with pytest.raises(hdd.discretizations.you_are_using_this_wrong):
        d.estimate(d.solve(), "eta_unknown")
    with pytest.raises(hdd.discretizations.wrong_parameter_type):
        d.solve(mu=[1.0])
    with pytest.raises(hdd.discretizations.NotImplemented_):
        hdd.SWIPDG(g, problems.ESV2007(), polorder=3)
    # index validation happens on the device (geometry / neighbour kernels of hdd_mesh_create)
    import copy
    for field, value in (("cell_verts", g.n_verts), ("cell_verts", -1), ("cell_neigh", g.n_cells), ("cell_neigh", -2)):
        gb = copy.deepcopy(g)
        getattr(gb, field)[5, 1] = value
        with pytest.raises(hdd.discretizations.index_out_of_range):
            hdd.SWIPDG(gb, problems.ESV2007())
    gp = grids.simplex(4, partitions=(2, 2))
    gp.cell_subdomain[3], gp.cell_subdomain[4] = gp.cell_subdomain[-1], gp.cell_subdomain[-1]  # not subdomain-major
    with pytest.raises(hdd.discretizations.wrong_input_given):
        hdd.BlockSWIPDG(gp, problems.ESV2007())
    bad = problems.ESV2007()
    bad.force = problems.AffinelyDecomposable(problems.Expression("cos(x[0]", 3))
    with pytest.raises(hdd.discretizations.wrong_input_given):
        hdd.SWIPDG(g, bad)
    # solution cache: same (options, mu) returns the cached vector
    u1, i1 = d.solve(return_info=True)
    u2, i2 = d.solve(return_info=True)
    assert np.array_equal(u1, u2) and i1 == i2


def test_nonzero_dirichlet_and_neumann_faces(gpu):
    g = grids.simplex(4)
    prob = problems.ESV2007()
    prob.dirichlet = problems.AffinelyDecomposable(problems.Expression("1+x[0]*x[1]", 2, "dirichlet"))
    d = hdd.SWIPDG(g, prob)
    d.init()
    m = oracle_mesh(g)
    gd = o.fn([(1.0, o.FN_ONE)], 2)  # oracle has no x*y term: compare with the constant part only through linearity
    b_ref = o.assemble_rhs(m, o.esv2007_force(), o.const(1.0), gd)
    prob2 = problems.ESV2007()
    prob2.dirichlet = problems.AffinelyDecomposable(problems.Expression("1+0*x[0]", 2, "dirichlet"))
    d2 = hdd.SWIPDG(g, prob2)
    d2.init()
    assert rel(d2.rhs().affine_part(), b_ref) <= ENTRY_TOL
    assert np.abs(d.rhs().affine_part() - d2.rhs().affine_part()).max() > 1e-3


def test_large_grid_properties(gpu):
    """size-independent properties at a size the oracle does not run in seconds: symmetry through <Ax,y> = <x,Ay>,
    row sums of the interior stiffness (constants are in the kernel of the volume + inner-face terms), CG residual."""
    g = grids.cube(512)
    d = hdd.SWIPDG(g, problems.ESV2007())
    d.init()
    rng = np.random.default_rng(1)
    x, y = rng.standard_normal(g.n_dofs), rng.standard_normal(g.n_dofs)
    ax, ay = d.apply(x), d.apply(y)
    assert abs(ax @ y - x @ ay) <= 1e-11 * abs(ax @ y)
    one = d.apply(np.ones(g.n_dofs)).reshape(-1, 4)
    interior = (g.cell_neigh >= 0).all(axis=1)
    assert np.abs(one[interior]).max() <= 1e-9 * np.abs(one).max()
    u, info = d.solve({"type": "cg.diagonal", "precision": 1e-10, "max_iter": 20000}, return_info=True)
    b = d.rhs().affine_part()
    # the stopping test is on the recursive residual; the true one drifts by a small factor at kappa ~ 1e6
    assert np.linalg.norm(d.apply(u) - b) <= 1e-9 * np.linalg.norm(b)
    c = g.centers()
    assert np.abs(u.reshape(-1, 4).mean(axis=1) - problems.esv2007_exact(c)).max() < 1e-4


def test_neumann_faces_and_pure_neumann_fix(gpu):
    """Neumann faces contribute nothing to the lhs (boundary terms live on DirichletIntersections only,
    discretizations/block-swipdg.hh:1158-1179); an all-Neumann problem takes the unit-row path of uncached_solve
    (discretizations/base.hh:337-345): unit row 0, rhs[0] = 0, solve, subtract the mean."""
    import scipy.sparse.linalg as spla
    for kind, n in (("sgrid", 8), ("alu", 4)):
        g = _grid(kind, n)
        m = oracle_mesh(g)
        rp, col = o.pattern(m)
        # mixed: left half of the boundary faces Neumann
        cen = g.centers()
        bt = np.ones((g.n_cells, g.n_loc), np.uint8)
        bt[(cen[:, 0] < 0)[:, None] & (g.cell_neigh < 0)] = 2
        d = hdd.SWIPDG(g, problems.ESV2007(), boundary_info=bt)
        d.init()
        A = o.assemble_lhs(m, o.const(1.0), None, rp, col, bnd_dirichlet=(bt == 1))
        assert rel(d.system_matrix().affine_part(), A) <= ENTRY_TOL
        b = o.assemble_rhs(m, o.esv2007_force())
        u = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 50000})
        assert rel(u, direct_solve(rp, col, A, b)) <= SOL_TOL
        # all Neumann (simplices only: with the reference's midpoint volume rule the Q1 matrix gains a second,
        # checkerboard null vector as soon as no Dirichlet face pins it, so the cube case is singular by construction)
        if kind != "alu":
            continue
        bt[:] = 2
        d = hdd.SWIPDG(g, problems.ESV2007(), boundary_info=bt)
        d.init()
        A = o.assemble_lhs(m, o.const(1.0), None, rp, col, bnd_dirichlet=np.zeros_like(bt))
        assert rel(d.system_matrix().affine_part(), A) <= ENTRY_TOL
        S = o.to_scipy(rp, col, A).tolil()
        S[0, :] = 0.0
        S[:, 0] = 0.0
        S[0, 0] = 1.0
        b2 = b.copy()
        b2[0] = 0.0
        x = spla.spsolve(S.tocsc(), b2)
        x -= x.mean()
        for typ in ("cg.diagonal", "cg.mg"):  # the multigrid hierarchy is built from the unit-row operator
            u = d.solve({"type": typ, "precision": 1e-13, "max_iter": 50000})
            assert abs(u.mean()) <= 1e-12 * np.abs(u).max(), typ
            assert rel(u, x) <= 1e-7, typ


# ---- polOrder 2 (BASELINE config 5: "SWIPDG p1 and p2"): P2 / Q2, GPU vs oracle -----------------------------------
def _oracle_system_p(g, polorder, factor, force, tensor=None):
    m = oracle_mesh(g).with_polorder(polorder)
    rp, col = o.pattern(m)
    return m, rp, col, o.assemble_lhs(m, factor, tensor, rp, col), o.assemble_rhs(m, force)


@pytest.mark.parametrize("kind,n", [("alu", 2), ("alu", 4), ("sgrid", 6), ("sgrid", 1), ("alu", 1)])
def test_p2_pattern_entries_and_solve(gpu, kind, n):
    g = _grid(kind, n)
    d = hdd.SWIPDG(g, problems.ESV2007(), polorder=2)
    d.init()
    m, rp, col, A, b = _oracle_system_p(g, 2, o.const(1.0), o.esv2007_force())
    assert d.num_dofs() == m.n_dofs == g.n_cells * (6 if kind == "alu" else 9)
    rp_g, col_g = d.pattern()
    assert np.array_equal(rp_g, rp) and np.array_equal(col_g, col)
    assert rel(d.system_matrix().affine_part(), A) <= ENTRY_TOL
    assert rel(d.rhs().affine_part(), b) <= ENTRY_TOL
    x = np.random.default_rng(0).standard_normal(m.n_dofs)
    assert rel(d.apply(x), o.spmv(rp, col, A, x)) <= 1e-13
    u_ref = direct_solve(rp, col, A, b)
    for typ in ("cg.diagonal", "cg.blockdiagonal", "cg.identity"):
        u, info = d.solve({"type": typ, "precision": 1e-13, "max_iter": 50000}, return_info=True)
        assert info["converged"]
        assert rel(u, u_ref) <= SOL_TOL
    # device error norms against the oracle's
    e_ref = o.error_norms(m, u_ref, o.esv2007_exact(), order=8)
    e = d.error_norms(*problems.ESV2007_EXACT, vector=u_ref, order=8)
    for key in ("L2", "H1_semi", "energy"):
        assert abs(e[key] - e_ref[key]) <= SOL_TOL * e_ref[key]


def test_p2_parametric_cellwise_and_block_views(gpu):
    """OS2014 (expression factor, two affine parts) and a cell-wise tensor on p2; block views on a 2x2 partition"""
    g = grids.simplex(4, partitions=(2, 2))
    prob = problems.OS2014ParametricESV2007()
    d = hdd.BlockSWIPDG(g, prob, polorder=2)
    d.init()
    m = oracle_mesh(g).with_polorder(2)
    rp, col = o.pattern(m)
    M = d.system_matrix()
    assert M.num_components() == 1 and M.has_affine_part()
    assert rel(M.affine_part(), o.assemble_lhs(m, o.os2014_affine(), None, rp, col)) <= ENTRY_TOL
    assert rel(M.component(0), o.assemble_lhs(m, o.os2014_component(), None, rp, col)) <= ENTRY_TOL
    A = o.assemble_lhs(m, o.os2014_factor(0.3), None, rp, col)
    assert rel(M.freeze_parameter(0.3), A) <= ENTRY_TOL
    b = o.assemble_rhs(m, o.esv2007_force())
    u = d.solve({"type": "cg.blockdiagonal", "precision": 1e-13, "max_iter": 50000}, mu=0.3)
    assert rel(u, direct_solve(rp, col, A, b)) <= SOL_TOL
    S = o.to_scipy(rp, col, o.assemble_lhs(m, o.os2014_affine(), None, rp, col))
    off = d.subdomain_offsets()
    assert off[-1] == m.n_dofs
    for ss in range(d.num_subdomains()):
        B = d.get_local_operator(ss)
        assert abs(B - S[off[ss]:off[ss + 1], off[ss]:off[ss + 1]]).max() <= ENTRY_TOL * abs(S).max()
        for nn in d.neighbouring_subdomains(ss):
            Cb = d.get_coupling_operator(ss, nn)
            assert abs(Cb - S[off[ss]:off[ss + 1], off[nn]:off[nn + 1]]).max() <= ENTRY_TOL * abs(S).max()
    # cell-wise tensor on Q2
    g2 = grids.cube(6)
    k = np.random.default_rng(3).uniform(0.1, 10.0, g2.n_cells)
    tensor = np.zeros((g2.n_cells, 4))
    tensor[:, 0] = tensor[:, 3] = k
    prob2 = problems.ESV2007()
    prob2.diffusion_tensor = tensor
    d2 = hdd.SWIPDG(g2, prob2, polorder=2)
    d2.init()
    m2, rp2, col2, A2, b2 = _oracle_system_p(g2, 2, o.const(1.0), o.esv2007_force(), tensor)
    assert rel(d2.system_matrix().affine_part(), A2) <= ENTRY_TOL
    ds = hdd.SWIPDG(grids.simplex(2), problems.ESV2007(), polorder=2)
    ds.init()
    with pytest.raises(hdd.discretizations.NotImplemented_):
        ds.estimate(np.zeros(ds.num_dofs()), "eta_ESV2007")
    with pytest.raises(hdd.discretizations.NotImplemented_):
        hdd.SWIPDG(g2, problems.ESV2007(), polorder=3)


# ---- a9: non-zero Neumann data (Functionals::L2Face, discretizations/swipdg.hh:335-356) --------------------------
def test_q2_closed_form_kernel_full_tensor_cellwise_factor_rectangles(gpu, monkeypatch):
    """the closed-form Q2 kernel (1-d quadrature matrices instead of quadrature loops) against the oracle's quadrature loops
    where its formulas have the most terms: cells with hx != hy, a full symmetric cell-wise tensor, a cell-wise factor"""
    g = grids.cube(7, 5, lower_left=(-1.0, 0.0), upper_right=(2.5, 1.0))
    rng = np.random.default_rng(11)
    k = rng.uniform(0.5, 4.0, (g.n_cells, 2))
    off = rng.uniform(-0.4, 0.4, g.n_cells)
    tensor = np.stack([k[:, 0], off, off, k[:, 1]], axis=1)
    a = rng.uniform(0.2, 5.0, g.n_cells)
    prob = problems.Problem(problems.AffinelyDecomposable(problems.Cellwise(a, "diffusion_factor")),
                            problems.AffinelyDecomposable(problems.Expression(problems.ESV2007_FORCE, 3, "force")),
                            diffusion_tensor=tensor, name="q2 closed form")
    d = hdd.SWIPDG(g, prob, polorder=2)
    d.init()
    m, rp, col, A, b = _oracle_system_p(g, 2, o.cellwise(a), o.esv2007_force(), tensor)
    rp_g, col_g = d.pattern()
    assert np.array_equal(rp_g, rp) and np.array_equal(col_g, col)
    assert rel(d.system_matrix().affine_part(), A) <= ENTRY_TOL
    assert rel(d.rhs().affine_part(), b) <= ENTRY_TOL
    # constant factor, same tensor
    prob_c = problems.ESV2007()
    prob_c.diffusion_tensor = tensor
    dc = hdd.SWIPDG(g, prob_c, polorder=2)
    dc.init()
    Ac = o.assemble_lhs(m, o.const(1.0), tensor, rp, col)
    assert rel(dc.system_matrix().affine_part(), Ac) <= ENTRY_TOL


@pytest.mark.parametrize("kind,n,polorder", [("alu", 4, 1), ("sgrid", 8, 1), ("alu", 2, 2), ("sgrid", 4, 2)])
def test_nonzero_neumann_and_dirichlet_data(gpu, kind, n, polorder):
    g = _grid(kind, n)
    cen = g.centers()
    bt = np.ones((g.n_cells, g.n_loc), np.uint8)
    bt[(cen[:, 0] < 0)[:, None] & (g.cell_neigh < 0)] = 2
    prob = problems.ESV2007()
    prob.neumann = problems.AffinelyDecomposable(problems.Expression("0.5+x[0]*x[1]-2*x[1]", 2, "neumann"))
    prob.dirichlet = problems.AffinelyDecomposable(problems.Expression("1+x[0]*x[1]", 2, "dirichlet"))
    d = hdd.SWIPDG(g, prob, boundary_info=bt, polorder=polorder)
    d.init()
    m = oracle_mesh(g).with_polorder(polorder)
    rp, col = o.pattern(m)
    gn = o.fn([(0.5, o.FN_ONE), (1.0, o.FN_XY), (-2.0, o.FN_Y)], 2)
    gd = o.fn([(1.0, o.FN_ONE), (1.0, o.FN_XY)], 2)
    b = o.assemble_rhs(m, o.esv2007_force(), o.const(1.0), gd, neumann=gn, bnd_type=bt)
    assert rel(d.rhs().affine_part(), b) <= ENTRY_TOL
    b0 = o.assemble_rhs(m, o.esv2007_force(), o.const(1.0), gd, bnd_type=bt)
    assert np.abs(b - b0).max() > 1e-3  # the Neumann term is really there
    A = o.assemble_lhs(m, o.const(1.0), None, rp, col, bnd_dirichlet=(bt == 1))
    u = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 50000})
    assert rel(u, direct_solve(rp, col, A, b)) <= SOL_TOL
    # parametric Neumann data: one rhs component per part, coefficient string preserved
    prob.neumann = problems.AffinelyDecomposable(problems.Constant(0.0, "neumann"),
                                                 [problems.Expression("x[1]", 1, "neumann_0")], ["2*mu"])
    prob.parameter_name, prob.parameter_size = "mu", 1
    dp = hdd.SWIPDG(g, prob, boundary_info=bt, polorder=polorder)
    dp.init()
    R = dp.rhs()
    assert R.num_components() == 1 and R.coefficient(0) == "2*mu"
    comp = o.assemble_rhs(m, None, neumann=o.fn([(1.0, o.FN_Y)], 1), bnd_type=bt)
    assert rel(R.component(0), comp) <= ENTRY_TOL


# ---- 8f rank 1: product matrices ----------------------------------------------------------------------------------
@pytest.mark.parametrize("kind,n,polorder", [("alu", 4, 1), ("sgrid", 8, 1), ("alu", 2, 2), ("sgrid", 4, 2)])
def test_products(gpu, kind, n, polorder):
    g = _grid(kind, n)
    ids = ["l2", "h1_semi", "elliptic", "boundary_l2", "penalty", "energy", "not_a_product"]
    d = hdd.SWIPDG(g, problems.OS2014ParametricESV2007(), polorder=polorder, only_these_products=ids)
    assert d.available_products() == sorted(ids[:-1])
    d.init()
    m = oracle_mesh(g).with_polorder(polorder)
    rp, col = o.pattern(m)
    rpv, colv = o.pattern_volume(m)
    rp_g, col_g = d.pattern_volume()
    assert np.array_equal(rp_g, rpv) and np.array_equal(col_g, colv)
    rng = np.random.default_rng(5)
    u, v = rng.standard_normal(m.n_dofs), rng.standard_normal(m.n_dofs)
    for pid in ("l2", "h1_semi", "boundary_l2"):
        P = d.get_product(pid)
        assert P.num_components() == 0 and P.has_affine_part() and P.volume_pattern()
        ref = o.assemble_product(m, pid, rpv, colv)
        assert rel(P.affine_part(), ref) <= ENTRY_TOL
        S = o.to_scipy(rpv, colv, ref)
        assert abs(P.apply2(u, v) - u @ (S @ v)) <= 1e-12 * np.abs(S).sum()
    for pid, (r, c) in (("elliptic", (rpv, colv)), ("penalty", (rp, col))):
        P = d.get_product(pid)
        assert P.num_components() == 1 and P.has_affine_part() and P.coefficient(0) == d.system_matrix().coefficient(0)
        assert P.volume_pattern() == (pid == "elliptic")
        assert rel(P.affine_part(), o.assemble_product(m, pid, r, c, factor=o.os2014_affine())) <= ENTRY_TOL
        assert rel(P.component(0), o.assemble_product(m, pid, r, c, factor=o.os2014_component())) <= ENTRY_TOL
        ref = o.assemble_product(m, pid, r, c, factor=o.os2014_factor(0.4))
        assert rel(P.freeze_parameter(0.4), ref) <= ENTRY_TOL
        S = o.to_scipy(r, c, ref)
        assert abs(P.apply2(u, v, mu=0.4) - u @ (S @ v)) <= 1e-12 * np.abs(S).sum()
        assert abs(P.induced_norm(u, mu=0.4) - np.sqrt(u @ (S @ u))) <= 1e-10 * np.sqrt(u @ (S @ u))
    E = d.get_product("energy")
    assert not E.volume_pattern() and E.num_components() == 1
    assert np.array_equal(E.affine_part(), d.system_matrix().affine_part())
    with pytest.raises(hdd.discretizations.wrong_input_given):
        d.get_product("h1")
    d0 = hdd.SWIPDG(g, problems.ESV2007(), polorder=polorder)
    d0.init()
    assert d0.available_products() == []
    with pytest.raises(hdd.discretizations.you_are_using_this_wrong):
        d0.get_product("l2")
    # products requested after init() are assembled at once; l2 norm of the constant 1 is sqrt(|Omega|)
    d1 = hdd.BlockSWIPDG(_grid(kind, n, (2, 2)), problems.ESV2007(), polorder=polorder)
    d1.init()
    L = capi_products(d1, ["l2", "elliptic"])
    one = np.ones(d1.num_dofs())
    assert abs(L["l2"].induced_norm(one) - 2.0) <= 1e-12
    assert abs(L["elliptic"].induced_norm(one)) <= 1e-6
    M = o.to_scipy(rpv, colv, o.assemble_product(m, "l2", rpv, colv))
    off = d1.subdomain_offsets()
    loc = d1.get_local_product(1, "l2")
    assert loc.shape == (off[2] - off[1],) * 2 and abs(loc.sum() - 1.0) <= 1e-12  # |subdomain| = 1


def capi_products(d, ids):
    import ctypes as C
    from dune_hdd_b200 import capi
    arr = (C.c_char_p * len(ids))(*[i.encode() for i in ids])
    capi.check(capi.lib().hdd_swipdg_only_these_products(d._h, arr, len(ids)))
    return {i: d.get_product(i) for i in ids}


def test_error_norms_on_the_device(gpu):
    for kind, n in (("alu", 8), ("sgrid", 16)):
        g = _grid(kind, n)
        d = hdd.SWIPDG(g, problems.ESV2007())
        d.init()
        u = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 50000})
        m = oracle_mesh(g)
        e_ref = o.error_norms(m, u, o.esv2007_exact(), order=5)
        for vec in (u, None):  # None: the last solution, resident on the device
            e = d.error_norms(*problems.ESV2007_EXACT, vector=vec, order=5)
            for key in ("L2", "H1_semi", "energy"):
                assert abs(e[key] - e_ref[key]) <= SOL_TOL * e_ref[key]


# ---- "cg.mg": two-level multigrid preconditioner on structured Q1 grids ---------------------------------------------
@pytest.mark.parametrize("n,parts", [(8, (1, 1)), (16, (2, 2)), (32, (1, 1)), (48, (4, 4)), (3, (1, 1))])
def test_cg_mg_matches_direct_solve(gpu, n, parts):
    g = grids.cube(n, partitions=parts)  # the partitioned grids have subdomain-major cell numbering
    d = hdd.SWIPDG(g, problems.ESV2007())
    d.init()
    assert "cg.mg" in d.solver_types()
    m, rp, col, A, b = oracle_system(g, o.const(1.0), o.esv2007_force())
    u_ref = direct_solve(rp, col, A, b)
    u, info = d.solve({"type": "cg.mg", "precision": 1e-13, "max_iter": 500}, return_info=True)
    assert info["converged"] and rel(u, u_ref) <= SOL_TOL
    _, ij = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 50000}, return_info=True)
    assert info["iterations"] <= 70 and (n < 16 or info["iterations"] < ij["iterations"] / 2)


def test_cg_mg_spe10_shape_parametric_and_requirements(gpu):
    g = grids.cube(100, 20, (0.0, 0.0), (5.0, 1.0))
    prob = problems.Spe10Model1(g)
    d = hdd.SWIPDG(g, prob)
    d.init()
    m = oracle_mesh(g)
    rp, col = o.pattern(m)
    A = o.assemble_lhs(m, o.const(1.0), prob.diffusion_tensor, rp, col)
    b = d.rhs().affine_part()
    u, info = d.solve({"type": "cg.mg", "precision": 1e-12, "max_iter": 2000}, return_info=True)
    assert info["converged"]
    assert np.linalg.norm(o.spmv(rp, col, A, u) - b) <= 1e-9 * np.linalg.norm(b)
    _, ij = d.solve({"type": "cg.blockdiagonal", "precision": 1e-12, "max_iter": 200000}, return_info=True)
    assert info["iterations"] < ij["iterations"] / 4
    # parametric operator: the hierarchy is rebuilt for every frozen A(mu)
    g2 = grids.cube(32)
    fac = problems.AffinelyDecomposable(problems.Constant(1.0), [problems.Expression("x[0]*x[0]+0.1", 2)], ["mu"])
    p2 = problems.Problem(fac, problems.ESV2007().force, parameter_name="mu", parameter_size=1)
    d2 = hdd.SWIPDG(g2, p2)
    d2.init()
    for mu in (0.1, 10.0):
        um = d2.solve({"type": "cg.mg", "precision": 1e-13, "max_iter": 1000}, mu=mu)
        ud = d2.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 100000}, mu=mu)
        assert rel(um, ud) <= SOL_TOL
    # needs a logically structured grid with p = 1: a simplex grid whose vertices are not numbered as a lattice is refused
    gs = grids.simplex(4)
    perm = np.random.default_rng(3).permutation(gs.n_verts).astype(np.int32)
    xy = np.empty_like(gs.xy)
    xy[perm] = gs.xy
    ds = hdd.SWIPDG(grids.Grid(gs.kind, xy, perm[gs.cell_verts], gs.cell_neigh), problems.ESV2007())
    ds.init()
    with pytest.raises(hdd.discretizations.requirements_not_met):
        ds.solve({"type": "cg.mg", "precision": 1e-10, "max_iter": 100})
    dp2 = hdd.SWIPDG(grids.simplex(4), problems.ESV2007(), polorder=2)
    dp2.init()
    with pytest.raises(hdd.discretizations.requirements_not_met):
        dp2.solve({"type": "cg.mg", "precision": 1e-10, "max_iter": 100})
    dq = hdd.SWIPDG(grids.cube(8), problems.ESV2007(), polorder=2)
    dq.init()
    with pytest.raises(hdd.discretizations.requirements_not_met):
        dq.solve({"type": "cg.mg", "precision": 1e-10, "max_iter": 100})
    # 42 x 42: halving stops at 21 x 21 vertex cells (484 vertices > 400, odd)
    d42 = hdd.SWIPDG(grids.cube(42), problems.ESV2007())
    d42.init()
    with pytest.raises(hdd.discretizations.requirements_not_met, match="21 x 21"):
        d42.solve({"type": "cg.mg", "precision": 1e-10, "max_iter": 100})


@pytest.mark.parametrize("kind,n,polorder", [("alu", 16, 1), ("alu", 32, 1), ("alu", 16, 2), ("sgrid", 32, 2), ("sgrid", 40, 1)])
def test_bulk_copy_spmv_paths(gpu, kind, n, polorder):
    """grids large enough (>= 1024 cells) for the TMA-staged CG SpMV kernels of every block size, against the direct
    solve and, iterate by iterate, against the oracle's CG"""
    g = _grid(kind, n)
    assert g.n_cells >= 1024
    os.environ["HDD_SPMV_CTAS"] = "3"  # few CTAs: every CTA walks its shared-memory ring several times
    try:
        _bulk_copy_case(g, polorder)
    finally:
        del os.environ["HDD_SPMV_CTAS"]
    _bulk_copy_case(g, polorder)


def _bulk_copy_case(g, polorder):
    d = hdd.SWIPDG(g, problems.ESV2007(), polorder=polorder)
    d.init()
    m = oracle_mesh(g).with_polorder(polorder)
    rp, col = o.pattern(m)
    A = o.assemble_lhs(m, o.const(1.0), None, rp, col)
    b = o.assemble_rhs(m, o.esv2007_force())
    u_ref = direct_solve(rp, col, A, b)
    u, info = d.solve({"type": "cg.diagonal", "precision": 1e-13, "max_iter": 100000}, return_info=True)
    assert info["converged"] and rel(u, u_ref) <= SOL_TOL
    # iterates: 10 iterations from the same start follow the oracle CG to rounding
    x10, it, _ = o.cg(rp, col, A, b, precond=1, rtol=1e-30, maxit=10)
    try:
        d.uncached_solve({"type": "cg.diagonal", "precision": 1e-30, "max_iter": 10})
    except hdd.discretizations.linear_solver_failed:
        pass
    import ctypes as C
    from dune_hdd_b200 import capi
    xp = C.POINTER(C.c_double)()
    capi.check(capi.lib().hdd_solution_dev(d._h, C.byref(xp)))
    xg = np.empty(d.num_dofs())
    capi.check(capi.lib().hdd_copy_to_host(d._h, capi.ptr(xg), xp, C.c_size_t(xg.nbytes)))
    assert rel(xg, x10) <= 1e-11


@pytest.mark.parametrize("level", [0, 1, 2, 3])
def test_sgrid_goldens_entirely_on_the_device(gpu, level):
    """the committed SGrid expectations (test/linearelliptic-swipdg-expectations_esv2007_2dsgrid.cxx:31-36) reproduced
    without the oracle: assembly, multigrid-preconditioned CG and the error norms all run on the GPU"""
    n = 8 * 2 ** level
    d = hdd.SWIPDG(grids.cube(n), problems.ESV2007())
    d.init()
    d.solve({"type": "cg.mg", "precision": 1e-12, "max_iter": 1000})
    e = d.error_norms(*problems.ESV2007_EXACT, order=7)
    stem = "linearelliptic-swipdg-expectations_esv2007_2dsgrid"
    assert abs(e["L2"] - golden(stem, "L2")[level]) <= 0.006 * e["L2"]
    assert abs(e["H1_semi"] - golden(stem, "H1_semi")[level]) <= 0.006 * e["H1_semi"]


@pytest.mark.parametrize("level", [0, 1, 2])
def test_alu_error_goldens_on_the_device(gpu, level):
    """test/linearelliptic-swipdg-expectations_esv2007_2daluconform.cxx:32-41 (L2, H1_semi, energy) with device norms"""
    d = hdd.SWIPDG(grids.simplex(4 * 2 ** level), problems.ESV2007())
    d.init()
    d.solve({"type": "cg.blockdiagonal", "precision": 1e-12, "max_iter": 100000})
    e = d.error_norms(*problems.ESV2007_EXACT, order=5)
    stem = "linearelliptic-swipdg-expectations_esv2007_2daluconform"
    for key in ("L2", "H1_semi", "energy"):
        assert abs(e[key] - golden(stem, key)[level]) <= 0.006 * golden(stem, key)[level]


def test_convergence_studies_reproduce_the_expectation_tables(gpu):
    """SWIPDGStudy / BlockSWIPDGStudy (test/linearelliptic-swipdg.cc:86-109, test/linearelliptic-block-swipdg.cc) on
    the first three levels of the ESV2007 ladder: every column of the committed expectations, computed on the device"""
    from dune_hdd_b200 import studies, testcases
    t = studies.SWIPDGStudy(testcases.ESV2007("alu", num_refinements=2)).run()
    stem = "linearelliptic-swipdg-expectations_esv2007_2daluconform"
    assert t["size"] == [128, 512, 2048]
    for col in ("L2", "H1_semi", "energy", "eta_NC_ESV2007", "eta_R_ESV2007", "eta_DF_ESV2007", "eta_ESV2007",
                "eff_ESV2007", "eta_ESV2007_alt", "eff_ESV2007_alt"):
        tol = 0.01 if col.startswith("eff") else 0.006
        for level in range(3):
            assert abs(t[col][level] - golden(stem, col)[level]) <= tol * golden(stem, col)[level], (col, level, t[col])
    assert all(abs(e - 2.0) < 0.05 for e in t["eoc"]["L2"]) and all(abs(e - 1.0) < 0.05 for e in t["eoc"]["energy"])
    b = studies.BlockSWIPDGStudy(testcases.ESV2007Multiscale((4, 4), num_refinements=1)).run()
    stem = "linearelliptic-block-swipdg-expectations_esv2007_2daluconform"
    for col in ("energy", "eta_NC_OS2014", "eta_R_OS2014", "eta_DF_OS2014", "eta_OS2014", "eff_OS2014"):
        tol = 0.01 if col.startswith("eff") else 0.006
        for level in range(2):
            ref = golden(stem, col, "[4 4 1]")[level]
            assert abs(b[col][level] - ref) <= tol * ref, (col, level, b[col])


# ---- prolongation and the reference-level error norms of the studies (SURVEY 8f rank 3) -------------------------
@pytest.mark.parametrize("kind", ["alu", "sgrid"])
@pytest.mark.parametrize("pc,pf", [(1, 1), (1, 2), (2, 1), (2, 2)])
def test_prolongation_matches_the_oracle(gpu, kind, pc, pf):
    """hdd_prolong = Operators::Prolongation (test/linearelliptic.hh:168-176) on partitioned (renumbered) grids"""
    gc, gf = _grid(kind, 2 if kind == "alu" else 3, (1, 1)), _grid(kind, 8 if kind == "alu" else 12, (2, 2))
    dc, df = hdd.SWIPDG(gc, problems.ESV2007(), polorder=pc), hdd.SWIPDG(gf, problems.ESV2007(), polorder=pf)
    mc, mf = oracle_mesh(gc).with_polorder(pc), oracle_mesh(gf).with_polorder(pf)
    father = grids.fathers(gc, gf)
    assert np.array_equal(father, o.fathers(mc, mf))
    u = np.random.default_rng(7).standard_normal(dc.num_dofs())
    ref = o.prolong(mc, u, mf)
    for fa in (None, father):
        assert np.abs(df.prolong(dc, u, father=fa) - ref).max() <= 1e-13 * np.abs(u).max()
    bad = father.copy()
    bad[3] = gc.n_cells
    with pytest.raises(hdd.discretizations.index_out_of_range):
        df.prolong(dc, u, father=bad)


def test_os2014_study_effectivities_on_the_reference_level(gpu):
    """BlockSWIPDGStudy on OS2014 [4 4 1] at mu = mu_bar = 1 (test/OS2014_parametric_convergence_study.cc:100-110): no exact
    solution, so the energy error is || u_ref - P u_h || in the Products::Elliptic norm on the 32768-triangle reference
    level; the effectivities of the committed expectations (lines 172-174, 202-204), device only"""
    from dune_hdd_b200 import studies, testcases
    stem = "linearelliptic-block-swipdg-expectations_os2014_2daluconform"
    for mu_hat in (1.0, 0.1):
        case = testcases.OS2014ParametricESV2007Multiscale({"mu": 1.0, "mu_bar": 1.0, "mu_hat": mu_hat}, (4, 4), num_refinements=3)
        study = studies.BlockSWIPDGStudy(case)
        assert "energy_mu" in study.available_norms()
        t = study.run(levels=(0, 1), only_these_estimators=("eta_OS2014", "eta_OS2014_*", "eff_OS2014_mu", "eff_OS2014_*_mu"))
        key = "1,1,%g" % mu_hat
        for col in ("eta_OS2014", "eta_OS2014_*", "eff_OS2014_mu", "eff_OS2014_*_mu"):
            for level in range(2):
                ref = golden(stem, col, "[4 4 1]", key)[level]
                assert abs(t[col][level] - ref) <= 0.012 * ref, (mu_hat, col, level, t[col])
        # mu = 1: a = 1, the energy norm is the H1 semi norm; implied by the goldens: 0.774 / 2.36 = 0.328
        assert abs(t["energy_mu"][0] - t["H1_semi"][0]) <= 1e-10 and abs(t["energy_mu"][0] - 0.3275) < 1e-3
        assert abs(t["eoc"]["energy_mu"][0] - 1.0) < 0.05 and abs(t["eoc"]["L2"][0] - 2.0) < 0.1


# ---- the config-file driver on the device (SURVEY 8f rank 4) and the localization study --------------------------
def test_example_driver_and_thermalblock_vector_parameter(gpu, tmp_path):
    """examples/swipdg_main.py (= examples/linearelliptic/swipdg_main.cc) end to end: default config -> ESV2007 on the 8 x 8
    SGrid of [0,1]^2 -> .vtu; then the thermalblock problem of the same config with its 4-component parameter
    diffusion_factor, one solve per [parameter] entry, against the oracle's direct solve"""
    import subprocess
    import sys
    import xml.etree.ElementTree as ET
    from dune_hdd_b200 import discreteproblem as dp
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = os.path.join(root, "examples", "swipdg_main.py")
    cls = dp.LinearellipticExampleSWIPDG
    for expected in ("Please review the configuration", "discretization is not parametric, solving..."):
        r = subprocess.run([sys.executable, script, str(tmp_path)], capture_output=True, text=True)
        assert r.returncode == 0 and expected in r.stdout, r.stdout + r.stderr
    g = grids.cube(8, 8, (0.0, 0.0), (1.0, 1.0))
    m, rp, col, A, b = oracle_system(g, o.const(1.0), o.esv2007_force())
    u_ref = direct_solve(rp, col, A, b)
    piece = ET.parse(str(tmp_path / "linearelliptic.swipdg.solution.vtu")).getroot().find("UnstructuredGrid/Piece")
    assert piece.find("PointData/DataArray").attrib["Name"] == "solution"
    val = np.array(piece.find("PointData/DataArray").text.split(), float).reshape(g.n_cells, 4)[:, [0, 1, 3, 2]]
    assert rel(val.reshape(-1), u_ref) <= 1e-6  # the driver solves with the default options (1e-10)
    cfg = tmp_path / (cls.static_id() + ".cfg")
    cfg.write_text(cfg.read_text().replace("problem = hdd.linearelliptic.problem.ESV2007", "problem = hdd.linearelliptic.problem.thermalblock"))
    example = cls("sgrid", device=0)
    example.initialize([str(tmp_path)])
    d = example.discretization()
    assert d.parametric() and d.parameter_type() == {"diffusion_factor": 4}
    ind = np.array([c.cell_values for c in d.problem.diffusion_factor.components])
    parameters = example.discrete_problem().parameters()
    assert len(parameters) == 2
    for parameter in parameters:
        mu = parameter["diffusion_factor"]
        u = d.solve({"type": "cg.blockdiagonal", "precision": 1e-13, "max_iter": 20000}, mu=mu)
        a = (np.array(mu)[:, None] * ind).sum(axis=0)
        A = o.assemble_lhs(m, o.cellwise(a), None, rp, col)
        assert rel(u, direct_solve(rp, col, A, o.assemble_rhs(m, o.const(1.0)))) <= SOL_TOL
    with pytest.raises(hdd.discretizations.wrong_parameter_type):
        d.solve(mu=[1.0, 2.0])


def test_reference_indicators_of_the_localization_study(gpu):
    """compute_reference_indicators (test/linearelliptic-block-swipdg.hh:122-199, test/linearelliptic-swipdg.hh:133-223):
    the energy of u_ref - P u_h per subdomain / per coarse cell, against the same quantity from oracle matrices"""
    from dune_hdd_b200 import studies, testcases
    case = testcases.OS2014ParametricESV2007Multiscale({"mu": 0.5, "mu_bar": 0.5, "mu_hat": 0.5}, (2, 2), num_refinements=1)
    grid, grid_r = case.level_grid(0), case.reference_grid()
    mc, mf = oracle_mesh(grid), oracle_mesh(grid_r)

    def oracle_solution(mesh):
        rp, col = o.pattern(mesh)
        return direct_solve(rp, col, o.assemble_lhs(mesh, o.os2014_factor(0.5), None, rp, col), o.assemble_rhs(mesh, o.esv2007_force()))

    father = o.fathers(mc, mf)
    diff = (oracle_solution(mf) - o.prolong(mc, oracle_solution(mc), mf, father)).reshape(mf.nc, 3)
    rpv, colv = o.pattern_volume(mf)
    blocks = o.assemble_product(mf, "elliptic", rpv, colv, factor=o.os2014_factor(0.5)).reshape(mf.nc, 3, 3)
    for cls, group, n in ((studies.BlockSWIPDGStudy, grid.cell_subdomain[father], 4), (studies.SWIPDGStudy, father, grid.n_cells)):
        study = cls(case)
        disc = study._make(grid)
        disc.init()
        u = disc.solve(study.solver_options, mu=0.5)
        ind = study.reference_indicators(disc, u)
        ref = studies.localize_energy(blocks, diff, group, n)
        assert ind.shape == (n,) and np.abs(ind - ref).max() <= 1e-7 * ref.max()
        assert abs((ind * np.bincount(group, minlength=n)).sum() - 1.0) < 1e-12
        local = study.indicators(disc, u, "eta_OS2014" if cls is studies.BlockSWIPDGStudy else "eta_ESV2007")
        assert local.shape == (n,)


def test_true_residual_and_vector_shape_checks(gpu):
    """hdd_residual recomputes ||b - A x|| / ||b|| of the device solution from scratch; the façade refuses vectors of
    the wrong size (shapes_do_not_match in the reference) before the C-ABI would copy num_owned_dofs() doubles."""
    g = grids.cube(24)
    d = hdd.SWIPDG(g, problems.ESV2007())
    d.init()
    with pytest.raises(hdd.discretizations.you_are_using_this_wrong):
        d.residual()  # no solution yet
    u, info = d.solve({"type": "cg.mg", "precision": 1e-12, "max_iter": 500}, return_info=True)
    m, rp, col, A, b = oracle_system(g, o.const(1.0), o.esv2007_force())
    res_ref = np.linalg.norm(b - o.spmv(rp, col, A, u)) / np.linalg.norm(b)
    res, floor = d.residual(with_floor=True)
    assert res <= 1e-11 and abs(res - res_ref) <= 0.5 * max(res, res_ref) + 1e-14
    assert 0.0 < floor < 1e-9
    # a solve that stops early leaves a large true residual
    with pytest.raises(hdd.discretizations.linear_solver_failed):
        d.uncached_solve({"type": "cg.diagonal", "precision": 1e-12, "max_iter": 3})
    assert d.residual() > 1e-3
    bad = np.zeros(g.n_dofs + 1)
    for call in (lambda: d.apply(bad), lambda: d.error_norms(*problems.ESV2007_EXACT, vector=bad),
                 lambda: d.uncached_solve(out=bad), lambda: d.uncached_solve(out=np.zeros(g.n_dofs, np.float32))):
        with pytest.raises(hdd.discretizations.wrong_input_given):
            call()
    gs = grids.simplex(4)
    ds = hdd.SWIPDG(gs, problems.ESV2007(), only_these_products=("l2",))
    ds.init()
    bad = np.zeros(gs.n_dofs - 3)
    for call in (lambda: ds.estimate(bad, "eta_ESV2007"), lambda: ds.estimate_local(bad, "eta_ESV2007"),
                 lambda: ds.indicators(bad), lambda: ds.get_product("l2").apply2(bad, bad)):
        with pytest.raises(hdd.discretizations.wrong_input_given):
            call()


def test_estimator_with_expression_factor_and_many_segments(gpu):
    """the expression branch of the indicator kernel (OS2014 factor at mu_hat != mu) on a grid whose subdomains span
    several reduction segments (> 8192 cells per subdomain), against the oracle"""
    g = grids.simplex(64, partitions=(1, 1))  # 32768 triangles in one subdomain: four segments
    prob = problems.OS2014ParametricESV2007()
    d = hdd.BlockSWIPDG(g, prob)
    d.init()
    mu = 0.3
    u = d.solve({"type": "cg.blockdiagonal", "precision": 1e-12, "max_iter": 20000}, mu=mu)
    prm = {"mu": mu, "mu_bar": mu, "mu_hat": 0.7, "parameter_range_min": 0.1, "parameter_range_max": 1.0}
    m = oracle_mesh(g)
    ind_ref = o.indicators(m, u, o.esv2007_force(), o.os2014_factor(mu), a_hat=o.os2014_factor(0.7),
                           a_bar=o.os2014_factor(mu), a_min=o.os2014_factor(0.1), a_max=o.os2014_factor(1.0))
    ind = d.indicators(u, prm)
    for k in ("nc2", "res2", "r2", "df2", "dfstar2", "rstar2", "amin", "resstar2"):
        assert np.abs(ind[k] - ind_ref[k]).max() <= SOL_TOL * np.abs(ind_ref[k]).max(), k
    assert abs(d.estimate(u, "eta_NC_OS2014", prm) - np.sqrt(ind_ref["nc2"].sum())) <= SOL_TOL
    assert abs(d.estimate(u, "eta_DF_OS2014", prm) - np.sqrt(ind_ref["df2"].sum())) <= SOL_TOL * np.sqrt(ind_ref["df2"].sum())


@pytest.mark.parametrize("nx,ny,parts", [(16, 16, (1, 1)), (24, 16, (4, 2)), (10, 7, (3, 2)), (64, 64, (8, 8))])
def test_cube_provider_on_the_device_equals_the_flat_array_path(gpu, nx, ny, parts):
    """hdd_mesh_create_cube (Stuff::Grid::Providers::Cube: three vectors, tables written on the device) against
    hdd_mesh_create from the host arrays of the same grid: identical pattern, bit-identical entries, same solution"""
    ll, ur = (-1.0, 0.0), (1.0, 2.0 * ny / nx)
    p = grids.CubeProvider(nx, ny, ll, ur, parts)
    g = grids.cube(nx, ny, ll, ur, parts)
    da, db = hdd.BlockSWIPDG(p, problems.ESV2007()), hdd.BlockSWIPDG(g, problems.ESV2007())
    da.init()
    db.init()
    (rpa, cola), (rpb, colb) = da.pattern(), db.pattern()
    assert np.array_equal(rpa, rpb) and np.array_equal(cola, colb)
    assert np.array_equal(da.system_matrix().affine_part(), db.system_matrix().affine_part())
    assert np.array_equal(da.rhs().affine_part(), db.rhs().affine_part())
    assert np.array_equal(da.subdomain_offsets(), db.subdomain_offsets())
    for ss in range(da.num_subdomains()):
        assert da.neighbouring_subdomains(ss) == db.neighbouring_subdomains(ss)
    opts = {"type": "cg.mg" if min(nx, ny) >= 16 else "cg.blockdiagonal", "precision": 1e-12, "max_iter": 5000}
    ua, ub = da.solve(opts), db.solve(opts)
    assert rel(ua, ub) <= 1e-12


@pytest.mark.parametrize("s,parts", [(4, (1, 1)), (8, (4, 4)), (16, (8, 8)), (24, (2, 3))])
def test_cg_mg_on_the_alu_ladder(gpu, s, parts):
    """cg.mg on lattice-structured simplex grids (BASELINE configs 1, 3, 4): conforming P1 auxiliary space on the vertex
    lattice, one hierarchy.  Against the direct solve, iteration counts flat in h (scipy prototype: 24-25, 28 for OS2014 at
    mu = 0.1), for ESV2007 and for the parametric OS2014 operator."""
    g = grids.simplex(s, partitions=parts)
    d = hdd.BlockSWIPDG(g, problems.ESV2007())
    d.init()
    m, rp, col, A, b = oracle_system(g, o.const(1.0), o.esv2007_force())
    u_ref = direct_solve(rp, col, A, b)
    u, info = d.solve({"type": "cg.mg", "precision": 1e-13, "max_iter": 500}, return_info=True)
    assert info["converged"] and rel(u, u_ref) <= SOL_TOL
    assert info["iterations"] <= 40, info["iterations"]
    _, ib = d.solve({"type": "cg.blockdiagonal", "precision": 1e-13, "max_iter": 50000}, return_info=True)
    assert s < 8 or info["iterations"] < ib["iterations"] / 2
    dp = hdd.BlockSWIPDG(g, problems.OS2014ParametricESV2007())
    dp.init()
    for mu in (0.1, 1.0):
        A_mu = o.assemble_lhs(m, o.os2014_factor(mu), None, rp, col)
        um, im = dp.solve({"type": "cg.mg", "precision": 1e-13, "max_iter": 500}, mu=mu, return_info=True)
        assert rel(um, direct_solve(rp, col, A_mu, b)) <= SOL_TOL and im["iterations"] <= 45, (mu, im["iterations"])
    # goldens of the ladder through the multigrid solve: eta_ESV2007 on 128 / 512 triangles
    if s in (4, 8) and parts == (1, 1):
        eta = d.estimate(u, "eta_ESV2007")
        assert abs(eta - golden("linearelliptic-swipdg-expectations_esv2007_2daluconform", "eta_ESV2007")[0 if s == 4 else 1]) < 0.006 * eta
