"""The preconditioners of the CG solver types, operator by operator, against the float64 restatement in
tests/mg_reference.py: the level operators of every multigrid hierarchy (hdd_mg_level_operator), the V-cycle results on
the finest vertex level and z = M^-1 r of one application through hdd_solve's own set-up (hdd_precondition), the r.z of
the fused reduction, block-Jacobi backward errors, and the symmetry and positivity of M^-1.  A wrong preconditioner does
not make CG converge to a wrong answer, only more slowly; these tests say which number changed.

Bars (max-norm, per quantity): level operators per row 1e-12 |S_ref[4]|; vertex vectors 1e-11 max|v_ref| per hierarchy;
z 1e-11 max|z_ref|; block Jacobi |D_c z_c - r_c| <= 1e-13 (|D_c| |z_c| + |r_c|) per cell; rz 1e-12 |r| |z_ref|; symmetry
|s.M^-1 r - r.M^-1 s| <= 1e-12 sqrt((r.M^-1 r)(s.M^-1 s))."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import dune_hdd_b200 as hdd
from dune_hdd_b200 import capi, grids, problems
from dune_hdd_b200.discretizations import _mu_array
from oracle import oracle as o
from tests import mg_reference as ref
from tests.helpers import oracle_mesh, rel

pytestmark = pytest.mark.gpu

OP_TOL, VERTEX_TOL, Z_TOL, BLOCK_TOL, RZ_TOL, SYM_TOL = 1e-12, 1e-11, 1e-11, 1e-13, 1e-12, 1e-12


# ---- the hooks --------------------------------------------------------------------------------------------------------
def precondition(d, typ, r, mu=None, n_vertex=0):
    """(z, rz, vertex results or None) of one application of the preconditioner of `typ`"""
    mu_a, ms = _mu_array(mu)
    r = np.ascontiguousarray(r, np.float64)
    z, rz = np.empty_like(r), C.c_double()
    v = np.empty(n_vertex) if n_vertex else None
    capi.check(capi.lib().hdd_precondition(d._h, typ.encode(), capi.ptr(mu_a), ms, capi.ptr(r), capi.ptr(z), C.byref(rz),
                                           capi.ptr(v)))
    return z, rz.value, v


def level_operator(d, level, hier, with_values=True):
    nx, ny = C.c_int(), C.c_int()
    capi.check(capi.lib().hdd_mg_level_operator(d._h, level, hier, C.byref(nx), C.byref(ny), None))
    if not with_values:
        return nx.value, ny.value, None
    S = np.empty((9, (nx.value + 1) * (ny.value + 1)))
    capi.check(capi.lib().hdd_mg_level_operator(d._h, level, hier, None, None, capi.ptr(S)))
    return nx.value, ny.value, S


def device_shapes(d):
    shapes = []
    while True:
        try:
            shapes.append(level_operator(d, len(shapes), 0, with_values=False)[:2])
        except capi.HddError as e:
            assert e.status == capi.HDD_ERR_WRONG_INPUT
            return shapes


# ---- the comparisons ----------------------------------------------------------------------------------------------------
def _max_rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(b).max(), 1e-300)


def check_operators(d, mg, what=""):
    """level shapes, and every stored level operator of every hierarchy, per row against the diagonal"""
    shapes = device_shapes(d)
    assert shapes == [(L["nx"], L["ny"]) for L in mg.levels[0]], (what, shapes)
    for h, levels in enumerate(mg.levels):
        for l, S_ref in enumerate(mg.stencils(h)):
            if l == 0 and h == 1 and mg.kind == "q1":
                with pytest.raises(capi.HddError):  # C A_c C is not stored
                    level_operator(d, 0, 1)
                continue
            _, _, S = level_operator(d, l, h)
            err = (np.abs(S - S_ref) / np.abs(S_ref[4])).max()
            assert err <= OP_TOL, (what, "hierarchy", h, "level", l, err)
    with pytest.raises(capi.HddError):
        level_operator(d, len(shapes), 0)
    with pytest.raises(capi.HddError):
        level_operator(d, 0, len(mg.levels))


def check_vertex(mg, v, r, what=""):
    """per hierarchy to 1e-11 max|v_ref|, or to u max|V_h(|Pi_h|^T |r|)| if that is larger: the restriction Pi_h^T r sums
    up to nine products in another order on the device, and when it cancels (the assembled rhs against the hourglass
    weights: Pi_h^T r ~ 1e-8 |Pi_h|^T |r|) that rounding, carried through the linear V-cycle, is all that can agree"""
    for h, (v_ref, scale) in enumerate(zip(mg.vertex(r), mg.vertex_scale(r))):
        err = np.abs(v[h] - v_ref).max()
        assert err <= max(VERTEX_TOL * np.abs(v_ref).max(), 2.0 ** -52 * scale), (what, "hierarchy", h, err, scale)


def check_block_jacobi(D, z, r, what=""):
    nl = D.shape[1]
    zc, rc = z.reshape(-1, nl), r.reshape(-1, nl)
    res = np.abs(np.einsum("cij,cj->ci", D, zc) - rc).max(1)
    scale = np.abs(D).sum(2).max(1) * np.abs(zc).max(1) + np.abs(rc).max(1)
    worst = np.where(scale > 0.0, res / np.where(scale > 0.0, scale, 1.0), res).max()  # r_c = 0 must give z_c = 0
    assert worst <= BLOCK_TOL, (what, worst)


def check_symmetry(apply, r, s, what=""):
    zr, zs = apply(r), apply(s)
    rr, ss = r @ zr, s @ zs
    assert rr > 0.0 and ss > 0.0, (what, rr, ss)
    assert abs(s @ zr - r @ zs) <= SYM_TOL * np.sqrt(rr * ss), (what, s @ zr, r @ zs)


def right_hand_sides(g, nl, b):
    """a seeded normal vector, the assembled rhs, a unit vector on the first DoF of a cell at vertex 0 (a corner)"""
    e = np.zeros(g.n_cells * nl)
    e[nl * int(np.flatnonzero((g.cell_verts == 0).any(1))[0])] = 1.0
    return {"normal": np.random.default_rng(7).standard_normal(g.n_cells * nl), "rhs": b, "corner": e}


def check_case(d, g, kind, typ, A, b, nx, ny, mu=None, what=""):
    """Tier A: everything against a reference built from the oracle-assembled A"""
    A = sp.csr_matrix(A)
    nl = A.shape[0] // g.n_cells
    D, _ = ref.block_inverses(A, nl)
    mg = ref.Multigrid(kind, g.cell_verts, nx, ny, A=A) if kind else None
    n_vertex = len(mg.levels) * (nx + 1) * (ny + 1) if mg else 0
    rhs = right_hand_sides(g, nl, b)
    for name, r in rhs.items():
        tag = (what, typ, mu, name)
        zb, rzb, _ = precondition(d, "cg.blockdiagonal", r, mu)
        check_block_jacobi(D, zb, r, tag)
        if mg is None:
            continue
        z, rz, v = precondition(d, typ, r, mu, n_vertex)
        v = v.reshape(len(mg.levels), -1)
        if name == "normal":
            check_operators(d, mg, tag)
        check_vertex(mg, v, r, tag)
        z_ref = mg(r)
        assert _max_rel(z, z_ref) <= Z_TOL, (tag, _max_rel(z, z_ref))
        assert _max_rel(z - zb, mg.correction(r)) <= Z_TOL, tag
        assert abs(rz - r @ z_ref) <= RZ_TOL * np.linalg.norm(r) * np.linalg.norm(z_ref), (tag, rz, r @ z_ref)
    check_symmetry(lambda x: precondition(d, typ, x, mu)[0], rhs["normal"], rhs["rhs"], (what, typ, mu))


# ---- Tier A: small grids, reference from the oracle matrix --------------------------------------------------------------
ESV = problems.ESV2007
FACTOR_XY = o.fn([(2.0, o.FN_ONE), (1.0, o.FN_XY)], 2)  # "2+x[0]*x[1]"


def _cube(nx, ny=None, ll=(-1.0, -1.0), ur=(1.0, 1.0), parts=(1, 1)):
    return grids.cube(nx, ny, ll, ur, partitions=parts)


def _mixed_boundary(g):
    bt = np.ones((g.n_cells, g.n_loc), np.uint8)
    bt[(g.centers()[:, 0] < 0)[:, None] & (g.cell_neigh < 0)] = 2
    return bt


def _parametric():
    fac = problems.AffinelyDecomposable(problems.Constant(1.0), [problems.Expression("2+x[0]*x[1]", 2)], ["mu"])
    return problems.Problem(fac, ESV().force, parameter_name="mu", parameter_size=1)


def build_case(name):
    """(discretization, grid, reference kind, solver type, [(mu, A(mu))], assembled rhs, nx, ny) of a named case"""
    kind_s, spec = name.split(":")
    polorder = 2 if kind_s == "q2" else 1
    args = dict(a.split("=") for a in spec.split(",")[1:])
    size = spec.split(",")[0]
    bt, tensor, factors, prob = None, None, None, None
    if kind_s == "p1":
        s = int(size)
        g = grids.simplex(s, partitions=tuple(map(int, args.get("parts", "1x1").split("x"))))
        nx = ny = 2 * s
    else:
        nx, ny = map(int, size.split("x"))
        ll, ur = (-1.0, -1.0), (1.0, 1.0)
        if args.get("domain") == "rect":
            ll, ur = (-1.0, 0.0), (2.0, 1.0)
        elif args.get("domain") == "square-cells":
            ll, ur = (0.0, 0.0), (nx / 2.0 if ny == 2 else 1.0, ny / 2.0 if nx == 2 else 1.0)
        elif args.get("domain") == "spe10":
            ll, ur = (0.0, 0.0), (5.0, 1.0)
        g = _cube(nx, ny, ll, ur, tuple(map(int, args.get("parts", "1x1").split("x"))))
    pb = args.get("problem", "esv")
    if pb == "spe10":
        prob = problems.Spe10Model1(g)
        tensor = prob.diffusion_tensor
    elif pb == "mixed":
        prob, bt = ESV(), _mixed_boundary(g)
    elif pb == "param":
        prob = _parametric()
        factors = [(mu, [(o.const(1.0), 1.0), (FACTOR_XY, mu)]) for mu in (0.1, 10.0)]
    elif pb == "os2014":
        prob = problems.OS2014ParametricESV2007()
        factors = [(mu, [(o.os2014_factor(mu), 1.0)]) for mu in (0.1, 1.0)]
    elif pb == "expr":
        prob = problems.Problem(problems.AffinelyDecomposable(problems.Expression("2+x[0]*x[1]", 2, "diffusion_factor")),
                                ESV().force)
        factors = [(None, [(FACTOR_XY, 1.0)])]
    else:
        prob = ESV()
    factors = factors or [(None, [(o.const(1.0), 1.0)])]
    d = hdd.SWIPDG(g, prob, boundary_info=bt, polorder=polorder)
    d.init()
    m = oracle_mesh(g).with_polorder(polorder)
    rp, col = o.pattern(m)
    dirichlet = None if bt is None else (bt == 1)
    mats = []
    for mu, parts in factors:
        A = sum(c * o.to_scipy(rp, col, o.assemble_lhs(m, f, tensor, rp, col, bnd_dirichlet=dirichlet)) for f, c in parts)
        mats.append((mu, A.tocsr()))
    b = o.assemble_rhs(m, o.esv2007_force())
    kind = {"q1": "q1", "p1": "p1", "q2": "q2"}[kind_s]
    typ = "cg.mg2" if kind == "q2" else "cg.mg"
    return d, g, kind, typ, mats, b, nx, ny


MG_CASES = [
    # cg.mg on Q1: one level (the dense inverse twists the plain arrays), one level at the 400-vertex cap, coarsest at the
    # cap, subdomain-major numbering, hx != hy and non-square, odd sizes, the Gauss-Jordan coarsest (band > 200 KB) and its
    # transpose (band 3), SPE10, mixed boundary, a parametric operator rebuilt in place
    "q1:3x3", "q1:19x19", "q1:38x38", "q1:64x64,parts=4x4", "q1:24x16,domain=rect,parts=4x2", "q1:10x7",
    "q1:398x2,domain=square-cells", "q1:2x398,domain=square-cells", "q1:100x20,domain=spe10,problem=spe10",
    "q1:32x32,problem=mixed", "q1:32x32,problem=param",
    # cg.mg2 on Q2
    "q2:3x3", "q2:19x19", "q2:38x38", "q2:48x48,parts=4x4", "q2:24x16,parts=4x2",
    "q2:398x2,domain=square-cells", "q2:100x20,domain=spe10,problem=spe10", "q2:16x16,problem=mixed",
    "q2:32x32,problem=param", "q2:16x16,problem=expr",
    # cg.mg on the P1 lattice: one level, two, coarsest at the cap, partitioned, OS2014
    "p1:4", "p1:16", "p1:19", "p1:24,parts=2x3", "p1:16,problem=os2014",
]


def run_case(name):
    d, g, kind, typ, mats, b, nx, ny = build_case(name)
    for mu, A in mats:
        check_case(d, g, kind, typ, A, b, nx, ny, mu, name)


@pytest.mark.parametrize("name", MG_CASES)
def test_multigrid_preconditioner_matches_the_reference(gpu, name):
    run_case(name)


@pytest.mark.parametrize("kind,n,polorder", [("alu", 4, 1), ("sgrid", 8, 1), ("alu", 2, 2), ("sgrid", 4, 2),
                                             ("sgrid", 5, 2)])
def test_diagonal_and_block_diagonal_preconditioners(gpu, kind, n, polorder):
    """cg.diagonal: z = r / diag(A) (two roundings); cg.blockdiagonal (k_invert_diag_blocks, n_loc = 3, 4, 6, 9): per-cell
    backward error, and symmetry"""
    g = grids.simplex(n) if kind == "alu" else grids.cube(n)
    d = hdd.SWIPDG(g, ESV(), polorder=polorder)
    d.init()
    m = oracle_mesh(g).with_polorder(polorder)
    rp, col = o.pattern(m)
    A = o.to_scipy(rp, col, o.assemble_lhs(m, o.const(1.0), None, rp, col)).tocsr()
    diag = o.to_scipy(rp, col, d.system_matrix().affine_part()).diagonal()  # the device's own entries: z is two roundings
    nl = A.shape[0] // g.n_cells
    D, _ = ref.block_inverses(A, nl)
    for name, r in right_hand_sides(g, nl, o.assemble_rhs(m, o.esv2007_force())).items():
        z, rz, _ = precondition(d, "cg.diagonal", r)
        z_ref = r / diag
        assert np.all(np.abs(z - z_ref) <= 2.3e-16 * np.abs(z_ref)), name
        assert abs(rz - r @ z_ref) <= RZ_TOL * np.linalg.norm(r) * np.linalg.norm(z_ref), name
        zb, rzb, _ = precondition(d, "cg.blockdiagonal", r)
        check_block_jacobi(D, zb, r, name)
        assert abs(rzb - r @ zb) <= RZ_TOL * np.linalg.norm(r) * np.linalg.norm(zb), name
    rhs = right_hand_sides(g, nl, o.assemble_rhs(m, o.esv2007_force()))
    check_symmetry(lambda x: precondition(d, "cg.blockdiagonal", x)[0], rhs["normal"], rhs["rhs"])
    # the hook refuses what it cannot show
    with pytest.raises(capi.HddError):
        precondition(d, "cg.diagonal", rhs["normal"], n_vertex=4)


def test_precondition_leaves_the_solution_alone(gpu):
    g = grids.cube(16)
    d = hdd.SWIPDG(g, ESV())
    d.init()
    u1 = d.uncached_solve({"type": "cg.mg", "precision": 1e-12, "max_iter": 200})
    x_dev = C.POINTER(C.c_double)()
    r = np.random.default_rng(1).standard_normal(g.n_dofs)
    precondition(d, "cg.mg", r)
    capi.check(capi.lib().hdd_solution_dev(d._h, C.byref(x_dev)))
    x = np.empty(g.n_dofs)
    capi.check(capi.lib().hdd_copy_to_host(d._h, capi.ptr(x), x_dev, C.c_size_t(x.nbytes)))
    assert np.array_equal(x, u1)
    # the next solve (which replays the cached graph) is the same solve
    assert np.array_equal(d.uncached_solve({"type": "cg.mg", "precision": 1e-12, "max_iter": 200}), u1)


def test_cg_mg2_refuses_an_indefinite_hourglass_operator(gpu):
    """Q2 with hx = 2 hy: H^T A H has a negative eigenvalue (tests/mg_reference.py shows it on the oracle matrix), so the
    SWIPDG matrix itself is indefinite there and cg.mg2 refuses instead of running CG on it"""
    g = grids.cube(16, 16, (-1.0, 0.0), (2.0, 1.0))
    d = hdd.SWIPDG(g, ESV(), polorder=2)
    d.init()
    m = oracle_mesh(g).with_polorder(2)
    rp, col = o.pattern(m)
    mg = ref.Multigrid("q2", g.cell_verts, 16, 16, A=o.to_scipy(rp, col, o.assemble_lhs(m, o.const(1.0), None, rp, col)))
    assert np.linalg.eigvalsh(mg.levels[1][0]["A"].toarray()).min() < 0.0
    with pytest.raises(hdd.discretizations.requirements_not_met, match="not positive definite"):
        d.solve({"type": "cg.mg2", "precision": 1e-10, "max_iter": 100})


# ---- Gauss-Jordan forced: HDD_MG_COARSE_GJ=1 is read once per process ----------------------------------------------------
GJ_CASES = ["q1:19x19", "q1:38x38", "q2:38x38"]


def test_gauss_jordan_coarsest_inverse(gpu):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, HDD_MG_COARSE_GJ="1")
    p = subprocess.run([sys.executable, "-m", "tests.test_gpu_preconditioners"] + GJ_CASES, cwd=root, env=env,
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]


# ---- Tier B: large grids, level-0 operators from the device --------------------------------------------------------------
def _twist(S):
    C_ = S.copy()
    C_[1::2] *= -1.0  # C A C: the edge-neighbour entries (e odd) change sign
    return C_


@pytest.mark.parametrize("kind,n", [("q1", 576), ("q2", 576), ("p1", 208), ("q1", 2560)])
def test_multigrid_preconditioner_on_large_grids(gpu, kind, n):
    """the grid-stride loops of the prolongation kernels (> 303 104 owned cells) and, at 2560^2, the unfused up-sweep
    (k_mg_prolong_add + k_mg_post) on level 1 (1281^2 vertices)"""
    g = grids.simplex(n) if kind == "p1" else grids.cube(n)
    nx = ny = 2 * n if kind == "p1" else n
    d = hdd.SWIPDG(g, ESV(), polorder=2 if kind == "q2" else 1)
    d.init()
    typ = "cg.mg2" if kind == "q2" else "cg.mg"
    nl = {"q1": 4, "p1": 3, "q2": 9}[kind]
    r = np.random.default_rng(11).standard_normal(g.n_cells * nl)
    n_hier = 1 if kind == "p1" else 2
    z, rz, v = precondition(d, typ, r, n_vertex=n_hier * (nx + 1) * (ny + 1))
    S0 = level_operator(d, 0, 0)[2]
    level0 = [S0, _twist(S0)] if kind == "q1" else [S0] if kind == "p1" else [S0, level_operator(d, 0, 1)[2]]
    mg = ref.Multigrid(kind, g.cell_verts, nx, ny, level0=level0)
    assert device_shapes(d) == [(L["nx"], L["ny"]) for L in mg.levels[0]]
    for h in range(n_hier):
        for l, S_ref in enumerate(mg.stencils(h)[1:], start=1):
            err = (np.abs(level_operator(d, l, h)[2] - S_ref) / np.abs(S_ref[4])).max()
            assert err <= OP_TOL, (h, l, err)
    check_vertex(mg, v.reshape(n_hier, -1), r)
    zb = precondition(d, "cg.blockdiagonal", r)[0]
    corr = mg.correction(r)
    assert np.abs(z - zb - corr).max() <= Z_TOL * np.abs(z).max()
    assert abs(rz - r @ z) <= RZ_TOL * np.linalg.norm(r) * np.linalg.norm(z)
    s = np.random.default_rng(12).standard_normal(r.size)
    zs = precondition(d, typ, s)[0]
    assert r @ z > 0.0 and s @ zs > 0.0
    assert abs(s @ z - r @ zs) <= SYM_TOL * np.sqrt((r @ z) * (s @ zs))


# ---- iterates: the CG of the solver with the reference M^-1 ---------------------------------------------------------------
def _pcg(A, b, M, iters):
    x, r = np.zeros_like(b), b.copy()
    z = M(r)
    p, rz = z.copy(), r @ z
    for _ in range(iters):
        q = A @ p
        alpha = rz / (p @ q)
        x += alpha * p
        r -= alpha * q
        z = M(r)
        rz_new = r @ z
        p = z + (rz_new / rz) * p
        rz = rz_new
    return x


@pytest.mark.parametrize("name", ["q1:32x32", "p1:16", "q2:32x32"])
def test_cg_iterates_follow_the_reference_pcg(gpu, name):
    """max_iter 20, 3, 1, 12 on one handle: the first call launches directly, the later ones replay the cached
    two-iteration graph, and the done latch falls in the middle of a batch"""
    d, g, kind, typ, mats, b, nx, ny = build_case(name)
    (_, A), = mats
    mg = ref.Multigrid(kind, g.cell_verts, nx, ny, A=A)
    for maxit in (20, 3, 1, 12):
        with pytest.raises(hdd.discretizations.linear_solver_failed):
            d.uncached_solve({"type": typ, "precision": 1e-30, "max_iter": maxit})
        p = C.POINTER(C.c_double)()
        capi.check(capi.lib().hdd_solution_dev(d._h, C.byref(p)))
        x = np.empty(A.shape[0])
        capi.check(capi.lib().hdd_copy_to_host(d._h, capi.ptr(x), p, C.c_size_t(x.nbytes)))
        x_ref = _pcg(A, b, mg, maxit)
        assert rel(x, x_ref) <= 1e-10, (maxit, rel(x, x_ref))


if __name__ == "__main__":
    # the named Tier A cases in this process (tests/test_gpu_preconditioners.py runs it with HDD_MG_COARSE_GJ=1)
    for case in sys.argv[1:]:
        run_case(case)
        print("ok", case)
