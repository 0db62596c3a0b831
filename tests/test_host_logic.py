"""CPU-only tests: the C-ABI library loads and exports every declared symbol, host-side logic (grid providers,
expression compiler, partition plan, Python mirror of the reference API) behaves - no compute calls without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import dune_hdd_b200 as hdd
from dune_hdd_b200 import capi, grids, parallel, problems
from oracle import oracle as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


HEADERS = {"hdd_b200.h": capi.SYMBOLS, "hdd_b200_testing.h": capi.TESTING_SYMBOLS}


def test_library_exports_every_symbol_the_header_declares():
    L = capi.lib()
    for name, symbols in HEADERS.items():
        header = open(os.path.join(ROOT, "include", name)).read()
        declared = set(re.findall(r"\b(hdd_[a-z0-9_]+)\s*\(", header))
        declared -= {"hdd_status"}
        assert declared == set(symbols), (name, declared ^ set(symbols))
        for sym in symbols:
            assert hasattr(L, sym), sym
    assert b"sm_100a" in L.hdd_version()


def test_header_is_plain_c_and_matches_the_definitions(tmp_path):
    """include/hdd_b200.h is the drop-in boundary: it has to compile as C99 (cgo / JNI / ctypes generators read it) and
    as C++ against the definitions - the csrc files include it, so a drifted prototype would already fail the build;
    here the C side is checked.  The same for include/hdd_b200_testing.h, the entry points of the tests."""
    import subprocess
    for name in HEADERS:
        header = os.path.join(ROOT, "include", name)
        subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-fsyntax-only", "-x", "c", header])
    src = tmp_path / "use.c"
    src.write_text('#include "hdd_b200_testing.h"\n'
                   'int main(void) { double c; return hdd_version() == 0 || hdd_fast_cos(&c, 0, &c) != HDD_OK; }\n')
    libdir = os.path.join(ROOT, "dune_hdd_b200")
    capi.lib()
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), str(src), "-L" + libdir,
                           "-lhdd_b200", "-Wl,-rpath," + libdir, "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64",
                           "-o", str(tmp_path / "use")])
    assert subprocess.run([str(tmp_path / "use")]).returncode == 0


def test_no_cpu_fallback_without_a_device():
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    g = grids.simplex(2)
    with pytest.raises(hdd.discretizations.device_error):
        hdd.SWIPDG(g, problems.ESV2007())


def _tri_set(xy, cv):
    pts = np.round(xy[cv] * 4096).astype(np.int64)
    return {tuple(sorted(map(tuple, t))) for t in pts}


@pytest.mark.parametrize("level", [0, 1, 2])
def test_simplex_provider_equals_recursive_bisection(level):
    """the closed-form union-jack generator produces exactly the triangles of ALU-style longest-edge bisection"""
    g = grids.simplex(4 * 2 ** level)
    m = o.mesh_bisect(4, -1.0, 1.0, 2 + 2 * level)
    assert g.n_cells == m.nc == 128 * 4 ** level and g.n_verts == m.nv
    assert _tri_set(g.xy, g.cell_verts) == _tri_set(m.xy, m.cv)


@pytest.mark.parametrize("maker,n", [(grids.simplex, 4), (grids.cube, 8), (grids.simplex, 1), (grids.cube, 1)])
@pytest.mark.parametrize("parts", [(1, 1), (2, 2), (4, 4), (8, 8)])
def test_grid_neighbours_orientation_and_subdomains(maker, n, parts):
    if n == 1 and parts != (1, 1):
        pytest.skip("partition finer than the grid")
    g = maker(n, partitions=parts)
    nl = g.n_loc
    fv = [(0, 1), (0, 2), (1, 2)] if g.kind == 0 else [(0, 2), (1, 3), (0, 1), (2, 3)]
    for c in range(g.n_cells):
        for f in range(nl):
            nb = g.cell_neigh[c, f]
            edge = {g.cell_verts[c, fv[f][0]], g.cell_verts[c, fv[f][1]]}
            if nb >= 0:
                assert c in g.cell_neigh[nb]  # symmetric
                assert edge <= set(g.cell_verts[nb])  # shares exactly this edge
            else:
                p = g.xy[list(edge)]
                assert np.any(np.all(np.abs(np.abs(p) - 1.0) < 1e-14, axis=0))  # both ends on the same domain side
    if g.kind == 0:
        a, b, c_ = (g.xy[g.cell_verts[:, k]] for k in range(3))
        det = (b[:, 0] - a[:, 0]) * (c_[:, 1] - a[:, 1]) - (c_[:, 0] - a[:, 0]) * (b[:, 1] - a[:, 1])
        assert np.all(det > 0)
    sub = g.cell_subdomain
    assert np.all(np.diff(sub) >= 0) and sub[0] == 0  # subdomain-major numbering
    assert g.n_subdomains == parts[0] * parts[1]
    cen = g.centers()
    sx = np.clip(((cen[:, 0] + 1) / 2 * parts[0]).astype(int), 0, parts[0] - 1)
    sy = np.clip(((cen[:, 1] + 1) / 2 * parts[1]).astype(int), 0, parts[1] - 1)
    if n > 1:
        assert np.array_equal(sub, sy * parts[0] + sx)


def test_cube_provider_matches_oracle_numbering():
    g = grids.cube(5, 3, (0.0, 0.0), (5.0, 1.0))
    m = o.mesh_cube(5, 3, 0.0, 5.0, 0.0, 1.0)
    assert np.array_equal(g.cell_verts, m.cv) and np.array_equal(g.cell_neigh, m.nb) and np.allclose(g.xy, m.xy)


def _eval(expr, var, values):
    out = C.c_double()
    v = np.asarray(values, dtype=np.float64)
    capi.check(capi.lib().hdd_expression_evaluate(expr.encode(), var.encode(), capi.ptr(v), len(v), C.byref(out)))
    return out.value


def test_expression_compiler():
    x = [0.3, -0.7]
    assert _eval("1+0.75*(sin(4*pi*(x[0]+0.5*x[1])))", "x", x) == pytest.approx(1 + 0.75 * np.sin(4 * np.pi * (0.3 - 0.35)), abs=1e-15)
    f = o.esv2007_force()
    assert _eval(problems.ESV2007_FORCE, "x", x) == pytest.approx(o.lib().or_fn_eval(C.byref(f), 0, C.c_double(0.3), C.c_double(-0.7)), rel=1e-15)
    assert _eval("mu", "mu", [0.1]) == 0.1 and _eval("-1.0*mu", "mu", [0.5]) == -0.5
    assert _eval("(mu)*(-1.0*mu)", "mu", [2.0]) == -4.0  # product coefficients of discretizations/swipdg.hh:319-321
    assert _eval("2^3^2", "x", x) == 512.0 and _eval("-2^2", "x", x) == -4.0 and _eval("1-2-3", "x", x) == -4.0
    assert _eval("pow(x[0],2)+sqrt(abs(x[1]))+exp(0)+min(1,2)*max(3,4)", "x", x) == pytest.approx(0.09 + np.sqrt(0.7) + 1 + 4)
    for bad in ("cos(x[0]", "1+", "foo(1)", "x[7]", "1 2", ""):
        with pytest.raises(capi.HddError) as e:
            _eval(bad, "x", x)
        assert e.value.status == capi.HDD_ERR_WRONG_INPUT


def test_problem_and_api_mirror():
    p = problems.OS2014ParametricESV2007()
    assert p.parametric() and p.parameter_type() == {"mu": 1}
    assert p.diffusion_factor.num_components() == 1 and p.diffusion_factor.coefficients == ["mu"]
    assert not problems.ESV2007().parametric()
    c = p.to_c()
    assert c.diffusion_factor.n_components == 1 and c.parameter_size == 1
    assert c.diffusion_factor.coefficients[0] == b"mu"
    g = grids.cube(100, 20, (0, 0), (5, 1))
    s = problems.Spe10Model1(g)
    k = s.diffusion_tensor.reshape(-1, 4)
    assert k[:, 0].min() >= problems.SPE10_MIN and k[:, 0].max() <= problems.SPE10_MAX and np.all(k[:, 1] == 0)
    f = s.force.affine.cell_values
    assert set(np.unique(f)) == {-1000.0, 0.0, 2000.0} and (f == 2000).sum() == 9 and (f == -1000).sum() == 18
    assert hdd.estimators.ESV2007_TYPES[4] == "eta_ESV2007" and "eta_OS2014_*" in hdd.estimators.OS2014_TYPES
    tc = hdd.testcases.ESV2007Multiscale((8, 8))
    assert tc.partitioning() == "[8 8 1]" and tc.level_grid(0).n_cells == 128 and tc.reference_grid().n_cells == 32768


@pytest.mark.parametrize("maker,n,world", [(grids.simplex, 8, 2), (grids.simplex, 8, 4), (grids.cube, 16, 3), (grids.cube, 16, 8)])
def test_partition_plan_is_consistent_between_ranks(maker, n, world):
    g = maker(n, partitions=(8, 8))
    off = parallel.rank_cell_offsets(g, world)
    assert off[0] == 0 and off[-1] == g.n_cells
    plans = [parallel.partition_plan(g, world, r) for r in range(world)]
    owner = np.searchsorted(off, np.arange(g.n_cells), side="right") - 1
    # vertex adjacency, independently with numpy
    v2c = [[] for _ in range(g.n_verts)]
    for c in range(g.n_cells):
        for v in g.cell_verts[c]:
            v2c[v].append(c)
    for r in range(world):
        halo, send = plans[r]
        own = set(range(off[r], off[r + 1]))
        expect = set()
        for c in own:
            for v in g.cell_verts[c]:
                expect.update(v2c[v])
        expect -= own
        assert list(halo) == sorted(expect)
        face_nb = set(g.cell_neigh[off[r]:off[r + 1]].ravel()) - own - {-1}
        assert face_nb <= set(halo)  # everything the SpMV needs is in the halo
        for peer, cells in send.items():
            peer_halo = plans[peer][0]
            assert np.array_equal(cells, peer_halo[owner[peer_halo] == r])  # send list == the peer's receive range


def test_pinned_allocation_falls_back_without_a_device():
    """hdd_host_alloc needs a CUDA context; on a CPU-only box the helper hands out ordinary memory instead"""
    from dune_hdd_b200 import capi
    a = capi.pinned_empty((5, 3), np.float64)
    a[:] = 1.5
    assert a.shape == (5, 3) and a.dtype == np.float64 and float(a.sum()) == 22.5
    g = grids.cube(4, pinned=True)
    g2 = grids.cube(4)
    assert np.array_equal(g.xy, g2.xy) and np.array_equal(g.cell_verts, g2.cell_verts) and np.array_equal(g.cell_neigh, g2.cell_neigh)


def test_golden_fixture_is_complete_and_cites_its_source():
    """tests/golden/reference_expectations.json carries the four reproducible expectation files with line numbers"""
    import json
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_expectations.json")
    with open(path) as f:
        d = json.load(f)
    stems = [k for k in d if not k.startswith("_")]
    assert sorted(stems) == sorted(["linearelliptic-swipdg-expectations_esv2007_2daluconform",
                                    "linearelliptic-swipdg-expectations_esv2007_2dsgrid",
                                    "linearelliptic-block-swipdg-expectations_esv2007_2daluconform",
                                    "linearelliptic-block-swipdg-expectations_os2014_2daluconform"])
    alu = d["linearelliptic-swipdg-expectations_esv2007_2daluconform"]["-"]["-"]
    assert alu["eta_ESV2007"]["values"] == [4.49e-01, 2.07e-01, 9.91e-02, 4.85e-02] and alu["eta_ESV2007"]["line"] > 0
    blk = d["linearelliptic-block-swipdg-expectations_esv2007_2daluconform"]
    assert sorted(blk) == ["[1 1 1]", "[2 2 1]", "[4 4 1]", "[8 8 1]"]


def test_father_search_finds_the_containing_coarse_cell():
    """hdd_grid_fathers (host): every fine centre lies strictly inside its father, every father has the same number of
    children on the nested ladders, the oracle's independent k-d tree search agrees, foreign domains are refused"""
    from dune_hdd_b200 import capi, grids
    from oracle import oracle as o
    from tests.helpers import oracle_mesh
    for make, nc, nf in ((grids.simplex, 2, 8), (grids.cube, 5, 20)):
        c, f = make(nc, partitions=(1, 1)), make(nf, partitions=(2, 2))
        fa = grids.fathers(c, f)
        assert np.array_equal(fa, o.fathers(oracle_mesh(c), oracle_mesh(f)))
        assert set(np.bincount(fa, minlength=c.n_cells)) == {16}
        inside = np.empty(f.n_cells, bool)
        cen = f.centers()
        for k in range(f.n_cells):
            v = c.xy[c.cell_verts[fa[k]]]
            if c.kind == grids.SIMPLEX2D:
                lam = np.linalg.solve(np.array([v[1] - v[0], v[2] - v[0]]).T, cen[k] - v[0])
                inside[k] = min(lam[0], lam[1], 1 - lam.sum()) > 1e-9
            else:
                inside[k] = ((cen[k] > v.min(0)) & (cen[k] < v.max(0))).all()
        assert inside.all()
    with pytest.raises(capi.HddError):
        grids.fathers(grids.cube(4, lower_left=(0.0, 0.0)), grids.cube(8))


@pytest.mark.parametrize("nx,ny,parts", [(8, 8, (1, 1)), (16, 12, (4, 3)), (10, 7, (3, 2)), (64, 64, (8, 8)), (5, 9, (5, 3))])
def test_cube_provider_describes_the_same_partition_as_the_flat_arrays(nx, ny, parts):
    """grids.CubeProvider (three vectors + partition, hdd_mesh_create_cube) against grids.cube (flat host arrays)"""
    from dune_hdd_b200 import grids
    p = grids.CubeProvider(nx, ny, partitions=parts)
    g = grids.cube(nx, ny, partitions=parts)
    assert (p.n_cells, p.n_verts, p.n_dofs, p.n_subdomains) == (g.n_cells, g.n_verts, g.n_dofs, g.n_subdomains)
    assert np.array_equal(p.subdomain_cell_offsets(), g.subdomain_cell_offsets())
    m = p.materialize()
    assert np.array_equal(m.cell_verts, g.cell_verts) and np.array_equal(m.cell_subdomain, g.cell_subdomain)


def test_fast_cos_is_within_two_ulp_of_cos():
    """csrc/expr.hpp fast_cos (the estimator kernel's branch-free cosine), run on the host through hdd_fast_cos: within two
    units in the last place of 1.0 of numpy's cos over its whole range of validity, exact at the special points"""
    import ctypes as C
    L = capi.lib()
    rng = np.random.default_rng(0)
    for lim in (1.0, 10.0, 1.0e3, 9.9e4):
        x = np.concatenate([rng.uniform(-lim, lim, 100000), [0.0, np.pi / 2, -np.pi / 2, np.pi, 1e-300, np.pi / 4, 1e-9]])
        out = np.empty_like(x)
        capi.check(L.hdd_fast_cos(capi.ptr(x), C.c_int64(x.size), capi.ptr(out)))
        assert np.abs(out - np.cos(x)).max() <= 2.0 * np.finfo(float).eps
    one = np.zeros(1)
    capi.check(L.hdd_fast_cos(capi.ptr(np.zeros(1)), C.c_int64(1), capi.ptr(one)))
    assert one[0] == 1.0  # a missing second factor of a TrigProduct is cos(0)


def test_trig_product_recognition_and_values():
    """csrc/expr.hpp as_trig_product through hdd_trig_product: products of at most two sines / cosines of affine arguments
    are recognised (sines become cosines with a phase shift), everything else is left to the general evaluation; the
    recognised form, evaluated with fast_cos, reproduces the expression"""
    L = capi.lib()
    rng = np.random.default_rng(3)
    x, y = rng.uniform(-2, 2, 200), rng.uniform(-2, 2, 200)
    pi = np.pi
    cases = {
        problems.ESV2007_FORCE: 0.5 * pi * pi * np.cos(0.5 * pi * x) * np.cos(0.5 * pi * y),
        "cos(0.5*pi*x[0])*cos(0.5*pi*x[1])": np.cos(0.5 * pi * x) * np.cos(0.5 * pi * y),
        "-0.5*pi*sin(0.5*pi*x[0])*cos(0.5*pi*x[1])": -0.5 * pi * np.sin(0.5 * pi * x) * np.cos(0.5 * pi * y),
        "sin(2*x[0]+1)*sin(x[1]-0.25)": np.sin(2 * x + 1) * np.sin(y - 0.25),
        "-3*sin(x[0]-x[1])": -3 * np.sin(x - y),
        "cos(4*pi*(x[0]+0.5*x[1]))": np.cos(4 * pi * (x + 0.5 * y)),
    }
    for expr, want in cases.items():
        out, valid = np.zeros(7), C.c_int()
        capi.check(L.hdd_trig_product(expr.encode(), capi.ptr(out), C.byref(valid)))
        assert valid.value == 1, expr
        c, a0, b0, d0, a1, b1, d1 = out
        args = np.concatenate([a0 * x + b0 * y + d0, a1 * x + b1 * y + d1])
        cosv = np.empty_like(args)
        capi.check(L.hdd_fast_cos(capi.ptr(args), C.c_int64(args.size), capi.ptr(cosv)))
        got = c * cosv[:x.size] * cosv[x.size:]
        assert np.abs(got - want).max() <= 1e-14 * max(1.0, np.abs(want).max()), expr
    for expr in ("x[0]*cos(x[1])", "cos(x[0])+1", "exp(x[0])*cos(x[1])", "cos(x[0])*cos(x[1])*cos(x[0]+x[1])",
                 "1+0.75*(sin(4*pi*(x[0]+0.5*x[1])))", "abs(x[0])"):
        out, valid = np.zeros(7), C.c_int()
        capi.check(L.hdd_trig_product(expr.encode(), capi.ptr(out), C.byref(valid)))
        assert valid.value == 0, expr
