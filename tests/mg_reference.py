"""The multigrid preconditioners of the solver types "cg.mg" and "cg.mg2" (dune_hdd_b200/csrc/multigrid.cu, DESIGN.md 6)
restated in float64 scipy from the comments of multigrid.cu, for the CPU prototypes (tests/test_mg_prototype.py,
tests/test_mg_q2_prototype.py) and the operator-by-operator GPU comparison (tests/test_gpu_preconditioners.py).

  Q1 on cubes ("cg.mg")       M^-1 r = D^-1 r + P V(P^T r) + P C V_C(C P^T r)
  P1 on lattice simplices      M^-1 r = D^-1 r + P V(P^T r)
  Q2 on cubes ("cg.mg2")      M^-1 r = D^-1 r + P V_P(P^T r) + H V_H(H^T r)

D: the n_loc x n_loc cell blocks of A.  P: the injection of the conforming Q1 / P1 vertex space (DG DoF (T, i) = value at
vertex i of T), for Q2 the bilinear interpolation of the Q1 vertex space at the nine nodes.  C: the checkerboard sign
(-1)^(ix+iy).  H: the Q2 hourglass family, cell c gets s[v0(c)] (2/3, -1/3, 2/3) x (2/3, -1/3, 2/3), v0(c) its lower-left
vertex.  Hierarchy h has the level-0 operator Pi_h^T A Pi_h, Pi in {P, PC} (Q1), {P} (P1), {P, H} (Q2); the rows of A_H
that no cell reaches (top vertex row, right vertex column) get the mean of the other rows' diagonal.  Every level-0
operator is a 9-point stencil on the (nx+1) x (ny+1) vertex lattice, numbered x-fastest.  V: one V(1,1)-cycle from a zero
guess - damped Jacobi (omega = 0.8), bilinear interpolation kron(I_y, I_x), its transpose as restriction, Galerkin coarse
operators, a dense inverse on the coarsest level.  The levels are halved while the level has more than `max_coarse`
vertices and both sizes are even and at least 2; a coarsest level still above `max_coarse` vertices is refused."""
import numpy as np
import scipy.sparse as sp

OMEGA = 0.8
MAX_COARSE = 400  # multigrid.cu kMaxCoarse
G1 = np.array([2.0 / 3.0, -1.0 / 3.0, 2.0 / 3.0])
HOURGLASS = np.outer(G1, G1).ravel()  # node a + 3 b


class CannotCoarsen(ValueError):
    pass


def level_shapes(nx, ny, max_coarse=MAX_COARSE):
    """the (nx, ny) of every vertex level, finest first, by the device's coarsening rule"""
    shapes = [(nx, ny)]
    while (nx + 1) * (ny + 1) > max_coarse and nx % 2 == 0 and ny % 2 == 0 and nx >= 2 and ny >= 2:
        nx, ny = nx // 2, ny // 2
        shapes.append((nx, ny))
    if (nx + 1) * (ny + 1) > max_coarse:
        raise CannotCoarsen("the %d x %d grid cannot be coarsened by halving down to at most %d vertices (stuck at %d x %d)"
                            % (shapes[0] + (max_coarse, nx, ny)))
    return shapes


def _interp1d(nc):
    rows, cols, vals = [], [], []
    for i in range(2 * nc + 1):
        if i % 2 == 0:
            rows.append(i); cols.append(i // 2); vals.append(1.0)
        else:
            rows += [i, i]; cols += [i // 2, i // 2 + 1]; vals += [0.5, 0.5]
    return sp.csr_matrix((vals, (rows, cols)), shape=(2 * nc + 1, nc + 1))


def interpolation(nxc, nyc):
    """bilinear interpolation from the (nxc+1) x (nyc+1) lattice to the (2 nxc + 1) x (2 nyc + 1) one (x fastest)"""
    return sp.kron(_interp1d(nyc), _interp1d(nxc)).tocsr()


def _offsets(nx, ny):
    nv = (nx + 1) * (ny + 1)
    ix, iy = np.arange(nv) % (nx + 1), np.arange(nv) // (nx + 1)
    return nv, ix, iy


def to_stencil(A, nx, ny):
    """the 9-point form S[e, v] = A[v, (ix+dx, iy+dy)], e = 3 (dy+1) + dx + 1 (0 outside the lattice); asserts that A has
    nothing at index distance 2 or more"""
    nv, ix, iy = _offsets(nx, ny)
    coo = sp.coo_matrix(A)
    dx, dy = ix[coo.col] - ix[coo.row], iy[coo.col] - iy[coo.row]
    far = (np.abs(dx) > 1) | (np.abs(dy) > 1)
    assert np.abs(coo.data[far]).max(initial=0.0) <= 1e-12 * np.abs(coo.data).max(), "not a 9-point stencil"
    S = np.zeros((9, nv))
    near = ~far
    np.add.at(S, (3 * (dy[near] + 1) + dx[near] + 1, coo.row[near]), coo.data[near])
    return S


def from_stencil(S, nx, ny):
    nv, ix, iy = _offsets(nx, ny)
    rows, cols, vals = [], [], []
    for e in range(9):
        dx, dy = e % 3 - 1, e // 3 - 1
        ok = (ix + dx >= 0) & (ix + dx <= nx) & (iy + dy >= 0) & (iy + dy <= ny)
        v = np.flatnonzero(ok)
        rows.append(v); cols.append(v + dx + dy * (nx + 1)); vals.append(S[e, v])
    return sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(nv, nv))


def checkerboard(nx, ny):
    _, ix, iy = _offsets(nx, ny)
    return np.where((ix + iy) % 2 == 1, -1.0, 1.0)


def hourglass_fill(S, nx, ny):
    """the empty rows of A_H (top vertex row, right vertex column) get the mean diagonal of the others (k_hourglass_fill)"""
    _, ix, iy = _offsets(nx, ny)
    inner = (ix < nx) & (iy < ny)
    S = S.copy()
    S[4, ~inner] = S[4, inner].sum() / (nx * ny)
    return S


def hierarchy(A0, nx, ny, max_coarse=MAX_COARSE):
    """the levels of one hierarchy: A (csr), nx, ny, dinv = omega / diagonal, P (to the next coarser level) and, on the
    coarsest, the dense inverse"""
    shapes = level_shapes(nx, ny, max_coarse)
    levels = [{"A": sp.csr_matrix(A0), "nx": nx, "ny": ny}]
    for nxc, nyc in shapes[1:]:
        Pm = interpolation(nxc, nyc)
        levels[-1]["P"] = Pm
        levels.append({"A": (Pm.T @ levels[-1]["A"] @ Pm).tocsr(), "nx": nxc, "ny": nyc})
    levels[-1]["inv"] = np.linalg.inv(levels[-1]["A"].toarray())
    for L in levels:
        L["dinv"] = OMEGA / L["A"].diagonal()
    return levels


def vcycle(levels, b, l=0):
    """one V(1,1)-cycle from a zero guess on level l"""
    L = levels[l]
    if "inv" in L:
        return L["inv"] @ b
    x = L["dinv"] * b
    x = x + L["P"] @ vcycle(levels, L["P"].T @ (b - L["A"] @ x), l + 1)
    return x + L["dinv"] * (b - L["A"] @ x)


def transfers(kind, cell_verts, n_verts):
    """the prolongations Pi_h of the hierarchies, DG DoFs x vertices: kind "q1" (P, PC), "p1" (P), "q2" (P, H)"""
    cv = np.asarray(cell_verts)
    nc = cv.shape[0]
    if kind in ("q1", "p1"):
        nl = cv.shape[1]
        P = sp.csr_matrix((np.ones(nl * nc), (np.arange(nl * nc), cv.reshape(-1))), shape=(nl * nc, n_verts))
        return [P] if kind == "p1" else [P, None]  # PC needs the lattice size: see Multigrid
    rows, cols, vals = [], [], []
    w = lambda i, a: 1.0 - a / 2.0 if i == 0 else a / 2.0  # noqa: E731
    for b in range(3):
        for a in range(3):
            for j in range(2):
                for i in range(2):
                    if w(i, a) * w(j, b):
                        rows.append(9 * np.arange(nc) + a + 3 * b); cols.append(cv[:, i + 2 * j])
                        vals.append(np.full(nc, w(i, a) * w(j, b)))
    P = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(9 * nc, n_verts))
    H = sp.csr_matrix((np.tile(HOURGLASS, nc), (np.arange(9 * nc), np.repeat(cv[:, 0], 9))), shape=(9 * nc, n_verts))
    return [P, H]


def block_inverses(A, nl):
    """np.linalg.inv of every n_loc x n_loc diagonal block: (n_cells, nl, nl)"""
    coo = sp.coo_matrix(A)
    keep = coo.row // nl == coo.col // nl
    D = np.zeros((A.shape[0] // nl, nl, nl))
    np.add.at(D, (coo.row[keep] // nl, coo.row[keep] % nl, coo.col[keep] % nl), coo.data[keep])
    return D, np.linalg.inv(D)


class Multigrid:
    """The preconditioner of one structured grid.  kind "q1" / "p1" / "q2"; nx, ny: the vertex lattice; A: the frozen
    system matrix (level-0 operators Pi_h^T A Pi_h), or level0: the level-0 stencils S (9, nv) of the hierarchies as given
    (then A may be None and only the vertex part is available)."""

    def __init__(self, kind, cell_verts, nx, ny, A=None, level0=None, max_coarse=MAX_COARSE):
        self.kind, self.nx, self.ny = kind, nx, ny
        nv = (nx + 1) * (ny + 1)
        self.Pi = transfers(kind, cell_verts, nv)
        if kind == "q1":
            self.Pi[1] = (self.Pi[0] @ sp.diags(checkerboard(nx, ny))).tocsr()
        self.nl = {"q1": 4, "p1": 3, "q2": 9}[kind]
        if level0 is None:
            A = sp.csr_matrix(A)
            level0 = [to_stencil(Pm.T @ A @ Pm, nx, ny) for Pm in self.Pi]
            if kind == "q2":
                level0[1] = hourglass_fill(level0[1], nx, ny)
        self.level0 = level0
        self.levels = [hierarchy(from_stencil(S, nx, ny), nx, ny, max_coarse) for S in level0]
        if A is not None:
            self.D, self.Dinv = block_inverses(A, self.nl)

    def stencils(self, h):
        """the 9-point form of every level of hierarchy h"""
        return [to_stencil(L["A"], L["nx"], L["ny"]) for L in self.levels[h]]

    def vertex(self, r):
        """the V-cycle results on the finest vertex level, one per hierarchy: V_h(Pi_h^T r)"""
        return [vcycle(lv, Pm.T @ r) for lv, Pm in zip(self.levels, self.Pi)]

    def vertex_scale(self, r):
        """max |V_h(|Pi_h|^T |r|)| per hierarchy: the size a rounding error of the restriction Pi_h^T r, relative to the
        magnitudes it sums, reaches after the V-cycle (Pi_h^T r cancels for a smooth r against the hourglass weights)"""
        return [np.abs(vcycle(lv, abs(Pm).T @ np.abs(r))).max() for lv, Pm in zip(self.levels, self.Pi)]

    def correction(self, r):
        return sum(Pm @ v for Pm, v in zip(self.Pi, self.vertex(r)))

    def block_jacobi(self, r):
        return np.einsum("cij,cj->ci", self.Dinv, r.reshape(-1, self.nl)).ravel()

    def __call__(self, r):
        return self.block_jacobi(r) + self.correction(r)
