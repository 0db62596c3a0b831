import os, sys, warnings
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, scipy.sparse as sp, scipy.sparse.linalg as spla
from oracle import oracle as o
from tests.test_mg_prototype import _hierarchy, _vcycle
warnings.filterwarnings("ignore")

def run(n, variant, diffusion=None):
    m = o.mesh_cube(n, n, -1.0, 1.0, -1.0, 1.0).with_polorder(2)
    rp, col = o.pattern(m)
    fac = o.const(1.0) if diffusion is None else o.cellwise(diffusion)
    A = o.to_scipy(rp, col, o.assemble_lhs(m, fac, None, rp, col)).tocsr()
    b = o.assemble_rhs(m, o.esv2007_force())
    N, nv, nc = m.n_dofs, m.nv, m.nc
    # Q1 vertex function -> Q2 nodal values
    rows, cols, vals = [], [], []
    w = lambda i, a: (1 - a / 2) if i == 0 else a / 2
    cv = m.cv.reshape(-1, 4)
    for c in range(nc):
        for bb in range(3):
            for aa in range(3):
                d = 9 * c + aa + 3 * bb
                for j in range(2):
                    for i in range(2):
                        ww = w(i, aa) * w(j, bb)
                        if ww:
                            rows.append(d); cols.append(cv[c, i + 2 * j]); vals.append(ww)
    P = sp.csr_matrix((vals, (rows, cols)), shape=(N, nv))
    Ac = (P.T @ A @ P).tocsr()
    ix, iy = np.arange(nv) % (n + 1), np.arange(nv) // (n + 1)
    coo = Ac.tocoo()
    far = (np.abs(ix[coo.row] - ix[coo.col]) > 1) | (np.abs(iy[coo.row] - iy[coo.col]) > 1)
    print("  far max", np.abs(coo.data[far]).max(initial=0.0) / np.abs(coo.data).max())
    C = sp.diags((-1.0) ** (ix + iy))
    lv, lvC = _hierarchy(Ac, n), _hierarchy((C @ Ac @ C).tocsr(), n)
    lu = spla.splu(Ac.tocsc())
    D = sp.block_diag([sp.csr_matrix(np.linalg.inv(A[9 * c:9 * c + 9, 9 * c:9 * c + 9].toarray())) for c in range(nc)], format="csr")
    dj = 1.0 / A.diagonal()
    def prec(r):
        if variant == "jacobi": return dj * r
        if variant == "block": return D @ r
        z, rc = D @ r, P.T @ r
        if variant == "exact":
            return z + P @ lu.solve(rc)
        z = z + P @ _vcycle(lv, 0, rc)
        if variant == "twisted":
            z = z + P @ (C @ _vcycle(lvC, 0, C @ rc))
        return z
    it = [0]
    x, info = spla.cg(A, b, rtol=1e-10, maxiter=5000, M=spla.LinearOperator((N, N), matvec=prec),
                      callback=lambda xk: it.__setitem__(0, it[0] + 1))
    return it[0], info

for n in (8, 16, 32):
    print(n, {v: run(n, v) for v in ("jacobi", "block", "exact", "plain", "twisted")})
