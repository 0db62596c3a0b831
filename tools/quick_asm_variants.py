"""matrix-assembly kernel time (ESV2007 data): python tools/quick_asm_variants.py n polorder [cube|simplex]"""
import sys, json, ctypes as C
sys.path.insert(0, '.')
import dune_hdd_b200 as hdd
from dune_hdd_b200 import capi
n, p = int(sys.argv[1]), int(sys.argv[2])
kind = sys.argv[3] if len(sys.argv) > 3 else "cube"
g = hdd.grids.cube(n) if kind == "cube" else hdd.grids.simplex(n)
d = hdd.SWIPDG(g, hdd.problems.ESV2007(), polorder=p)
d.init()
L = capi.lib()
sec, byt = C.c_double(), C.c_double()
capi.check(L.hdd_profile_kernel(d._h, 3, 10, C.byref(sec)))
capi.check(L.hdd_kernel_bytes(d._h, 3, C.byref(byt)))
print(json.dumps({"n": n, "p": p, "kind": kind, "ms": sec.value * 1e3, "GBs": byt.value / sec.value / 1e9}))
