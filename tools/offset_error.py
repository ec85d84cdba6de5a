"""Force error of the MIXED paths on offset fields V = C + noise (noise amplitude 1, spacing 0.05 nm, FP32-representable),
against the C oracle: max|F - F_ref| / max|F_ref| per path and offset C. The cases are those of
tests/test_gpu_coverage.py::test_offset_field. Usage: python tools/offset_error.py   (GFB_LIB_PATH selects another build)"""
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
import openmmgridforce_b200 as gf  # noqa: E402
from oracle import bindings  # noqa: E402
import test_gpu_coverage as T  # noqa: E402

dev = gf.Device(0)
print("device", dev.props()["name"])
offsets = T.OFFSETS
print(f"{'path':24s}" + "".join(f"{o:>10g}" for o in offsets))
for name, precision, layout, n_grids in T.OFFSET_PATHS:
    if precision != 0:
        continue
    row = []
    for offset in offsets:
        c = T._offset_case(n_grids, 7, 300, offset, T.METHOD[layout], seed=len(name) * 31 + int(abs(offset)) % 97 + (offset < 0))
        _, f_ref = T._oracle(bindings, c)
        grids, k = T._make(gf, dev, c, precision, layout)
        _, forces, _ = k.execute_host(c["pos"])
        row.append(T._err_f(forces, f_ref))
        T._close(grids, k)
    print(f"{name:24s}" + "".join(f"{e:10.1e}" for e in row))
