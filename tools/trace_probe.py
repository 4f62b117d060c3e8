import os, sys, ctypes as C
os.environ["C3R_TRACE"] = "1"
sys.path.insert(0, os.getcwd())
import numpy as np
from clair3_rna_b200 import weights
from clair3_rna_b200.engine import Engine
g = np.load("tests/golden/cfg1_ont_drna.npz")
x = np.concatenate([g["tensor"]] * 40)[:29696]     # 116 tiles like the bench
eng = Engine(0, 18); eng.set_weights(weights.synthetic(18, sharpen=8.0))
for _ in range(3): p, ms = eng.forward(x)
print("forward ms", ms)
buf = np.zeros(2 * 33 * 8 * 8, np.int64); nb = C.c_int64(0)
eng.lib.c3r_debug_fetch(eng.ctx, 4, buf.ctypes.data, buf.nbytes, C.byref(nb))
T = buf.reshape(2, 33, 8, 8)     # LSTM1: rank, step, chunk, event
t0 = T[0, 2, 0, 0]
for step in (2, 3, 4):
    for c in range(4):
        m = T[0, step, c]; g1 = T[1, step, c]
        print("step %d c %d | mma wait_done %7d commit +%5d | r0 gate: accf %7d ld +%4d arrive +%5d | r1 gate(own clk): accf->arrive %5d relay-after-arrive %5d" % (
            step, c, m[0] - t0, m[1] - m[0], m[2] - t0, m[3] - m[2], m[4] - m[2], g1[4] - g1[2], g1[5] - g1[4]))
    l = T[0, step, 0]
    print("   loader r0: start %7d dur %6d" % (l[6] - t0, l[7] - l[6]))
