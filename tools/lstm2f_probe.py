"""Fused-LSTM2 probe: numerics against the oracle (h2 and probabilities) and forward time at a bench-sized batch.
Usage: [C3R_LSTM2F_NP=1|2|4] python tools/lstm2f_probe.py [n_sites] [out.npy]"""
import os, sys, time, numpy as np
sys.path.insert(0, os.getcwd())
from clair3_rna_b200 import weights
from clair3_rna_b200.engine import Engine
from oracle import model
n_big = int(sys.argv[1]) if len(sys.argv) > 1 else 14617
tag = "NP=%s" % os.environ.get("C3R_LSTM2F_NP", "-")
g = np.load("tests/golden/cfg1_ont_drna.npz")
x = g["tensor"][:300]
w = weights.synthetic(18, sharpen=8.0)
eng = Engine(0, 18, nn_impl=1); eng.set_weights(w)
p, ms = eng.forward(x)
inter = {}
ref = model.forward(w, x, intermediates=inter)
h2 = eng.debug_fetch(2, len(x))
print(tag, "n=300 h2 err %.3e  probs err %.3e" % (np.abs(h2 - inter["h2"]).max(), np.abs(p - ref).max()), flush=True)
xb = np.concatenate([g["tensor"]] * (n_big // len(g["tensor"]) + 1))[:n_big]
for _ in range(3): pb, ms = eng.forward(xb)
t = [eng.forward(xb)[1] for _ in range(5)]
print(tag, "n=%d forward ms best %.4f median %.4f" % (n_big, min(t), sorted(t)[2]), flush=True)
# a site's result must not depend on where in the batch it sits
k = len(g["tensor"])
print(tag, "batch-position invariance:", bool(np.array_equal(pb[:k], pb[k:2 * k])) if n_big >= 2 * k else "n/a", flush=True)
if os.environ.get("C3R_TRACE"):
    import ctypes as C
    buf = np.zeros(2 * 2 * 33 * 8 * 8, np.int64); nb = C.c_int64(0)
    eng.lib.c3r_debug_fetch(eng.ctx, 4, buf.ctypes.data, buf.nbytes, C.byref(nb))
    buf = buf[2 * 33 * 8 * 8:]
    names = ["acc_empty", "acc_empty_peer", "x", "h_ready", "w_full", "w_peer_full", "total", "steps", "producer_wait_empty", "gate0_wait_acc"]
    tot, steps = float(buf[6]), float(buf[7])
    print(tag, "MMA thread cycles/step %.0f;" % (tot / max(steps, 1)), " ".join("%s %.0f" % (nm, buf[i] / max(steps, 1)) for i, nm in enumerate(names) if i not in (6, 7)), flush=True)
    tr = buf[16:16 + 30 * 4].reshape(30, 4).astype(np.int64)
    t0 = tr[0, 0]
    print(tag, "step-3 stage trace (cycles from step start: top, waits done, MMAs issued, commit issued):")
    for i in range(30):
        print("   c%d s%02d  %6d %6d %6d %6d" % (i // 6, i % 6, tr[i, 0] - t0, tr[i, 1] - t0, tr[i, 2] - t0, tr[i, 3] - t0))
if len(sys.argv) > 2: np.save(sys.argv[2], pb)
eng.close()
