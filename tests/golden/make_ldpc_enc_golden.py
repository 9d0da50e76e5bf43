"""Generate tests/golden/ldpc_enc_golden.npz from the reference's 28 generator-matrix goldens.

Needs /root/reference (build container only). For every /root/reference/test/codes/ldpc/k{K}_n{N}_G.npy (the matrices
the reference's own encoder test multiplies with, test/unit/fec/test_ldpc_encoding.py:97-148) draw 4 seeded random
information words u, compute c = u G mod 2 with the golden G, and store (k, n, packbits(u), packbits(c)). The smallest
matrix (k = 64, n = 128) is also stored whole, as packbits(G), so that every row of the encoder can be checked. The
fixture (~120 KB) is all the tests need; the 18 MB of G matrices are not part of the repository.
"""
import os, re
import numpy as np

src = "/root/reference/test/codes/ldpc"
out = {}
params = []
for f in sorted(os.listdir(src)):
    mt = re.match(r"k(\d+)_n(\d+)_G\.npy", f)
    if not mt:
        continue
    k, n = int(mt.group(1)), int(mt.group(2))
    gm_sp = np.array(np.load(os.path.join(src, f), allow_pickle=True))
    gm = np.zeros((k, n), np.uint8)
    gm[gm_sp[0].astype(int) - 1, gm_sp[1].astype(int) - 1] = 1            # 1-based (row, col) pairs
    rng = np.random.default_rng(1000 * k + n)
    u = rng.integers(0, 2, (4, k)).astype(np.uint8)
    u[0, :] = 0
    u[0, rng.integers(0, k)] = 1                                            # one unit vector = one row of G
    c = (u.astype(np.int64) @ gm.astype(np.int64)) % 2
    out[f"u_{k}_{n}"] = np.packbits(u, axis=1)
    out[f"c_{k}_{n}"] = np.packbits(c.astype(np.uint8), axis=1)
    if (k, n) == (64, 128):
        out["g_64_128"] = np.packbits(gm, axis=1)
    params.append((k, n))
    print(k, n, gm.sum())
out["params"] = np.array(params, np.int32)
np.savez_compressed(os.path.join(os.path.dirname(__file__), "ldpc_enc_golden.npz"), **out)
