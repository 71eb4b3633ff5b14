"""make_golden_linear.py — Linear golden vectors at the headline shapes, minted on a GPU box from the REFERENCE's
own cublasSgemm calls (oracle/_ref: linear_kernel.cu:76-80 forward, :220-231 backward, the reference's arguments).

    python tests/golden/make_golden_linear.py [out.npz]        # needs a GPU and oracle/_ref/libroc_ref.so

1000 x 602 . 64 x 602 and 1000 x 64 . 41 x 64: the shapes of BASELINE.json configs[1].  The GPU tests feed them
row-padded (ld % 4 == 0), so the tcgen05 kernels — not the SIMT fallback the small unpadded golden case reaches —
are what meets the reference library's outputs.  Inputs are regenerated from the seed by the test.  Y and dX are
stored at `rows_<shape>` (ROWS of the 1000 rows), dW at `wrows_<shape>` (WROWS output features): every stored
value is a complete dot product, and the file stays small."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402

SHAPES = [(1000, 602, 64), (1000, 64, 41)]
ROWS, WROWS = 128, 16


def inputs(n, i, o):
    r = np.random.RandomState(1000 * i + o)
    return (r.rand(n, i).astype(np.float32) * 2 - 1, r.rand(o, i).astype(np.float32) * 2 - 1,
            r.rand(n, o).astype(np.float32) * 2 - 1)


def sample(n, k, seed):
    return np.sort(np.random.RandomState(seed).choice(n, k, replace=False)).astype(np.int64)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "ref_golden_linear.npz")
    assert ref.available(), "oracle/_ref/libroc_ref.so missing"
    G = {}
    for (n, i, o) in SHAPES:
        X, W, dY = inputs(n, i, o)
        x, w, gy = (torch.from_numpy(a).cuda() for a in (X, W, dY))
        y = ref.linear_fwd(x, w, relu=False)
        gw, gx = torch.zeros_like(w), torch.zeros_like(x)
        ref.linear_bwd(x, w, y, gy.clone(), gw, gx, relu=False)
        torch.cuda.synchronize()
        k = "%dx%dx%d" % (n, i, o)
        rows, wrows = sample(n, ROWS, i + o), sample(o, WROWS, i * o)
        G["rows_" + k], G["wrows_" + k] = rows, wrows
        G["Y_" + k], G["dW_" + k], G["dX_" + k] = (y.cpu().numpy()[rows], gw.cpu().numpy()[wrows],
                                                   gx.cpu().numpy()[rows])
    np.savez_compressed(out, **G)
    print("wrote", out, {k: v.shape for k, v in G.items()}, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
