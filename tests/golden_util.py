import glob
import os

import numpy as np

from tests.fixtures import gaussian, sincos_dataset

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# A checkout of the reference project (leolee9086/better-binary-quantization), the source golden/from_ts was generated
# from.  Only the tests that execute the reference's own files read it; they skip when BBQ_REFERENCE_DIR is not set.
REFERENCE_DIR = os.environ.get("BBQ_REFERENCE_DIR", "")
HAVE_REFERENCE = bool(REFERENCE_DIR) and os.path.isdir(os.path.join(REFERENCE_DIR, "src"))


def golden_cases():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


def load_golden(name):
    g = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz")))
    for key in ("n", "dim", "query_bits", "k", "iters", "seed"):
        g[key] = int(g[key])
    g["lam"] = float(g["lam"])
    g["sim"] = str(g["sim"])
    nq = g["top_idx"].shape[0]
    if g["seed"] >= 0:
        g["base"], g["queries"] = gaussian(g["n"], g["dim"], g["seed"]), gaussian(nq, g["dim"], g["seed"] + 100)
    else:
        g["base"], g["queries"] = sincos_dataset(g["dim"], g["n"], nq)
    return g
