"""Test helpers: oracle evaluation in K-chunks (memory-light at full BASELINE sizes), golden fixture loading."""
import glob
import os

import numpy as np

from oracle import moco_oracle as O


def load_contrast_golden(golden_dir):
    """tests/golden/contrast*.npz as one mapping.  ``<case>_memory_final`` (the reference's queue after the last step)
    is stored as the ring slots it wrote and rebuilt here from ``<case>_memory0``."""
    g = {}
    for path in sorted(glob.glob(os.path.join(golden_dir, "contrast*.npz"))):
        with np.load(path) as z:
            g.update({k: z[k] for k in z.files})
    for key in [k for k in g if k.endswith("_memory_final_rows")]:
        case = key[:-len("_memory_final_rows")]
        final = g[f"{case}_memory0"].copy()
        final[g[key]] = g[f"{case}_memory_final_vals"]
        g[f"{case}_memory_final"] = final
    return g


def oracle_head_chunked(q, k, memory, T, chunk=16384, want_dq=True):
    """(lse[N], loss, prob, dq[N,C]) of the reference head, evaluated with the oracle's own
    functions on column chunks of the queue and merged with the log-sum-exp identity
    logsumexp(concat(a, b)) = logaddexp(logsumexp(a), logsumexp(b))."""
    N, C = q.shape
    K = memory.shape[0]
    q64, k64 = q.astype(np.float64), k.astype(np.float64)
    x0 = (q64 * k64).sum(-1) / T
    lse = x0.copy()
    for j0 in range(0, K, chunk):
        part = O.MemoryMoCoOracle(memory[j0:j0 + chunk], T).logits(q, k)[:, 1:]      # Contrast.py:25-27
        lse = np.logaddexp(lse, O.logsumexp_rows(part.astype(np.float64)))
    loss = float((lse - x0).mean())
    prob_rows = np.exp(x0 - lse)
    dq = None
    if want_dq:
        acc = (prob_rows - 1.0)[:, None] * k64
        for j0 in range(0, K, chunk):
            m = memory[j0:j0 + chunk].astype(np.float64)
            p = np.exp(q64 @ m.T / T - lse[:, None])
            acc += p @ m
        dq = acc / (T * N)
    return lse, loss, float(prob_rows.mean()), dq


def rand_unit(rng, n, c):
    x = rng.standard_normal((n, c)).astype(np.float32)
    return O.bf16_round(O.l2_normalize(x))
