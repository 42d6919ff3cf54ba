"""TEST INFRASTRUCTURE ONLY -- the AssoIter fixture at a scale above c3 where AssoIter accepts a column and then stops in
the middle of a sweep (c3 accepts nothing).

    python oracle/make_iter_digest.py [threads]      # seconds

Asso(k) and then AssoIter(k) on its factors, both by the bit-packed C restatement (oracle/asso_oracle_c.py), on the
seeded synthetic matrix of ITER_SCALE; writes tests/golden/iter_scale_digest.json: the config, the SHA-256 of the Asso
factors, and of AssoIter the accept / skip trace, the logged score / error bits and the SHA-256 of the refined U.
"""
import hashlib
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from oracle import asso_oracle_c as OC  # noqa: E402
from oracle.make_digests import OUT, fit_digest  # noqa: E402
from pybmf_b200 import synth  # noqa: E402

# synth.planted arguments, then Asso's tau / k / w_fp
ITER_SCALE = {"planted": [10000, 4000, 6, 0.2, 0.2, 0.3, 0.05, 15], "tau": 0.35, "k": 6, "w_fp": 0.5}


def main():
    threads = int(sys.argv[1]) if len(sys.argv) > 1 else None
    cfg = ITER_SCALE
    X = synth.planted(*cfg["planted"])
    d, r = fit_digest("iter_scale", X, cfg["k"], cfg["tau"], cfg["w_fp"], threads)
    t0 = time.time()
    U, V = np.stack(r["U_cols"], 1), np.stack(r["V_cols"], 1)
    it = OC.asso_iter_fit(X, U, V, cfg["k"], cfg["w_fp"])
    h = hashlib.sha256()
    for c in range(it["U"].shape[1]):
        h.update(OC.column_bytes(it["U"][:, c]))
    out = dict(cfg, config="iter_scale", m=int(X.shape[0]), n=int(X.shape[1]), nnz=int(X.nnz),
               asso_u_sha256=d["u_sha256"], asso_v_sha256=d["v_sha256"],
               trace=[[int(a), int(b)] for a, b in it["trace"]],
               score_bits=[np.float64(s).tobytes().hex() for s in it["scores"]],
               error_bits=[np.float64(s).tobytes().hex() for s in it["errors"]],
               u_sha256=h.hexdigest(), u_ones=int(it["U"].sum()), oracle_seconds=time.time() - t0,
               made_by="oracle/make_iter_digest.py (AssoIter on the C restatement's Asso factors)")
    with open(os.path.join(OUT, "iter_scale_digest.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print("iter_scale: %d column passes, %d accepted" % (len(out["trace"]), len(out["score_bits"])))


if __name__ == "__main__":
    main()
