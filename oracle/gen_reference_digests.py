#!/usr/bin/env python
"""Record what the UNMODIFIED reference produces for the committed goldens, as one SHA-256 per array.

TEST INFRASTRUCTURE ONLY.  Needs the reference checkout (``REF`` of oracle/gen_golden.py), like the
generators it re-runs: oracle/gen_golden.compute_case for the solver cases below and
oracle/gen_golden_tfshim.generate for picnn_tfshim.npz.  The digests go to
tests/golden/reference_digests.json, so that the tests can check, without the reference, that every
committed golden array is bit for bit what the reference computed.

Usage:  python oracle/gen_reference_digests.py
"""
import contextlib
import hashlib
import io
import json
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PATH = os.path.join(ROOT, "tests", "golden", "reference_digests.json")
SOLVER_CASES = ["c1_pc", "c1_dual", "c1_rl", "c1_boyd", "c4_rl"]


def array_digest(a):
    """SHA-256 over dtype, shape and bytes: equal digests mean bit-identical arrays."""
    a = np.asarray(a)
    h = hashlib.sha256()
    h.update(a.dtype.str.encode())
    h.update(repr(a.shape).encode())
    h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def load():
    """-> {golden file name: {array name: digest}}."""
    with open(PATH) as f:
        return json.load(f)


def main():
    from oracle import gen_golden, gen_golden_tfshim
    out = {}
    with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
        warnings.simplefilter("ignore")       # the reference runs under np.seterr(all='warn')
        for case in SOLVER_CASES:
            spec = [c for c in gen_golden.CASES if c[0] == case][0]
            fresh = gen_golden.compute_case(*spec)[0]
            out[case + ".npz"] = {k: array_digest(v) for k, v in sorted(fresh.items())}
        fresh = gen_golden_tfshim.generate()
        out["picnn_tfshim.npz"] = {k: array_digest(v) for k, v in sorted(fresh.items())}
    with open(PATH, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", PATH, sum(len(v) for v in out.values()), "digests")


if __name__ == "__main__":
    main()
