"""Convert the reference's pickled walking log into the compact fixture.

Needs a checkout of the reference (it ships the log; this repository does not):
    python tests/golden/make_walking_log.py <reference>/test_data/id_qp_log_walking.npz
Writes walking_log_compact.npz and walking_log_sha256.json (SHA-256 of every stacked array of the
reference's log, which tests/test_boundary.py checks the compact copy against).
"""
import hashlib, json, os, sys
import numpy as np
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", ".."))
from fcc_qp_b200.logdata import stack_reference_log, save_compact, load_compact

KEYS = ("Q", "b", "A_eq", "b_eq", "friction_coeffs", "lb", "ub")


def digests(qp):
    return {k: {"shape": list(getattr(qp, k).shape),
                "sha256": hashlib.sha256(np.ascontiguousarray(getattr(qp, k), dtype="<f8").tobytes()).hexdigest()}
            for k in KEYS}


if __name__ == "__main__":
    src = sys.argv[1]
    dst = os.path.join(os.path.dirname(__file__), "walking_log_compact.npz")
    full = stack_reference_log(src)
    save_compact(full, dst)
    back = load_compact(dst)
    for k in KEYS:
        assert np.array_equal(getattr(full, k), getattr(back, k)), k
    with open(os.path.join(os.path.dirname(__file__), "walking_log_sha256.json"), "w") as f:
        json.dump(digests(full), f, indent=1)
        f.write("\n")
    print("ok", full.batch, os.path.getsize(dst) / 1e6, "MB")
