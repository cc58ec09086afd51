"""Records tests/golden/ref_kernels.json: the digest of every output tests/test_ref_gpu_kernels.py compares.

Runs that test module on a B200 with its comparison replaced by a recorder, so the cases and the digest are the test's
own.  Record only from kernels known to give the reference kernels' bits on every case — the file is what all later
builds are held to.

    python tests/golden/make_ref_kernel_digests.py [OUT.json]
"""
import json
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)

ABOUT = ("SHA-256 digests (digest() in tests/test_ref_gpu_kernels.py) of the outputs of the reference's CUDA kernels - "
         "kornia-rs' kernel strings compiled with NVRTC (compute_100, --fmad=false) and launched with its launch geometry - "
         "on the inputs of tests/test_ref_gpu_kernels.py.  Recorded on a B200 by tests/golden/make_ref_kernel_digests.py from "
         "this project's kernels, at a revision whose kernels that test, then running the reference's kernels side by side, "
         "had found bit-identical to them in every case.")


def main() -> int:
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref_kernels.json")
    sys.path.insert(0, TESTS)
    import test_ref_gpu_kernels as t   # pytest reuses this module object, so the recorder below is what the tests call

    digests = {}

    def record(key, got, what=""):
        d = t.digest(got)
        assert digests.setdefault(key, d) == d, f"case key {key!r} names two different outputs"

    t.same_bits = record
    rc = pytest.main([t.__file__, "-q", "-p", "no:cacheprovider"])
    if rc != 0:
        print(f"[ref-digests] pytest failed (exit {int(rc)}): nothing written", file=sys.stderr)
        return 1
    with open(out, "w") as f:
        json.dump({"about": ABOUT, "digests": dict(sorted(digests.items()))}, f, indent=1)
        f.write("\n")
    print(f"[ref-digests] {len(digests)} digests written to {out}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
