"""Re-export of the A/B main-loop harness (lives in oracle/ because bench.py's reference arm uses it too), and the stored results
of the reference's own kernels that the A/B tests compare with."""
import json
import os

from oracle.mainloop import MainLoop, pitch, ptr, to_dev, to_host  # noqa: F401

REFERENCE_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_ab.json")


def reference_golden(key):
    """One record of tests/golden/ref_ab.json (written by tests/golden/gen_golden_ab.py)."""
    with open(REFERENCE_GOLDEN) as f:
        return json.load(f)[key]
