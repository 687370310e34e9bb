"""Regenerates tests/golden/ref_extend_signatures.json: the positional signatures of the reference's
`find_nearest_point_idx` and `uncertainty_pnp_v2` (lib/utils/extend_utils/extend_utils.py:39, :116), derived
from its source with `ast` by the same function as make_golden_signatures.py.  tests/test_metrics_cpu.py
compares them with the shim's.

    python tests/golden/make_golden_extend_signatures.py REFERENCE_ROOT
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

from make_golden_signatures import signatures  # noqa: E402

NAMES = ("find_nearest_point_idx", "uncertainty_pnp_v2")


def main():
    with open(os.path.join(sys.argv[1], "lib", "utils", "extend_utils", "extend_utils.py")) as f:
        found = signatures(f.read(), NAMES)
    path = os.path.join(HERE, "ref_extend_signatures.json")
    with open(path, "w") as f:
        json.dump(found, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", path, len(found), "signatures")


if __name__ == "__main__":
    main()
