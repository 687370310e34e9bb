"""Regenerates tests/golden/ref_signatures.json: the positional signatures (parameter names and defaults)
of the public functions of the reference's lib/ransac_voting_gpu_layer/ransac_voting_gpu.py, derived from
its source with `ast`.  tests/test_dropin_imports.py compares them with the signatures it expects of the
drop-in shim.

    python tests/golden/make_golden_signatures.py REFERENCE_ROOT
"""
import ast
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests.test_dropin_imports import EXPECTED  # noqa: E402


def signatures(source, names):
    found = {}
    for node in ast.parse(source).body:
        if isinstance(node, ast.FunctionDef) and node.name in names:
            a = node.args
            names_ = [x.arg for x in a.args]
            defaults = [None] * (len(names_) - len(a.defaults)) + [ast.literal_eval(d) for d in a.defaults]
            found[node.name] = ", ".join(n if d is None and i < len(names_) - len(a.defaults) else f"{n}={d!r}"
                                         for i, (n, d) in enumerate(zip(names_, defaults)))
    return found


def main():
    src = os.path.join(sys.argv[1], "lib", "ransac_voting_gpu_layer", "ransac_voting_gpu.py")
    with open(src) as f:
        found = signatures(f.read(), EXPECTED)
    path = os.path.join(HERE, "ref_signatures.json")
    with open(path, "w") as f:
        json.dump(found, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", path, len(found), "signatures")


if __name__ == "__main__":
    main()
