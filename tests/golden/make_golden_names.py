"""Writes tests/golden/reference_names.json: the public names the reference's utils/utils.py and utils/datasets.py define
themselves (imported modules and names excluded).  tests/test_abi_cpu.py builds a stub checkout that defines these names and
checks that the mirror resolves every one of them: its own function where it has one, the reference's otherwise.

Run where the reference checkout is available (needs its imports: OpenCV, tqdm, torchvision):
    python tests/golden/make_golden_names.py --reference <checkout>
"""
import argparse
import importlib.util
import json
import os

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", required=True)
    args = ap.parse_args()
    out = {}
    for rel in ("utils/utils.py", "utils/datasets.py"):
        spec = importlib.util.spec_from_file_location("_reference_" + os.path.basename(rel)[:-3], os.path.join(args.reference, rel))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        out[rel] = sorted(n for n in dir(m) if not n.startswith("_") and getattr(getattr(m, n), "__module__", None) == m.__name__)
    with open(os.path.join(HERE, "reference_names.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print(out)


if __name__ == "__main__":
    main()
