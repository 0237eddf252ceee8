"""Generates tests/golden/run_imitator.json from a checkout of the reference tree (CPU only):
  * main_block: SHA-256 of the body of run_imitator.py's ``if __name__ == "__main__":`` block, and
  * tables: tests/test_run_imitator_cpu.py's table_digests of the reference's own utils/mesh.py, run on the synthetic asset
    files (impersonator_b200.synthetic.write_synthetic_assets).

  python tests/golden/make_run_imitator_golden.py REFERENCE_TREE
"""
import importlib.util
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

from impersonator_b200 import synthetic as S  # noqa: E402
import test_run_imitator_cpu as T  # noqa: E402


def main(ref):
    src = open(os.path.join(ref, "run_imitator.py")).read()
    main_block = src[src.index('if __name__ == "__main__":'):]
    main_block = main_block[main_block.index("\n") + 1:]
    spec = importlib.util.spec_from_file_location("ref_mesh", os.path.join(ref, "utils", "mesh.py"))
    R = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(R)
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        S.write_synthetic_assets(tmp, n_targets=1)
        os.chdir(tmp)                                            # utils/mesh.py resolves 'assets/pretrains/*' against the cwd
        try:
            tables = T.table_digests(R)
        finally:
            os.chdir(cwd)
    with open(os.path.join(HERE, "run_imitator.json"), "w") as fp:
        json.dump({"main_block": T.sha256(main_block.rstrip("\n").encode()), "tables": tables}, fp, indent=1)
        fp.write("\n")


if __name__ == "__main__":
    main(sys.argv[1])
