#!/usr/bin/env python3
"""Copies the UNMODIFIED reference (danieleschmidt/connectome-gnn-suite, pure Python: package, tests, example) from the
checkout that the environment variable CGNN_REFERENCE names into oracle/_ref/ (git-ignored).  Test / baseline
infrastructure only: `bench.py --impl reference` and the cpu_baseline leg time its Trainer.train_epoch / evaluate on the
host cores, and tests/test_gpu_reference_suite.py runs its own 43 tests and examples/demo.py against the B200 package.
Nothing under connectome-gnn-suite_b200/ imports it.  No-op when CGNN_REFERENCE is unset: a copy made earlier is kept."""
import os
import shutil
import sys

SRC = os.environ.get("CGNN_REFERENCE", "")
DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def main() -> int:
    if not SRC:
        print(f"make_ref: CGNN_REFERENCE is not set, keeping {DST} as it is")
        return 0
    if not os.path.isdir(os.path.join(SRC, "connectome_gnn")):
        print(f"make_ref: CGNN_REFERENCE={SRC} is not a checkout of the reference (no connectome_gnn/ in it)", file=sys.stderr)
        return 1
    os.makedirs(DST, exist_ok=True)
    # the package on its own; its callers (tests, example) in a sibling tree WITHOUT the package next to them - demo.py puts
    # its grandparent directory first on sys.path, and the acceptance test wants `import connectome_gnn` to find the B200 build
    for name, rel in (("connectome_gnn", "connectome_gnn"), ("tests", os.path.join("callers", "tests")),
                      ("examples", os.path.join("callers", "examples"))):
        dst = os.path.join(DST, rel)
        if os.path.isdir(dst):
            shutil.rmtree(dst)
        shutil.copytree(os.path.join(SRC, name), dst, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    for stale in ("tests", "examples"):
        if os.path.isdir(os.path.join(DST, stale)):
            shutil.rmtree(os.path.join(DST, stale))
    print(f"make_ref: copied the reference package, tests and example into {DST}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
