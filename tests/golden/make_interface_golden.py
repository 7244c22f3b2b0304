"""Records the interface the mirrors share with the reference as tests/golden/interface_golden.json:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_interface_golden.py

  * signatures: parameter names of the agent methods the reference's callers use (tests/test_agent_mirrors.py SHARED_METHODS);
  * loader: the loader's output on the seeded on-disk tree of tests/test_loader_on_disk.py (_scenes(), loader_record()).
The values are taken from this repository's mirrors: the reference's source is not part of the repository.  With MSC_REFERENCE_SRC
naming its src/ directory, test_patch_reference_on_the_real_reference_classes and test_reference_loader_and_mirror_agree_on_the_same_tree
check the mirrors against the reference itself; the tests that read this file check the mirrors against the record on every run.
"""
import json
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.dont_write_bytecode = True
sys.path[:0] = [ROOT, os.path.join(ROOT, "multimodal-scene-captioning_b200"), os.path.join(ROOT, "tests", "devkit_shim")]

from msc_geom import io as mio  # noqa: E402
from msc_geom import nuscenes_loader as nl  # noqa: E402
from tests.test_agent_mirrors import mirror_signatures  # noqa: E402
from tests.test_loader_on_disk import _scenes, loader_record  # noqa: E402


def main():
    assert nl.NUSCENES_AVAILABLE  # the devkit shim stands in for the devkit's table access
    with tempfile.TemporaryDirectory() as root:
        mio.write_nuscenes_tree(root, _scenes())
        loader = loader_record(nl.create_loader(root, "v1.0-mini"))
    out = {"signatures": mirror_signatures(), "loader": loader}
    with open(os.path.join(HERE, "interface_golden.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote interface_golden.json:", len(loader["samples"]), "samples,", sum(len(v) for v in out["signatures"].values()), "signatures")


if __name__ == "__main__":
    main()
