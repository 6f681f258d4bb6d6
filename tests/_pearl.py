"""Where facebookresearch/Pearl is, for the tests of the plugin boundary with it (subclassing its learners, running under
its PearlAgent).  Pearl is not a dependency of pearl_b200 and is not part of this repository: those tests use the build
of it that build() leaves in oracle/_ref/ (oracle/ref_build.py), a checkout named by $PEARL_REFERENCE_ROOT, or an
importable `pearl`, and skip where there is none."""
import importlib.util
import os

from conftest import ROOT


def pearl_root():
    for root in (os.environ.get("PEARL_REFERENCE_ROOT", ""), os.path.join(ROOT, "oracle", "_ref")):
        if root and os.path.isdir(os.path.join(root, "pearl")):
            return root
    spec = importlib.util.find_spec("pearl")
    if spec is not None and spec.submodule_search_locations:
        return os.path.dirname(list(spec.submodule_search_locations)[0])
    return None


PEARL_ROOT = pearl_root()
