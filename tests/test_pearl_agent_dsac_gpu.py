"""PearlAgent (the reference's own facade, pearl/pearl_agent.py) driving B200SoftActorCritic, the discrete SAC plugin.  Needs
facebookresearch/Pearl (tests/_pearl.py: the build of it in oracle/_ref/, $PEARL_REFERENCE_ROOT or an importable `pearl`).
Skipped otherwise."""
import os
import subprocess
import sys

import pytest

from _pearl import PEARL_ROOT as REF
from conftest import ROOT


@pytest.mark.gpu
@pytest.mark.skipif(REF is None, reason="facebookresearch/Pearl is not available")
def test_discrete_sac_plugin_subclasses_the_reference_and_runs_under_pearl_agent():
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "pearl_agent_dsac_worker.py"), REF], capture_output=True,
                         text=True, env=env, timeout=900)
    print(out.stdout[-3000:])
    assert out.returncode == 0 and "PEARL_AGENT_DSAC_OK" in out.stdout, (out.stdout[-2000:], out.stderr[-6000:])
