"""PearlAgent (the reference's own facade, pearl/pearl_agent.py) on top of the CUDA path.  Needs facebookresearch/Pearl
(tests/_pearl.py: the build of it in oracle/_ref/, $PEARL_REFERENCE_ROOT or an importable `pearl`).  Skipped otherwise."""
import os
import subprocess
import sys

import pytest

from _pearl import PEARL_ROOT as REF
from conftest import ROOT


@pytest.mark.gpu
@pytest.mark.skipif(REF is None, reason="facebookresearch/Pearl is not available")
def test_pearl_agent_drives_the_b200_plugins_like_the_reference_plugins():
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "pearl_agent_worker.py"), REF], capture_output=True, text=True,
                         env=env, timeout=900)
    print(out.stdout[-3000:])
    assert out.returncode == 0 and "PEARL_AGENT_OK" in out.stdout, (out.stdout[-2000:], out.stderr[-6000:])


@pytest.mark.gpu
@pytest.mark.skipif(REF is None, reason="facebookresearch/Pearl is not available")
def test_actor_critic_plugins_subclass_the_reference_and_run_under_pearl_agent():
    """SAC / TD3 / DDPG / PPO: the plugins are the reference classes with learn() replaced (pearl_b200/actor_critic.py)."""
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "pearl_agent_ac_worker.py"), REF], capture_output=True, text=True,
                         env=env, timeout=900)
    print(out.stdout[-3000:])
    assert out.returncode == 0 and "PEARL_AGENT_AC_OK" in out.stdout, (out.stdout[-2000:], out.stderr[-6000:])
