"""The discrete SAC restatement (oracle/dsac_oracle.py) against the recordings of the reference's
PearlAgent(SoftActorCritic, BasicReplayBuffer).learn(), agent.reset(), learn() (tests/golden/dsac_small.npz with the
entropy coefficient tuned, dsac_fixed.npz with it fixed)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle.dsac_oracle import OracleDiscreteSAC
from oracle.pearl_oracle import flat


def make_oracle(fx):
    init = {k: fx[f"init_{k}"] for k in ("actor", "q1", "q2", "q1t", "q2t")}
    return OracleDiscreteSAC(int(fx["obs"]), int(fx["n_act"]), (32, 32), (32, 32), actor_lr=float(fx["actor_lr_call"][0]),
                             critic_lr=float(fx["critic_lr"]), gamma=float(fx["gamma"]), tau=float(fx["tau"]),
                             entropy_coef=float(fx["entropy_coef"]), autotune=bool(fx["autotune"]), init=init)


def batch_of(fx, idx):
    t = lambda k: torch.from_numpy(fx[k][idx])  # noqa: E731
    return dict(state=t("state"), action=t("action"), reward=t("reward"), next_state=t("next_state"), terminated=t("terminated"))


@pytest.mark.parametrize("name", ["dsac_small", "dsac_fixed"])
def test_dsac_oracle_reproduces_reference(name):
    torch.set_num_threads(1)
    fx = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    R = int(fx["rounds"])
    orc = make_oracle(fx)
    if bool(fx["autotune"]):
        np.testing.assert_array_equal(np.float32(orc.target_entropy), fx["target_entropy"])
    tol = dict(rtol=5e-6, atol=5e-7)
    for call in (1, 2):
        if call == 2:
            orc.scheduler_step()
            assert orc.opt_actor.param_groups[0]["lr"] == float(fx["actor_lr_call"][1])
        for r in range(R):
            out = orc.learn_batch(batch_of(fx, fx["idx"][(call - 1) * R + r]))
            np.testing.assert_allclose(out["actor_loss"], fx[f"actor_loss{call}"][r], rtol=5e-6, atol=1e-7)
            np.testing.assert_allclose(out["critic_loss"], fx[f"critic_loss{call}"][r], rtol=5e-6)
            if bool(fx["autotune"]):
                np.testing.assert_allclose(out["entropy_coef"], fx[f"entropy_loss{call}"][r], rtol=5e-6, atol=1e-7)
        np.testing.assert_allclose(flat(orc.actor).numpy(), fx[f"after{call}_actor"], **tol)
        np.testing.assert_allclose(flat(orc.q[0]).numpy(), fx[f"after{call}_q1"], **tol)
        np.testing.assert_allclose(flat(orc.q[1]).numpy(), fx[f"after{call}_q2"], **tol)
        np.testing.assert_allclose(flat(orc.qt[0]).numpy(), fx[f"after{call}_q1t"], **tol)
        np.testing.assert_allclose(flat(orc.qt[1]).numpy(), fx[f"after{call}_q2t"], **tol)
        np.testing.assert_allclose(np.float32(orc.alpha), fx[f"after{call}_entropy_coef"], **tol)
        if bool(fx["autotune"]):
            st = orc.opt_alpha.state[orc.log_alpha]
            np.testing.assert_allclose(orc.log_alpha.detach().numpy(), fx[f"after{call}_log_entropy"], **tol)
            np.testing.assert_allclose(st["exp_avg"].numpy(), fx[f"after{call}_entropy_exp_avg"], **tol)
            np.testing.assert_allclose(st["exp_avg_sq"].numpy(), fx[f"after{call}_entropy_exp_avg_sq"], rtol=5e-6, atol=1e-12)
