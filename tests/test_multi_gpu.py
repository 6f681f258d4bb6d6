"""N>1: host-side logic on CPU with gloo (world_size 2), and — on a box with >= 2 GPUs — the
data-parallel learner with the in-kernel NVLink gradient exchange against the oracle."""
import os
import subprocess
import sys

import pytest
import torch

from conftest import ROOT


def _run_workers(script, nproc, extra_env=None, timeout=600):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1", **(extra_env or {}))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 400), script]
    return subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=timeout, cwd=ROOT)


GLOO_WORKER = r'''
import os, sys
sys.path.insert(0, %r)
import torch, torch.distributed as dist
dist.init_process_group("gloo")
from pearl_b200.dist import all_gather_bytes, shard_owner
rank, world = dist.get_rank(), dist.get_world_size()
blob = bytes([rank * 16 + i %% 16 for i in range(128)])
got = all_gather_bytes(blob)
assert len(got) == world and all(got[r] == bytes([r * 16 + i %% 16 for i in range(128)]) for r in range(world))
# interleaved shard ownership: balanced, FIFO-consistent
own = [shard_owner(g, world) for g in range(10)]
assert [o[0] for o in own] == [g %% world for g in range(10)] and own[5] == (5 %% world, 5 // world)
# max-over-ranks reduction used by bench.py
t = torch.tensor([float(rank + 1)])
dist.all_reduce(t, op=dist.ReduceOp.MAX)
assert t.item() == world
if rank == 0: print("GLOO_OK")
dist.destroy_process_group()
'''


def test_host_logic_world2_gloo(tmp_path):
    script = tmp_path / "gloo_worker.py"
    script.write_text(GLOO_WORKER % ROOT)
    out = _run_workers(str(script), 2, timeout=300)
    assert out.returncode == 0 and "GLOO_OK" in out.stdout, out.stderr[-3000:]


@pytest.mark.gpu
@pytest.mark.parametrize("double", [0, 1])
def test_data_parallel_learner_matches_oracle_on_concatenated_batch(double):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    out = _run_workers(os.path.join(ROOT, "tests", "dp_worker.py"), min(n, 4), {"DP_DOUBLE": str(double)})
    assert out.returncode == 0 and "DP_OK" in out.stdout, (out.stdout[-2000:], out.stderr[-4000:])


@pytest.mark.gpu
@pytest.mark.parametrize("double", [0, 1])
def test_sharded_replay_learner_draws_the_single_gpu_indices(double):
    """SURVEY.md 8e partitioning: replicated MT19937 stream, interleaved ownership, summed partial gradients."""
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs (bench.py --gpus N repeats this check in-run)")
    out = _run_workers(os.path.join(ROOT, "tests", "dp_shard_worker.py"), min(n, 4), {"DP_DOUBLE": str(double)})
    assert out.returncode == 0 and "DP_SHARD_OK" in out.stdout, (out.stdout[-2000:], out.stderr[-4000:])


GAE_SHARD_WORKER = r'''
import os, sys
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
dist.init_process_group("gloo")
from pearl_b200.dist import sharded_gae_fixup
from oracle.ppo_oracle import gae_reference_loop
rank, world = dist.get_rank(), dist.get_world_size()
n, gamma, lam = 90 * world, 0.97, 0.9
rng = np.random.Generator(np.random.PCG64(5))
values = torch.from_numpy(rng.standard_normal(n).astype(np.float32))
reward = torch.from_numpy(rng.standard_normal(n).astype(np.float32))
term = torch.zeros(n, dtype=torch.bool); trunc = torch.zeros(n, dtype=torch.bool)
# chunk 1 (of 3) has NO episode end: its chains must wait for chunk 2 (sequential propagation); the others have some
for t in (17, 55, 56): term[t] = True
if world > 2: trunc[2 * 90 + 30] = True; term[n - 1 - 40] = True
last_v = float(rng.standard_normal())
want_g, want_l = gae_reference_loop(values, last_v, reward, term, trunc, gamma, lam)
a, b = rank * 90, (rank + 1) * 90
v, r, te, tr = values[a:b], reward[a:b], term[a:b], trunc[a:b]
state = {}
def run(next_value, incoming):
    g, l = gae_reference_loop(v, next_value, r, te, tr, gamma, lam, incoming_gae=incoming)
    state["g"], state["l"] = g, l
    return float(g[0])
run(last_v if rank == world - 1 else 0.0, 0.0)             # local pass
rounds = sharded_gae_fixup(float(v[0]), float(state["g"][0]), bool((te | tr).any()), run)
assert torch.equal(state["g"], want_g[a:b]) and torch.equal(state["l"], want_l[a:b]), (rank, rounds)
out = [None] * world
dist.all_gather_object(out, rounds)
assert len(set(out)) == 1
if rank == 0: print("GAE_SHARD_OK rounds", rounds)
dist.destroy_process_group()
'''


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_gae_protocol_gloo(tmp_path, world):
    """The cross-shard GAE stitching (host protocol) on CPU, with the oracle loop standing in for the kernel: bit-identical to
    the whole rollout, including a chunk without any episode end."""
    script = tmp_path / "gae_shard_worker.py"
    script.write_text(GAE_SHARD_WORKER % ROOT)
    out = _run_workers(str(script), world, timeout=300)
    assert out.returncode == 0 and "GAE_SHARD_OK" in out.stdout, (out.stdout[-1000:], out.stderr[-3000:])


PPO_SHARD_WORKER = r'''
import os, sys
sys.path.insert(0, %r)
import numpy as np, torch, torch.distributed as dist
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
import pearl_b200
obs, A, per = 12, 4, 3000
n = per * world
rng = np.random.Generator(np.random.PCG64(17))
q8 = lambda x: (np.rint(x * 256) / 256).astype(np.float32)
states, reward = q8(rng.standard_normal((n + 1, obs))), q8(rng.standard_normal(n))
action = rng.integers(0, A, size=n).astype(np.int64)
term, trunc = rng.random(n) < 0.002, rng.random(n) < 0.001
term[per:2 * per] = False; trunc[per:2 * per] = False          # chunk 1 has no episode end
def make(a, b):
    buf = pearl_b200.B200ReplayBuffer(b - a)
    t = torch.from_numpy
    buf.push_batch(t(states[a:b]), t(action[a:b]), t(reward[a:b]), t(states[a + 1:b + 1]), t(term[a:b]), t(trunc[a:b]), max_number_actions=A)
    return buf
def learner():
    pl = pearl_b200.B200ProximalPolicyOptimization(state_dim=obs, n_actions=A, actor_hidden_dims=[32, 32], critic_hidden_dims=[32, 32],
                                                   training_rounds=1, batch_size=64, discount_factor=0.97, trace_decay_param=0.9, epsilon=0.2)
    g = torch.Generator().manual_seed(3)
    pl.load_parameters(torch.randn(pl.actor_params.numel(), generator=g) * 0.2, torch.randn(pl.critic_params.numel(), generator=g) * 0.2)
    return pl
whole = learner().preprocess_replay_buffer(make(0, n))                       # every rank: the unsharded rollout
pl = learner()
part = pl.preprocess_replay_buffer(make(rank * per, (rank + 1) * per), process_group=dist.group.WORLD)
a, b = rank * per, (rank + 1) * per
for k in ("values", "action_probs"):
    assert torch.allclose(part[k], whole[k][a:b], rtol=1e-5, atol=1e-6), k
# the chains are stitched exactly: identical fp32 operations on identical state values
if not torch.equal(part["values"], whole["values"][a:b]):
    # GEMM tiling is row-independent, so the values agree bit for bit; if a future kernel changes that, compare the chains on
    # the shard's own values instead
    raise AssertionError("row-parallel value pass is no longer bit-identical")
assert torch.equal(part["gae"], whole["gae"][a:b]) and torch.equal(part["lam_return"], whole["lam_return"][a:b]), rank
if rank == 0: print("PPO_SHARD_OK rounds", pl.last_shard_rounds)
dist.barrier()
dist.destroy_process_group()
'''


@pytest.mark.gpu
def test_sharded_ppo_preprocessing_matches_unsharded(tmp_path):
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    script = tmp_path / "ppo_shard_worker.py"
    script.write_text(PPO_SHARD_WORKER % ROOT)
    out = _run_workers(str(script), min(n, 3), timeout=600)
    assert out.returncode == 0 and "PPO_SHARD_OK" in out.stdout, (out.stdout[-2000:], out.stderr[-4000:])
