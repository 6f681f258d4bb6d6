"""Time the discrete SAC learner (pearl_b200.B200SoftActorCritic) on one GPU against the eager-PyTorch restatement of the
reference on the host (oracle/dsac_oracle.py), and print one JSON line:

  * `cartpole`: microseconds per learn() call at Pearl's SAC_method configuration (obs 4, 2 actions, [64, 64] networks,
    batch 32) with training_rounds = 1 — PearlAgent calls learn() once per environment step — including the CPython RNG
    hand-over and the report read-back;
  * `stress`: gradient steps per second at obs 128, 16 actions, [256, 256] networks, batch 256, 1e5-transition ring, 512
    rounds per learn() call;
  * the CartPole round replayed 512 times in one call (the device time of a round, without the per-call host work);
  * kernels launched per round, and the host oracle at both shapes (one learn_batch per step, torch CPU threads as set);
  * the GPU's name and power limit, read in the same run.

Every timed shape is warmed up first; each measurement is repeated and reported as median, min and max.  CUDA events
bracket the timed loops (each learn() call ends in the report read-back, a device synchronisation).

    python tools/dsac_bench.py [--repeats 5] [--calls 400] [--rounds 512] [--oracle-steps 20]
"""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import pearl_b200  # noqa: E402
from oracle.dsac_oracle import OracleDiscreteSAC  # noqa: E402

SHAPES = {"cartpole": dict(obs=4, A=2, hidden=64, B=32, n=10_000), "stress": dict(obs=128, A=16, hidden=256, B=256, n=100_000)}


def gpu_info() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in out.split(",")]
    except Exception as e:  # pragma: no cover - nvidia-smi missing
        info["power_limit"] = f"unavailable ({type(e).__name__})"
    return info


def data(shape, seed=1):
    rng = np.random.Generator(np.random.PCG64(seed))
    n, obs, A = shape["n"], shape["obs"], shape["A"]
    st, ns = rng.standard_normal((n, obs), dtype=np.float32), rng.standard_normal((n, obs), dtype=np.float32)
    return st, rng.integers(0, A, size=n).astype(np.int64), rng.standard_normal(n, dtype=np.float32), ns, rng.random(n) < 0.05


def make_gpu(shape, rounds, arrays):
    st, ac, rw, ns, term = arrays
    buf = pearl_b200.B200ReplayBuffer(shape["n"], rng="python")
    buf.push_batch(torch.from_numpy(st), torch.from_numpy(ac).to(torch.int32), torch.from_numpy(rw), torch.from_numpy(ns),
                   torch.from_numpy(term), torch.zeros(shape["n"], dtype=torch.bool), max_number_actions=shape["A"])
    h = shape["hidden"]
    pl = pearl_b200.B200SoftActorCritic(state_dim=shape["obs"], n_actions=shape["A"], actor_hidden_dims=[h, h],
                                        critic_hidden_dims=[h, h], training_rounds=rounds, batch_size=shape["B"],
                                        actor_learning_rate=3e-4, critic_learning_rate=3e-4, seed=3)
    return pl, buf


def timed(fn, calls):
    """ms for `calls` calls of fn, between CUDA events (fn ends in a device synchronisation)."""
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(calls):
        fn()
    t1.record()
    t1.synchronize()
    return t0.elapsed_time(t1)


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": [round(x, 3) for x in xs]}


def oracle_step_ms(shape, arrays, steps):
    st, ac, rw, ns, term = arrays
    h = shape["hidden"]
    orc = OracleDiscreteSAC(shape["obs"], shape["A"], (h, h), (h, h), actor_lr=3e-4, critic_lr=3e-4)
    rnd = random.Random(5)

    def step():
        idx = rnd.sample(range(shape["n"]), shape["B"])
        t = lambda x: torch.from_numpy(x[idx])  # noqa: E731
        orc.learn_batch(dict(state=t(st), action=t(ac), reward=t(rw), next_state=t(ns), terminated=t(term)))
    for _ in range(3):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) * 1e3 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--calls", type=int, default=400, help="learn() calls per timed CartPole window")
    ap.add_argument("--rounds", type=int, default=512, help="rounds per learn() call at the stress shape")
    ap.add_argument("--oracle-steps", type=int, default=20)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    random.seed(0)
    res = {"gpu": gpu_info(), "torch_cpu_threads": torch.get_num_threads()}

    # ---- CartPole (SAC_method): one round per learn() call, as PearlAgent drives it
    shape = SHAPES["cartpole"]
    arrays = data(shape)
    pl, buf = make_gpu(shape, 1, arrays)
    for _ in range(50):
        pl.learn(buf)                                    # capture + warm-up
    pl.learn(buf)
    launches = int(pl._lib.prl_dsac_last_launches(pl._handle))
    us = [timed(lambda: pl.learn(buf), args.calls) * 1e3 / args.calls for _ in range(args.repeats)]
    # the same round replayed `rounds` times in one call: the device time of a round without the per-call host work
    pl._training_rounds = args.rounds
    pl.learn(buf)
    in_call = [timed(lambda: pl.learn(buf), 1) * 1e3 / args.rounds for _ in range(args.repeats)]
    orc_ms = oracle_step_ms(shape, arrays, args.oracle_steps * 10)
    res["cartpole"] = dict(shape=shape, training_rounds=1, us_per_learn_call=spread(us), launches_per_round=launches,
                           us_per_round_when_512_per_call=spread(in_call),
                           oracle_host_us_per_learn_call=round(orc_ms * 1e3, 1),
                           speedup_vs_host_oracle=round(orc_ms * 1e3 / statistics.median(us), 2))

    # ---- stress shape: many rounds per call
    shape = SHAPES["stress"]
    arrays = data(shape, seed=2)
    pl, buf = make_gpu(shape, args.rounds, arrays)
    pl.learn(buf)                                        # capture + warm-up
    launches = int(pl._lib.prl_dsac_last_launches(pl._handle)) // args.rounds
    sps = [args.rounds / (timed(lambda: pl.learn(buf), 1) / 1e3) for _ in range(args.repeats)]
    orc_ms = oracle_step_ms(shape, arrays, args.oracle_steps)
    res["stress"] = dict(shape=shape, rounds_per_call=args.rounds, grad_steps_per_s=spread(sps), us_per_grad_step=round(1e6 / statistics.median(sps), 2),
                         launches_per_round=launches, oracle_host_grad_steps_per_s=round(1e3 / orc_ms, 1),
                         speedup_vs_host_oracle=round(statistics.median(sps) * orc_ms / 1e3, 2))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
