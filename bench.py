#!/usr/bin/env python
"""bench.py — learner gradient-steps/sec (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one `learn()` call of the hot path (`ReplayBuffer.sample ->
PolicyLearner.learn()`) with `training_rounds = --rounds` gradient steps at
batch 256 on a 1e6-transition replay buffer (BASELINE cfg2: obs=128, A=16,
hidden [64,64]); value = K * rounds * n_gpus / max-over-ranks device time.
Timing: CUDA events on the launch stream around the K timed calls, barrier +
synchronize on both sides, W >= 3 warm-up calls; the 1.04 GB buffer is larger
than the 126 MB L2, so sampled rows come from HBM.

  value : buffer already resident in HBM, private device RNG stream
  e2e   : through the plugin API with HOST data — every step pushes `rounds`
          fresh transitions from pinned host memory (one per gradient step, the
          reference's online replay ratio), then learn() with the Python-RNG
          hand-off, and reads the loss report back (device->host)
  roofline      : the persistent learner kernel, algorithmic (factored) FLOPs
                  / its CUDA-event duration, vs MEASURED_PEAKS.json
  cpu_baseline  : the oracle port (oracle/pearl_oracle.py — eager PyTorch on the
                  host cores, the reference's own algorithm) on a bounded sample
`--impl reference` times that CPU port alone (rank 0), same metric/config.
N > 1: one process per GPU, each with its own buffer shard (see DESIGN.md §multi-GPU).
`--dump-outputs DIR` writes what the last timed call computed (rank 0) as .npy files in DIR; the
inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OBS, N_ACT, HIDDEN, BATCH = 128, 16, (64, 64), 256
METRIC = "learner gradient-steps/sec (batch=256, 1e6 replay)"


TC_DRAM_BYTES_PER_STEP = 1.165e6   # measured under ncu (4.042 GB read + 1.327 GB written over 144 learners x 32 rounds), profiles/r2b_k_dqn_tc_final_ncu_raw.csv


def flops_per_step(obs=OBS, A=N_ACT, H1=HIDDEN[0], H2=HIDDEN[1], B=BATCH, double=False):
    """Algorithmic FLOPs of one DQN gradient step (SURVEY.md §8d)."""
    D = obs + A
    P = H1 * D + H1 + H2 * H1 + H2 + H2 + 1
    f = 2 * (D * H1 + H1 * H2 + H2)
    f_s, f_r = 2 * obs * H1, 2 * (H1 * H2 + H2)
    as_written = B * f + B * (2 * f - 2 * D * H1) + B * A * f + 12 * P
    factored = B * (f_s + f_r) + B * (2 * (f_s + f_r) - f_s) + B * f_s + B * A * f_r + 12 * P
    if double:
        as_written += B * f
        factored += B * (f_s + f_r)
    return factored, as_written


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 9 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 9 and r[2].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower() == "active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": reasons, "samples": len(sm)}


def peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "hbm_gbs": d["hbm_gbs"], "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


# ----------------------------------------------------------------------------- CPU reference arm
def make_cpu_learner(n_store: int, rounds: int, threads: int):
    import torch
    from oracle.pearl_oracle import OracleDQN, OracleReplayBuffer
    import random
    torch.set_num_threads(threads)
    random.seed(1234)
    torch.manual_seed(1234)
    g = torch.Generator().manual_seed(4321)
    buf = OracleReplayBuffer(n_store, N_ACT)
    st = torch.randn((n_store, OBS), generator=g)
    ns = torch.randn((n_store, OBS), generator=g)
    rw = torch.randn(n_store, generator=g)
    tm = torch.rand(n_store, generator=g) < 0.02
    for i in range(n_store):
        buf.push(st[i], i % N_ACT, float(rw[i]), bool(tm[i]), False, ns[i])
    dqn = OracleDQN(OBS, N_ACT, HIDDEN, batch_size=BATCH, training_rounds=rounds, target_update_freq=10, tau=0.75)
    return buf, dqn


def _cpu_worker(wid, rounds, n_store, cmd_q, res_q):
    """One single-threaded learner process.  Commands: ("run", t_start, t_end) -> learn() calls back to back from t_start
    until t_end (wall clock), answer (wid, gradient steps done, seconds they took); ("stop",)."""
    import random
    random.seed(1234 + wid)
    buf, dqn = make_cpu_learner(n_store, rounds, 1)
    dqn.learn(buf)                         # warm-up call
    res_q.put((wid, "ready", 0.0))
    while True:
        cmd = cmd_q.get()
        if cmd[0] == "stop":
            return
        _, t_start, t_end = cmd
        while time.time() < t_start:
            time.sleep(0.001)
        t0, done = time.perf_counter(), 0
        while time.time() < t_end:
            dqn.learn(buf)
            done += rounds
        res_q.put((wid, done, time.perf_counter() - t0))


def cpu_reference(args, steps: int, warmup: int) -> dict:
    """The oracle port (the reference's own eager-PyTorch algorithm) on the host cores: independent single-threaded learner
    processes (its best configuration at batch 256).  Process counts {16, 32, 64, all} are swept; each measurement is a
    fixed WINDOW in which the chosen processes run learn() back to back and the aggregate is the sum of their own rates —
    a process that the (shared) host deschedules lowers its own share instead of defining the wall time of the whole
    configuration, which is what made the round-1 figure jump by 2x between runs.  Median of `steps` (>= 3) windows."""
    import multiprocessing as mp
    cores = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    nall = max(1, min(len(cores), args.ref_procs if args.ref_procs > 0 else len(cores)))
    rounds, n_store = args.ref_rounds, args.ref_capacity
    reps, window = max(3, steps), args.ref_window
    ctx = mp.get_context("spawn")
    res_q = ctx.Queue()
    cmd_qs = [ctx.Queue() for _ in range(nall)]
    procs = [ctx.Process(target=_cpu_worker, args=(w, rounds, n_store, cmd_qs[w], res_q), daemon=True) for w in range(nall)]
    t_start = time.perf_counter()
    for p in procs:
        p.start()
    for _ in range(nall):
        res_q.get(timeout=900)
    sweep = {}
    try:
        counts = sorted({c for c in (16, 32, 64) if c < nall} | {nall})
        for p in counts:
            ids = sorted({int(i * nall / p) for i in range(p)})
            aggs, per = [], []
            for _ in range(reps):
                t0 = time.time() + 0.2
                for w in ids:
                    cmd_qs[w].put(("run", t0, t0 + window))
                rates = []
                for _ in ids:
                    _, done, sec = res_q.get(timeout=600)
                    rates.append(done / sec if sec > 0 else 0.0)
                aggs.append(sum(rates))
                per.append(sum(rates) / len(rates))
            aggs.sort(); per.sort()
            sweep[str(p)] = {"aggregate": aggs[len(aggs) // 2], "per_process": per[len(per) // 2], "repeats": len(aggs),
                             "spread": [aggs[0], aggs[-1]]}
    finally:
        for q in cmd_qs:
            q.put(("stop",))
        for p in procs:
            p.join(timeout=10)
    best_p = max(sweep, key=lambda k: sweep[k]["aggregate"])
    best = sweep[best_p]
    return {"value": best["aggregate"], "unit": "gradient-steps/s", "cores": int(best_p), "kind": "port", "host_cores": len(cores),
            "per_process": best["per_process"], "sweep": sweep, "seconds": time.perf_counter() - t_start,
            "sample": f"independent single-threaded learner processes (not pinned: the host is shared), process counts "
                      f"{sorted(int(k) for k in sweep)} swept, {reps} windows of {window:g} s each in which every process runs learn() "
                      f"({rounds} rounds) back to back, aggregate = sum of the processes' own rates, median window per count, best count "
                      f"reported; batch {BATCH}, deque of {n_store} transitions each (1e6 Python pushes take minutes "
                      f"and do not change the per-step cost); reference = oracle/pearl_oracle.py (eager PyTorch, the reference's algorithm; "
                      f"facebookresearch/Pearl itself needs gymnasium, absent on the box)"}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference(args, steps=min(args.steps, 5), warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "gradient-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * args.ref_rounds * r["cores"] / r["value"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "DeepQLearning synthetic obs_dim=128 n_act=16, 1M replay, batch=256 (configs[1])",
                   "step": f"one learn() = {args.ref_rounds} gradient steps, in each of {r['cores']} independent learner processes",
                   "training_rounds_per_step": args.ref_rounds, "hidden": list(HIDDEN), "cpu_buffer": args.ref_capacity,
                   "same_config": False,
                   "differences": "the CPU learners sample from deques of 20k transitions (not 1e6) and run 40 rounds per learn() "
                                  "(the B200 arm: 512); neither changes the cost of a gradient step"},
        "cpu_baseline": r,
        "e2e": {"value": r["value"], "unit": "gradient-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- B200 arm
class Space:
    def __init__(self, n):
        import torch
        self.n = n
        self.actions = [torch.tensor([i]) for i in range(n)]
        self.actions_batch = torch.arange(n).view(n, 1)


def run_b200(args) -> None:
    import torch
    import torch.distributed as dist
    import pearl_b200

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cap, rounds = args.capacity, args.rounds
    torch.manual_seed(1234)
    gen = torch.Generator(device=dev).manual_seed(4321 + rank)

    def make_buffer(rng, seed):
        buf = pearl_b200.B200ReplayBuffer(cap, device=dev, rng=rng)
        chunk = 1 << 18
        for s in range(0, cap, chunk):
            m = min(chunk, cap - s)
            buf.push_batch(torch.randn((m, OBS), generator=gen, device=dev),
                           (torch.arange(s, s + m, device=dev) % N_ACT).to(torch.int32),
                           torch.randn(m, generator=gen, device=dev),
                           torch.randn((m, OBS), generator=gen, device=dev),
                           torch.rand(m, generator=gen, device=dev) < 0.02,
                           torch.zeros(m, dtype=torch.bool, device=dev), max_number_actions=N_ACT)
        buf.seed(seed)
        return buf

    def make_learner(engine, rds):
        return pearl_b200.B200DeepQLearning(
            state_dim=OBS, action_space=Space(N_ACT), hidden_dims=list(HIDDEN), learning_rate=1e-3,
            discount_factor=0.99, training_rounds=rds, batch_size=BATCH, target_update_freq=10,
            soft_update_tau=0.75, action_representation_module=pearl_b200.OneHotActionTensorRepresentationModule(N_ACT),
            max_rounds_per_call=max(rds, 1), rows_per_cta=args.rows_per_cta, engine=engine).to(dev)

    # ---- how many independent learners fit: one SM each, each with its OWN `cap`-transition replay
    from pearl_b200 import _lib
    sms = _lib.init(local).prl_sm_count()
    free_b, _ = torch.cuda.mem_get_info(dev)
    rec_bytes = 1040
    R = args.learners if args.learners > 0 else max(1, min(sms - 4, int((free_b - (10 << 30)) // (cap * rec_bytes))))
    bufs = [make_buffer("device", 1234 + 1000 * rank + i) for i in range(R)]
    learners = [make_learner("tc", rounds) for _ in range(R)]
    group = pearl_b200.B200LearnerGroup(learners, bufs)
    group.set_kernel_timing(True)
    W_ = max(args.warmup, 3)
    for _ in range(W_):
        group.learn()
    clocks = ClockSampler(local)
    barrier()
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    e0.record()
    for _ in range(args.steps):
        reports = group.learn()
        kernel_ms.append(group.last_kernel_ms())
    e1.record()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, reports, learners)
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = args.steps * rounds * R * world / (ms_max / 1e3)

    # ---- e2e: host data through the plugin API (every learner pushes `rounds` fresh transitions per step from pinned
    #      host memory; loss reports read back).  Every learner keeps its OWN device-resident MT19937 stream
    #      (rng="device"), like the reference's replicas, which are separate processes with their own `random` state
    #      (utils/scripts/benchmark.py:80-116); the CPython-global-stream hand-off of a single learner is measured in
    #      `single_learner_e2e`.
    n_new = rounds
    pin = lambda x: x.pin_memory()
    hg = torch.Generator().manual_seed(99 + rank)
    host = dict(state=pin(torch.randn((R, n_new, OBS), generator=hg)), next_state=pin(torch.randn((R, n_new, OBS), generator=hg)),
                reward=pin(torch.randn((R, n_new), generator=hg)), action=pin((torch.arange(R * n_new) % N_ACT).to(torch.int32).view(R, n_new)),
                term=pin((torch.rand((R, n_new), generator=hg) < 0.02).to(torch.uint8)), trunc=pin(torch.zeros((R, n_new), dtype=torch.uint8)))
    h2d = R * n_new * (2 * OBS * 4 + 4 + 4 + 1 + 1)
    d2h = R * rounds * 4

    def e2e_step():
        group.push_batch(host["state"], host["action"], host["reward"], host["next_state"], host["term"], host["trunc"])
        return group.learn()[0]["loss"][-1]

    for _ in range(2):
        e2e_step()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2e_steps = args.steps
    f0.record()
    for _ in range(e2e_steps):
        last_loss = e2e_step()
    f1.record()
    barrier()
    t2 = torch.tensor([f0.elapsed_time(f1)], device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = e2e_steps * rounds * R * world / (float(t2.item()) / 1e3)

    # ---- one sequential learner (cooperative fp32 SIMT kernel over 64 SMs + index producer CTA): latency view
    single = None
    if rank == 0 and not args.no_single:
        for b in bufs[1:]:
            b._storage = None
        sl = make_learner("simt", rounds)
        bufs[0]._rng_mode = "device"
        for _ in range(3):
            sl.learn(bufs[0])
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(5):
            sl.learn(bufs[0])
        s1.record()
        torch.cuda.synchronize()
        info = sl.launch_info()
        single = {"value": 5 * rounds / (s0.elapsed_time(s1) / 1e3), "unit": "gradient-steps/s",
                  "engine": f"k_dqn_learn: {info['ctas']} learner CTAs x {info['rows_per_cta']} rows + 1 index-producer CTA, fp32 SIMT"}
        # the same learner end to end as PearlAgent drives it: push from pinned host memory, CPython's global MT19937
        # stream handed to the device and back around learn(), loss report read back
        import random
        random.seed(1234)
        bufs[0]._rng_mode = "python"

        def single_e2e():
            bufs[0].push_batch(host["state"][0], host["action"][0], host["reward"][0], host["next_state"][0], host["term"][0], host["trunc"][0])
            return sl.learn(bufs[0])["loss"][-1]
        single_e2e()
        s0.record()
        for _ in range(5):
            single_e2e()
        s1.record()
        torch.cuda.synchronize()
        single["e2e"] = {"value": 5 * rounds / (s0.elapsed_time(s1) / 1e3), "unit": "gradient-steps/s",
                         "what": f"push_batch({n_new} from pinned host) + learn() incl. CPython RNG hand-off (2 x 2500 B) and loss report"}

    # ---- N > 1: ONE learner over a replay buffer sharded across the GPUs (SURVEY.md 8e), gradient-only exchange
    dp = None
    if world > 1 and not args.no_dp:
        launches_group = learners[0].launch_info()["launches"]
        del group
        for b in bufs:
            b._storage = None
        del bufs[:], learners[:]
        if single is not None:
            del sl
        torch.cuda.empty_cache()
        try:
            dp = dp_record(args, dev, rank, world, make_learner, barrier)
        except Exception as exc:
            dp = {"error": f"{type(exc).__name__}: {exc}"}
    else:
        launches_group = learners[0].launch_info()["launches"]

    if rank == 0:
        pk = peaks()
        fact, as_written = flops_per_step()
        k_ms = sum(kernel_ms) / len(kernel_ms)
        achieved = fact * rounds * R / (k_ms / 1e3) / 1e12
        peak = pk["bf16_tflops_sustained"] or pk["bf16_tflops"]
        line = {
            "metric": METRIC, "value": value, "unit": "gradient-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": W_, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 (3xTF32 tensor-core products, fp32 accumulate)", "data": "synthetic",
            "config": {"workload": "DeepQLearning synthetic obs_dim=128 n_act=16, 1M replay, batch=256 (configs[1])",
                       "step": f"one B200LearnerGroup.learn() = {rounds} sequential gradient steps of EACH of {R} independent "
                               f"learners per GPU (one SM per learner, each with its own {cap}-transition replay)",
                       "learners_per_gpu": R, "training_rounds_per_step": rounds, "hidden": list(HIDDEN),
                       "replay_capacity_per_learner": cap, "replay_bytes_per_gpu": R * cap * rec_bytes,
                       "l2": "inputs larger than L2 (no flush needed)",
                       "multi_gpu": "single GPU" if world == 1 else "value / e2e: independent learners sharded over the GPUs, no data-path collective; "
                                    "`dp`: ONE learner over a replay buffer sharded across the GPUs with the in-kernel NVLink gradient exchange",
                       "loss_last": last_loss},
            "e2e": {"value": e2e_value, "unit": "gradient-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "what": f"group.push_batch({n_new} fresh transitions per learner from pinned host memory, one library call) + group.learn() with the "
                            "loss reports read back; device-resident RNG streams"},
            "gpu_launches": args.steps * launches_group,
            "clocks": clk,
            "roofline": {"bound": "tensor", "kernel": "k_dqn_tc", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": TC_DRAM_BYTES_PER_STEP * rounds * R,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of the `ncu --set full` capture of k_dqn_tc in "
                                           "profiles/r2b_k_dqn_tc_final_ncu_raw.csv (1.17 MB per gradient step with 144 learners' parameters, AdamW state and operand "
                                           "tiles competing for L2; algorithmic gather 266 KB), "
                                           "scaled to the gradient steps of one bench launch",
                         "peak_source": f"{pk['source']} bf16 dense (sustained: kernel timed inside a long step)",
                         "flops_per_gradient_step_factored": fact, "flops_per_gradient_step_as_written": as_written,
                         "kernel_ms_per_launch": k_ms, "gradient_steps_per_launch": rounds * R,
                         "note": "3xTF32: every algorithmic FLOP is issued 3x on the TF32 pipe (half the bf16 rate), so the "
                                 "precision-matched ceiling is peak/6; frac_of_3xtf32_ceiling = %.3f" % (achieved / (peak / 6))},
            "single_learner": single,
        }
        if dp is not None:
            line["dp"] = dp
        if not args.no_cpu and world == 1:
            line["cpu_baseline"] = cpu_reference(args, steps=3, warmup=1)
        if world == 1 and not args.no_extras:
            del group, learners[:], bufs[:]
            if single is not None:
                del sl
            torch.cuda.empty_cache()
            try:
                line["other_paths"] = other_paths(dev, args)
            except Exception as exc:   # the headline line must survive a failure in the side measurements
                line["other_paths"] = {"error": f"{type(exc).__name__}: {exc}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(path: str, reports: list, learners: list) -> None:
    """What the caller of the last timed group.learn() receives, as float32 .npy files: loss.npy [k, rounds] (the
    reports) and parameters.npy / target_parameters.npy [k, P] (the online and target networks that call left).
    k is every learner unless that exceeds DUMP_BYTES; then it is the first k, which are the same learners
    with the same buffers and seeds whatever the learner count."""
    import numpy as np
    import torch
    rounds, p = len(reports[0]["loss"]), learners[0].flat_parameters.numel()
    k = max(1, min(len(learners), DUMP_BYTES // (4 * (rounds + 2 * p))))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "loss.npy"), np.asarray([r["loss"] for r in reports[:k]], dtype=np.float32))
    np.save(os.path.join(path, "parameters.npy"), torch.stack([l.flat_parameters for l in learners[:k]]).float().cpu().numpy())
    np.save(os.path.join(path, "target_parameters.npy"),
            torch.stack([l.flat_target_parameters for l in learners[:k]]).float().cpu().numpy())


def dp_record(args, dev, rank, world, make_learner, barrier) -> dict:
    """ONE DeepQLearning learner at world = N (SURVEY.md 8e): the 1e6-transition replay buffer is sharded by interleaved
    global write counter (rank g mod W), every rank runs the SAME MT19937 stream and so draws the same 256 global indices
    as one GPU would, works on the rows it owns, and the unnormalised partial gradients are summed by the in-kernel
    NVLink exchange before the (replicated, bit-identical) AdamW step.  In-run parity: rank 0 also holds the whole
    buffer and runs the ordinary single-GPU learner from the same weights and seed — indices must be bit-identical,
    parameters within 1e-4."""
    import ctypes as C

    import torch
    import torch.distributed as dist
    import pearl_b200
    from pearl_b200 import _lib
    cap = (args.capacity // world) * world
    rounds, par_rounds = args.dp_rounds, 32
    gen = torch.Generator(device=dev).manual_seed(777)           # the SAME stream on every rank: a replicated producer
    shard = pearl_b200.B200ReplayBuffer(cap // world, device=dev, rng="device")
    full = pearl_b200.B200ReplayBuffer(cap, device=dev, rng="device") if rank == 0 else None
    chunk = 1 << 18
    for s0 in range(0, cap, chunk):
        m = min(chunk, cap - s0)
        t = (torch.randn((m, OBS), generator=gen, device=dev), (torch.arange(s0, s0 + m, device=dev) % N_ACT).to(torch.int32),
             torch.randn(m, generator=gen, device=dev), torch.randn((m, OBS), generator=gen, device=dev),
             torch.rand(m, generator=gen, device=dev) < 0.02, torch.zeros(m, dtype=torch.bool, device=dev))
        shard.push_batch_sharded(rank, world, *t, max_number_actions=N_ACT)
        if full is not None:
            full.push_batch(*t, max_number_actions=N_ACT)
    shard.seed(4242)
    torch.manual_seed(4242)                                       # identical initial weights on every rank
    dp = make_learner("simt", rounds)
    w0, wt0 = dp.flat_parameters.clone(), dp.flat_target_parameters.clone()
    comm = pearl_b200.B200Communicator(w0.numel() + 1, dev)
    dp.set_communicator(comm)

    def clocked(learner, buf, calls):
        """(seconds per call over `calls` timed learn() calls, max over ranks; microseconds of the reduce + exchange + AdamW
        phase per round from the SM-clock stamps of CTA 0)"""
        for _ in range(2):
            learner.learn(buf)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            learner.learn(buf)
        e1.record()
        torch.cuda.synchronize()
        sec = e0.elapsed_time(e1) / 1e3 / calls
        st = torch.zeros((rounds, 16), dtype=torch.int64, device=dev)
        _lib.check(learner._libh.prl_dqn_set_profile(learner._handle, C.c_void_p(st.data_ptr())))
        learner.learn(buf)
        torch.cuda.synchronize()
        _lib.check(learner._libh.prl_dqn_set_profile(learner._handle, None))
        sc = st.cpu()[2:].double()
        clk_round = float((sc[1:, 0] - sc[:-1, 0]).mean())
        upd = float((sc[:, 11] - sc[:, 10]).mean()) / clk_round * sec / rounds * 1e6
        return sec, upd

    # ---- parity (before any timing call so that weights, step counts and streams line up)
    dp._training_rounds = par_rounds
    rep = dp.learn(shard, trace=True)
    flat = dp.flat_parameters.clone()
    same = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(same, flat)
    parity = {"ranks_bit_identical": all(torch.equal(x, same[0]) for x in same)}
    if rank == 0:
        solo = make_learner("simt", rounds)
        solo.flat_parameters.copy_(w0)
        solo.flat_target_parameters.copy_(wt0)
        full.seed(4242)
        solo._training_rounds = par_rounds
        srep = solo.learn(full, trace=True)
        want, got = solo.flat_parameters.double(), flat.double()
        bad = (got - want).abs() > 1e-6 + 1e-4 * want.abs()
        parity.update(indices_bit_identical=bool(torch.equal(rep["idx"], srep["idx"])), rounds=par_rounds,
                      params_max_rel_err=float(((got - want).abs() / (want.abs() + 1e-2)).max()),
                      params_outside_1e4=int(bad.sum()),
                      loss_max_rel_err=float(max(abs(a - b) / (abs(b) + 1e-6) for a, b in zip(rep["loss"], srep["loss"]))))
        ok = parity["ranks_bit_identical"] and parity["indices_bit_identical"] and parity["params_outside_1e4"] <= 4 and parity["loss_max_rel_err"] < 1e-4
        parity["verdict"] = "ok" if ok else "FAILED"
    # ---- timing
    dp._training_rounds = rounds
    sec, upd = clocked(dp, shard, args.steps)
    t = torch.tensor([sec], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = None
    if rank == 0:
        solo._training_rounds = rounds
        ssec, supd = clocked_solo(solo, full, args.steps, rounds, dev)
        out = {"what": f"ONE DeepQLearning learner, replay of {cap} transitions sharded over {world} GPUs (interleaved ownership), the same "
                       f"{BATCH} global indices per round on every rank, in-kernel NVLink exchange of the partial gradient (+ sum |q - y|)",
               "value": rounds / float(t.item()), "unit": "gradient-steps/s (one sequential learner)", "world": world,
               "rounds_per_call": rounds, "us_per_round": float(t.item()) / rounds * 1e6,
               "reduce_exchange_adamw_us_per_round": upd,
               "single_gpu": {"value": rounds / ssec, "us_per_round": ssec / rounds * 1e6, "reduce_adamw_us_per_round": supd},
               "exchange_us_per_round": upd - supd, "exchange_bytes_per_rank_per_round": 8 * (w0.numel() + 1) * world,
               "engine": "k_dqn_learn (cooperative fp32 SIMT kernel), exchange = 8-byte (value, sequence) stores into every peer's inbox",
               "parity": parity["verdict"], "parity_detail": parity}
    barrier()
    comm.close()
    return out


def clocked_solo(learner, buf, calls, rounds, dev):
    import ctypes as C

    import torch
    from pearl_b200 import _lib
    for _ in range(2):
        learner.learn(buf)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        learner.learn(buf)
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) / 1e3 / calls
    st = torch.zeros((rounds, 16), dtype=torch.int64, device=dev)
    _lib.check(learner._libh.prl_dqn_set_profile(learner._handle, C.c_void_p(st.data_ptr())))
    learner.learn(buf)
    torch.cuda.synchronize()
    _lib.check(learner._libh.prl_dqn_set_profile(learner._handle, None))
    sc = st.cpu()[2:].double()
    clk_round = float((sc[1:, 0] - sc[:-1, 0]).mean())
    return sec, float((sc[:, 11] - sc[:, 10]).mean()) / clk_round * sec / rounds * 1e6


def other_paths(dev, args) -> dict:
    """The remaining BASELINE configs on ONE GPU (rank 0, N = 1): SAC configs[2], PPO configs[3] (one GPU's rollout),
    prioritized DoubleDQN configs[4] (one GPU's shard).  Each: device-resident synthetic data, CUDA-event timing after a
    warm-up call, and the oracle port timed on the host cores on a bounded sample."""
    import time

    import torch
    import pearl_b200
    out = {}
    from pearl_b200 import _lib
    lib = _lib.init(dev.index if isinstance(dev, torch.device) and dev.index is not None else 0)
    gen = torch.Generator(device=dev).manual_seed(777)
    rn = lambda *shape: torch.randn(*shape, device=dev, generator=gen)
    cores = os.cpu_count() or 1

    def timed(fn, reps):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3 / reps

    def cpu_rate(step):
        """steps/s of `step` on the host, best of a few intra-op thread counts (eager PyTorch at these batch sizes does
        not scale to all cores; the best setting is what a user of the reference would run)."""
        best = (0.0, 1)
        for nt in sorted({1, min(8, cores), min(32, cores)}):
            torch.set_num_threads(nt)
            step()
            t0, k = time.perf_counter(), 0
            while time.perf_counter() - t0 < 1.5:
                step()
                k += 1
            best = max(best, (k / (time.perf_counter() - t0), nt))
        return best

    def section(fn):
        try:
            fn()
        except Exception as exc:   # one failing side measurement must not take the others (or the headline) with it
            out[fn.__name__] = {"error": f"{type(exc).__name__}: {exc}"}
        torch.cuda.empty_cache()

    # ---- SAC, Humanoid-shaped (configs[2]): obs 376, act 17, 1M replay, batch 512, [256, 256] networks
    def sac():
        obs, act, cap, B, R = 376, 17, 1_000_000, 512, 200
        buf = pearl_b200.B200ReplayBuffer(cap, device=dev, rng="device")
        buf.is_action_continuous = True
        for s0 in range(0, cap, 1 << 17):
            m = min(1 << 17, cap - s0)
            buf.push_batch(rn(m, obs), (torch.rand(m, act, device=dev, generator=gen) * 0.8 - 0.4), rn(m), rn(m, obs),
                           torch.rand(m, device=dev, generator=gen) < 0.01,
                           torch.zeros(m, dtype=torch.bool, device=dev))
        buf.seed(5)
        def run(engine):       # the engine is read when the learner's round is captured into its CUDA graph
            _lib.check(lib.prl_set_contraction_engine(engine))
            pl = pearl_b200.B200ContinuousSoftActorCritic(state_dim=obs, low=[-0.4] * act, high=[0.4] * act, actor_hidden_dims=[256, 256],
                                                           critic_hidden_dims=[256, 256], training_rounds=R, batch_size=B, device=dev, seed=1)
            sec = timed(lambda: pl.learn(buf), 3)
            return sec, int(pl._lib.prl_sac_last_launches(pl._handle)) // R
        sec, kps = run(1)
        sec2, _ = run(2)
        _lib.check(lib.prl_set_contraction_engine(1))
        out["sac"] = {"workload": "SAC continuous obs_dim=376 act_dim=17, 1M replay, batch=512 (configs[2])", "value": R / sec,
                      "unit": "gradient-steps/s (actor + twin-critic + entropy steps)", "us_per_step": sec / R * 1e6,
                      "kernels_per_step": kps,
                      "engine": "automatic contraction engine: at batch 512 every product runs on the fp32 SIMT tiles with the contraction "
                                "axis sliced over 4 warp groups (k_gemm<32,32,2,4>); CUDA-graph replay",
                      "with_tcgen05_contractions_forced": {"value": R / sec2, "us_per_step": sec2 / R * 1e6,
                                                           "note": "engine 2: every product on k_gemm_tc (3xTF32 tcgen05, 128 x 64 tiles); slower at this "
                                                                   "batch size, see profiles/r2_gemm_tc.md"}}
        del buf
        if not args.no_cpu:
            from oracle.sac_oracle import OracleSAC
            orc = OracleSAC(obs, act, (256, 256), (256, 256), [-0.4] * act, [0.4] * act)
            b = dict(state=torch.randn(B, obs), action=torch.rand(B, act) * 0.8 - 0.4, reward=torch.randn(B), next_state=torch.randn(B, obs),
                     terminated=torch.zeros(B, dtype=torch.bool))
            n1, n2 = torch.randn(B, act), torch.randn(B, act)
            rate, nt = cpu_rate(lambda: orc.learn_batch(b, n1, n2))
            out["sac"]["cpu_baseline"] = {"value": rate, "unit": "gradient-steps/s", "cores": nt, "host_cores": cores, "kind": "port",
                                          "sample": "1.5 s of learn_batch calls of oracle/sac_oracle.py on one fixed batch (no sampling cost), "
                                                    "best of 1 / 8 / 32 intra-op threads"}

    # ---- PPO (configs[3], one GPU's rollout): 64k-step rollout, obs 210, [256, 256] networks, batch 256
    def ppo():
        obs, A, n, B, R, hid = 210, 16, 65536, 256, 100, [64, 64]      # SURVEY.md §8 cfg4
        buf = pearl_b200.B200ReplayBuffer(n, device=dev, rng="device")
        buf.push_batch(rn(n, obs), torch.randint(0, A, (n,), device=dev, generator=gen).to(torch.int32), rn(n), rn(n, obs),
                       (torch.arange(n, device=dev) % 500) == 499, torch.zeros(n, dtype=torch.bool, device=dev), max_number_actions=A)
        buf.seed(6)
        def run(engine):
            _lib.check(lib.prl_set_contraction_engine(engine))
            pl = pearl_b200.B200ProximalPolicyOptimization(state_dim=obs, n_actions=A, actor_hidden_dims=hid, critic_hidden_dims=hid,
                                                            training_rounds=R, batch_size=B, epsilon=0.1, discount_factor=0.99,
                                                            trace_decay_param=0.95, device=dev, seed=2)
            pre = timed(lambda: pl.preprocess_replay_buffer(buf), 5)
            return pre, timed(lambda: pl.learn(buf), 3)
        pre_sec, sec = run(1)
        pre0, sec0 = run(0)
        _lib.check(lib.prl_set_contraction_engine(1))
        out["ppo"] = {"workload": "PPO 64k-step rollout obs_dim=210, 16 actions, [64,64] networks, GAE + clipped surrogate, batch=256 "
                                  "(configs[3] / SURVEY cfg4, one GPU)",
                      "preprocess_ms": pre_sec * 1e3, "preprocess_transitions_per_s": n / pre_sec,
                      "value": R / (sec - pre_sec), "unit": "gradient-steps/s (actor + critic steps, preprocessing excluded)",
                      "learn_ms": sec * 1e3, "training_rounds": R,
                      "engine": "rollout passes (8192 rows each): 3xTF32 tcgen05 contractions (k_gemm_tc); training rounds at batch 256: fp32 SIMT "
                                "tiles (k_gemm<32,32,2,*>), CUDA-graph replay",
                      "with_simt_contractions_only": {"value": R / (sec0 - pre0), "preprocess_ms": pre0 * 1e3}}
        del buf
        if not args.no_cpu:
            from oracle.ppo_oracle import OraclePPO
            orc = OraclePPO(obs, A, tuple(hid), tuple(hid), epsilon=0.1, batch_size=B, training_rounds=1)
            ns = 4096
            st, ac = torch.randn(ns + 1, obs), torch.randint(0, A, (ns,))
            torch.set_num_threads(min(8, cores))
            t0 = time.perf_counter()
            pre = orc.preprocess(st[:ns], ac, torch.randn(ns), torch.zeros(ns, dtype=torch.bool), torch.zeros(ns, dtype=torch.bool), st[ns])
            t_pre = time.perf_counter() - t0
            idx = torch.arange(B)
            rate, nt = cpu_rate(lambda: orc.learn_batch(st[idx], ac[idx], pre["gae"][idx], pre["lam_return"][idx], pre["action_probs"][idx]))
            out["ppo"]["cpu_baseline"] = {"value": rate, "unit": "gradient-steps/s", "cores": nt, "host_cores": cores, "kind": "port",
                                          "preprocess_transitions_per_s": ns / t_pre,
                                          "sample": f"preprocess of a {ns}-step rollout (8 threads) + 1.5 s of learn_batch calls of "
                                                    "oracle/ppo_oracle.py, best of 1 / 8 / 32 intra-op threads"}

    # ---- prioritized DoubleDQN (configs[4], one GPU's shard): obs 512, 16 actions, batch 256, sum / min trees in HBM
    def prioritized_ddqn():
        obs, A, B, R = 512, 16, 256, 200
        free_b, _ = torch.cuda.mem_get_info(dev)
        cap = 4_000_000 if free_b > (40 << 30) else 500_000
        buf = pearl_b200.B200PrioritizedReplayBuffer(cap, device=dev, seed=11)
        for s0 in range(0, cap, 1 << 17):
            m = min(1 << 17, cap - s0)
            buf.push_batch(rn(m, obs), (torch.arange(s0, s0 + m, device=dev) % A).to(torch.int32), rn(m), rn(m, obs),
                           torch.rand(m, device=dev, generator=gen) < 0.02, torch.zeros(m, dtype=torch.bool, device=dev), max_number_actions=A)
        ddqn = pearl_b200.B200DoubleDQN(state_dim=obs, action_space=Space(A), hidden_dims=[64, 64], training_rounds=R, batch_size=B,
                                        target_update_freq=10, soft_update_tau=0.75,
                                        action_representation_module=pearl_b200.OneHotActionTensorRepresentationModule(A),
                                        max_rounds_per_call=R).to(dev)
        sec = timed(lambda: ddqn.learn(buf), 3)
        out["prioritized_ddqn"] = {"workload": f"prioritized segment-tree replay {cap} x obs_dim=512, DoubleDQN [64,64], batch=256 (configs[4] / SURVEY cfg5 on one GPU)",
                                   "value": R / sec, "unit": "gradient-steps/s (stratified tree draw + weighted step + priority update)",
                                   "us_per_step": sec / R * 1e6, "replay_bytes": cap * buf.record_bytes}
        del ddqn, buf
    # ---- the HBM-side kernels of the path (write side, sample() = indices + gather, GAE scan, prioritized draw / update):
    #      algorithmic bytes / CUDA-event time against the measured copy bandwidth
    def hbm_paths():
        pk = peaks()
        hbm = pk["hbm_gbs"]
        rec = {}

        def entry(name, bytes_per_call, sec, note):
            gbs = bytes_per_call / sec / 1e9
            rec[name] = {"us_per_call": sec * 1e6, "algorithmic_bytes_per_call": bytes_per_call, "achieved_gbs": gbs,
                         "peak_gbs": hbm, "frac": gbs / hbm, "peak_source": f"{pk['source']} copy bandwidth", "note": note}

        n = 1 << 18
        cap = 1 << 20
        buf = pearl_b200.B200ReplayBuffer(cap, device=dev, rng="device")
        st, ns, rw = rn(n, OBS), rn(n, OBS), rn(n)
        ac = (torch.arange(n, device=dev) % N_ACT).to(torch.int32)
        tm = torch.rand(n, device=dev, generator=gen) < 0.02
        tr = torch.zeros(n, dtype=torch.bool, device=dev)
        push = lambda: buf.push_batch(st, ac, rw, ns, tm, tr, max_number_actions=N_ACT)
        for _ in range(4):
            push()                                                   # fills the ring
        rbytes = buf.record_bytes
        entry("push_batch_device (k_pack_records)", n * (2 * OBS * 4 + 4 + 4 + 1 + 1 + rbytes), timed(push, 10),
              f"{n} transitions per call: struct-of-arrays inputs read once, {rbytes}-byte records written once")
        hst = [x.cpu().pin_memory() for x in (st, ac, rw, ns, tm, tr)]
        hpush = lambda: (buf.push_batch(*hst, max_number_actions=N_ACT), torch.cuda.synchronize())
        sec = timed(hpush, 5)
        rec["push_batch_host (pack on the host + cudaMemcpyAsync)"] = {
            "us_per_call": sec * 1e6, "h2d_bytes_per_call": n * rbytes, "achieved_gbs": n * rbytes / sec / 1e9,
            "note": "bound by the host-side packing threads and PCIe, not HBM; listed for completeness"}
        buf.seed(3)
        k = 1 << 16
        slots = torch.randint(0, cap, (k,), device=dev, generator=gen).to(torch.int32)
        entry("gather (k_gather, sample()'s collation)", k * (rbytes + 2 * OBS * 4 + 8 + 4 + 2 + 16 * 5), timed(lambda: buf._gather_slots(slots), 20),
              f"{k} random records -> TransitionBatch fields (records read once, every field written once)")
        sec = timed(lambda: buf.sample(BATCH), 20)
        rec["sample(256) (k_sample_indices + k_gather + TransitionBatch)"] = {
            "us_per_call": sec * 1e6, "note": "latency-bound at batch 256: MT19937-exact index stream (one warp resolves rejections in order) + "
                                              "one gather launch + torch allocations of the batch fields; 266 KB moved"}
        del buf
        torch.cuda.empty_cache()
        from pearl_b200.ppo import gae_and_lambda_returns
        ng = 1 << 24
        vals, rws = rn(ng), rn(ng)
        te = ((torch.arange(ng, device=dev) % 500) == 499).to(torch.uint8)   # the flags as the rollout kernels hold them
        tu = torch.zeros(ng, dtype=torch.uint8, device=dev)
        entry("k_ppo_gae (GAE + lambda returns)", ng * 18, timed(lambda: gae_and_lambda_returns(vals, 0.1, rws, te, tu, 0.99, 0.95), 10),
              f"{ng} transitions, episodes of 500: 10 bytes read + 8 written per transition (the reference's Python loop: ppo.py:271-293)")
        del vals, rws, te, tu
        torch.cuda.empty_cache()
        capp = 1 << 22
        pb = pearl_b200.B200PrioritizedReplayBuffer(capp, device=dev, seed=3)
        pb.push_batch(rn(1 << 16, 8), torch.zeros(1 << 16, dtype=torch.int32, device=dev), rn(1 << 16), rn(1 << 16, 8),
                      torch.zeros(1 << 16, dtype=torch.bool, device=dev), torch.zeros(1 << 16, dtype=torch.bool, device=dev), max_number_actions=2)
        sl, _ = pb.sample_prioritized(BATCH)
        td = torch.rand(BATCH, device=dev, generator=gen)
        lv = 22
        entry("k_per_sample (256 stratified sum-tree draws)", BATCH * 2 * lv * 4, timed(lambda: pb.sample_prioritized(BATCH), 50),
              "latency-bound by construction: 22 dependent tree reads per draw (top 11 levels from shared memory)")
        entry("k_per_update (256 priority updates)", BATCH * 4 * lv * 4, timed(lambda: pb.update_priorities(sl, td), 50),
              "latency-bound: 22 levels rewritten bottom-up per updated leaf")
        out["hbm_side_kernels"] = rec

    for fn in (sac, ppo, prioritized_ddqn, hbm_paths):
        section(fn)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rounds", type=int, default=512, help="training_rounds per learn() call")
    ap.add_argument("--learners", type=int, default=0, help="independent learners per GPU (0 = one per SM that fits in memory)")
    ap.add_argument("--no-single", action="store_true", help="skip the single-sequential-learner latency measurement")
    ap.add_argument("--ref-procs", type=int, default=0, help="CPU reference processes (0 = one per host core)")
    ap.add_argument("--capacity", type=int, default=1_000_000)
    ap.add_argument("--rows-per-cta", type=int, default=0)
    ap.add_argument("--ref-rounds", type=int, default=40)
    ap.add_argument("--ref-window", type=float, default=3.0, help="seconds per timed window of the CPU reference arm")
    ap.add_argument("--ref-capacity", type=int, default=20_000)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-dp", action="store_true", help="N > 1: skip the sharded-replay single-learner record")
    ap.add_argument("--dp-rounds", type=int, default=256)
    ap.add_argument("--no-extras", action="store_true", help="skip the SAC / PPO / prioritized-replay side measurements")
    ap.add_argument("--extras-only", action="store_true", help="developer: run only the side measurements on cuda:0")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the losses and parameters of the last timed step to DIR/*.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries the ONE JSON line and nothing else: libraries that print there (NCCL's version banner, torch warnings
    # routed to fd 1) are sent to stderr for the duration of the run; print() is bound to the saved descriptor
    global print
    sys.stdout.flush()
    real_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    import builtins

    def print(*a, **kw):   # noqa: A001
        kw.setdefault("file", real_out)
        builtins.print(*a, **kw)
        real_out.flush()
    if args.extras_only:
        import torch
        torch.cuda.set_device(0)
        print(json.dumps({"other_paths": other_paths(torch.device("cuda", 0), args)}), flush=True)
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
