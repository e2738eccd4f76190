#!/usr/bin/env python
"""bench.py -- learner updates/sec of the Rainbow hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C2|C3|C4] [--dump-outputs DIR]

One step = `dqn.reset_noise(); dqn.learn(mem)` (reference main.py:150-151,163-164) on synthetic 84x84x4
transitions.  N=1 workload = BASELINE.json configs[1] ("C2": 1M-transition replay in HBM, batch 32, 51
atoms, n=3, canonical net).  N>1 (torchrun, one rank per GPU): every rank owns a private replay + stream
and the ranks exchange only the flat gradient (NCCL all-reduce) -> weak scaling, value = per-rank batch-32
updates summed over ranks per second.

Printed JSON (one line, rank 0): value (inputs resident in HBM, CUDA-graph replay), e2e (through the public
Agent/ReplayMemory API with HOST frames: 4 appends from pinned memory + update + loss read-back per step,
like main.py's replay_frequency=4 loop), roofline of the dominant hand-written kernel (CUDA events around
the kernel, live), cpu_baseline (oracle port of the reference's CPU path on this box's cores).

--impl reference: the CPU arm (oracle/learner.py port of the reference path, all host threads), same
metric/config/unit; under torchrun only rank 0 runs it.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    # name: capacity, batch, n, architecture, hidden   (SURVEY.md 8(d))
    "C2": dict(cap=1_000_000, B=32, n=3, arch="canonical", hidden=512),
    "C3": dict(cap=100_000, B=32, n=20, arch="data-efficient", hidden=256),
    "C4": dict(cap=1_000_000, B=512, n=3, arch="canonical", hidden=512),
}
ACTIONS = 6
REPLAY_FREQUENCY = 4  # main.py:37 -- env steps (appends) per learner update in the e2e loop


def make_args(cfg, device, peer_optimizer=False):
    return argparse.Namespace(peer_optimizer=peer_optimizer, device=device, history_length=4, discount=0.99, multi_step=cfg["n"], priority_weight=0.4,
                              priority_exponent=0.5, atoms=51, V_min=-10.0, V_max=10.0, batch_size=cfg["B"],
                              norm_clip=10.0, model=None, learning_rate=6.25e-5, adam_eps=1.5e-4,
                              architecture=cfg["arch"], hidden_size=cfg["hidden"], noisy_std=0.1, cuda_graph=True)


class FakeEnv:
    def action_space(self):
        return ACTIONS


def synthetic_meta(cap, seed):
    """BASELINE.md synthetic fill (everything except the frames), identical for both arms."""
    rs = np.random.RandomState(seed)
    timestep = (np.arange(cap) % 1000).astype(np.int32)
    return dict(timestep=timestep, nonterminal=(timestep != 999).astype(np.uint8),
                action=rs.randint(0, ACTIONS, cap).astype(np.int32), reward=rs.randint(-1, 2, cap).astype(np.float32),
                priority=(rs.uniform(0, 1, cap) ** 0.5 + 1e-3).astype(np.float32), head=12345 % cap)


T0 = time.time()


def log(*a):
    print(f"[bench {time.time() - T0:7.1f}s]", *a, file=sys.stderr, flush=True)


def host_threads():
    """Threads the CPU arm may really use: affinity mask and cgroup CPU quota, not the host's core count
    (hundreds of OpenMP threads inside a small cgroup quota would crawl)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, min(n, 64))


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed regions run."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.max_mhz, self.ok = index, period, [], set(), None, False
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop_evt.wait(self.period)

    def finish(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
def run_cpu_port(cfg, updates, warmup, with_appends, seed=1, budget_s=None):
    """The reference's CPU path (oracle port) on this box's cores: returns updates/s over at most `updates`
    updates (fewer if `budget_s` seconds run out first; at least 3)."""
    import torch

    from oracle.learner import OracleLearner, OracleReplay
    torch.set_num_threads(host_threads())
    log(f"cpu port: os.cpu_count={os.cpu_count()} usable threads={host_threads()} torch threads={torch.get_num_threads()}")
    torch.manual_seed(0)
    np.random.seed(123)
    cap = cfg["cap"]
    args = make_args(cfg, "cpu")
    mem = OracleReplay(cap, 4, cfg["n"], 0.99, 0.4, 0.5)
    meta = synthetic_meta(cap, seed)
    t = mem.tree
    t.timestep[:], t.nonterminal[:], t.action[:], t.reward[:] = meta["timestep"], meta["nonterminal"], meta["action"], meta["reward"]
    # frame bytes do not affect timing; a cheap non-constant fill touches every page of the 7 GB ring
    pat = np.random.RandomState(seed).randint(0, 256, (1024, 7056), dtype=np.uint8)
    for s in range(0, cap, 1024):
        e = min(cap, s + 1024)
        t.frames[s:e] = pat[:e - s]
    for s in range(0, cap, 4096):
        e = min(cap, s + 4096)
        t.update(np.arange(s, e) + t.tree_start, meta["priority"][s:e])
    t.index, t.full = meta["head"], True
    learner = OracleLearner(args, ACTIONS)
    frame_src = [torch.rand(4, 84, 84) for _ in range(8)]

    def step(i):
        if with_appends:
            for j in range(REPLAY_FREQUENCY):
                mem.append(frame_src[(i + j) % 8].numpy(), (i + j) % ACTIONS, float((i % 3) - 1), (i * 4 + j) % 1000 == 999)
        learner.reset_noise()
        learner.learn(mem)

    log("cpu port: ring filled, warm-up")
    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    done = 0
    while done < updates:
        step(warmup + done)
        done += 1
        if budget_s is not None and done >= 3 and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    log(f"cpu port: {done} updates in {dt:.1f}s")
    return done / dt, dt, torch.get_num_threads(), done


def run_cpu_reference(cfg, updates, warmup, budget_s, also_gpu=None):
    """The UNMODIFIED reference (oracle/_ref, `make -C oracle _ref`) on this box's host cores, same synthetic workload:
    returns (updates/s, seconds, threads, updates done, extra) or None when oracle/_ref is not there.  `also_gpu`: a CUDA
    device -> additionally time the reference's own GPU path (args.device = cuda, eager PyTorch, host numpy replay) on the
    same replay object for `extra["reference_gpu_path"]`."""
    import torch

    from oracle import ref_arm
    if not ref_arm.available():
        return None
    torch.set_num_threads(host_threads())
    log(f"reference arm: os.cpu_count={os.cpu_count()} usable threads={host_threads()} torch threads={torch.get_num_threads()}")
    torch.manual_seed(0)
    np.random.seed(123)
    sess = ref_arm.Session(make_args(cfg, torch.device("cpu")), ACTIONS, cfg["cap"], synthetic_meta(cfg["cap"], 1), log=log)
    ups, dt, done = sess.time("cpu", updates, warmup, with_appends=True, replay_frequency=REPLAY_FREQUENCY, budget_s=budget_s)
    log(f"reference arm (cpu): {done} updates in {dt:.1f}s")
    extra = {}
    if also_gpu is not None:
        flags = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = True, False, False  # torch's stock settings
        try:
            g_ups, g_dt, g_done = sess.time(also_gpu, 200, 5, with_appends=True, replay_frequency=REPLAY_FREQUENCY, budget_s=12)
        finally:
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = flags
        log(f"reference arm (cuda, eager): {g_done} updates in {g_dt:.1f}s")
        extra["reference_gpu_path"] = {"value": g_ups, "unit": "updates/s", "ms_per_step": 1e3 * g_dt / g_done,
                                       "what": f"the unmodified reference with args.device=cuda (eager PyTorch, stock torch flags, numpy sum tree on the host, "
                                               f"per-update H2D of the batch and D2H of the losses), {g_done} updates each preceded by {REPLAY_FREQUENCY} appends"}
    return ups, dt, torch.get_num_threads(), done, extra


def cpu_arm(cfg, updates, warmup, budget_s, also_gpu=None):
    """(value, seconds, threads, updates done, kind, sample text, extra): the reference itself when it travelled with the
    snapshot (oracle/_ref), otherwise the oracle port."""
    r = run_cpu_reference(cfg, updates, warmup, budget_s, also_gpu)
    if r is not None:
        ups, dt, threads, done, extra = r
        return ups, dt, threads, done, "reference", (
            f"{done} updates of the same workload (each preceded by {REPLAY_FREQUENCY} appends) after {warmup} warm-up updates, {dt:.1f} s; "
            f"UNMODIFIED reference modules (oracle/_ref/reference_modules.zip: memory.py, agent.py, model.py, sha256-checked) on torch-CPU with "
            f"{threads} threads; the 1M-record replay object is assembled without the reference's 242 s list constructor"), extra
    ups, dt, threads, done = run_cpu_port(cfg, updates, warmup, with_appends=True, budget_s=budget_s)
    return ups, dt, threads, done, "port", (
        f"{done} updates of the same workload (each preceded by {REPLAY_FREQUENCY} appends) after {warmup} warm-up updates, {dt:.1f} s; "
        f"oracle port (oracle/_ref absent): replay tree/gather in C, nets in torch-CPU with {threads} threads"), {}


def reference_arm(opts, cfg, rank):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores (the unmodified modules
    from oracle/_ref when present -- kind "reference" --, else the oracle port -- kind "port")."""
    if rank != 0:
        return
    per_step = 1  # one update (preceded by its 4 appends) per bench "step", exactly like our arm's e2e step
    ups, dt, threads, total, kind, sample, _ = cpu_arm(cfg, opts.steps * per_step, min(5, max(3, opts.warmup)), budget_s=150)
    line = {"impl": "reference", "metric": "learner updates/sec (batch32, 1M buffer, 51 atoms)", "value": ups,
            "unit": "updates/s", "n_gpus": opts.gpus, "steps": total, "warmup": opts.warmup,   # the 150 s budget may stop it early
            "ms_per_step": 1e3 * dt / total, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "gpu_launches": 0,
            "config": workload_config(opts.config, cfg, opts.gpus),
            "cpu_baseline": {"value": ups, "unit": "updates/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": ups, "unit": "updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(name, cfg, gpus, param_elems=None):
    if param_elems is None:
        l2 = "host arm: no GPU cache involved"
    else:
        # distinct device addresses one update walks: online + target parameters, the gradient, both Adam moments, the [s; s'] batch
        mb = (5 * param_elems * 4 + 2 * cfg["B"] * 4 * 84 * 84 * 4) / 1e6
        l2 = (f"no explicit flush: an update walks {mb:.0f} MB of distinct addresses (two parameter sets, gradient, two Adam moments, "
              f"the state batch) -- {'more' if mb > 126 else 'LESS'} than the 126 MB L2"
              f"{'' if mb > 126 else ' (this configuration stays L2-resident, in training as here)'} -- plus {2 * cfg['B']} random "
              f"4-frame states of a {cfg['cap'] * 7056 / 1e9:.1f} GB frame ring")
    return {"workload": f"{name}: synthetic 84x84x4 transitions, {cfg['cap']}-transition replay per GPU, batch {cfg['B']} per GPU, "
                        f"51 atoms, n={cfg['n']}, {cfg['arch']} net hidden {cfg['hidden']}, {ACTIONS} actions",
            "global_batch": cfg["B"] * gpus, "parallelism": f"dp{gpus} (independent replay per rank, grad all-reduce)" if gpus > 1 else "single",
            "l2": l2}


# ------------------------------------------------------------------------------------------------
def algorithmic_bytes(cfg, P, noisy_elems):
    """SURVEY.md 8(d) per-launch algorithmic bytes of each hand-written kernel."""
    B, n, H, F, Z, A = cfg["B"], cfg["n"], 4, 7056, 51, ACTIONS
    K1 = 3136 if cfg["arch"] == "canonical" else 576
    head = dict(K1=K1, H=cfg["hidden"], N2=Z * (1 + A), w1=2 * cfg["hidden"] * K1, w2=Z * (1 + A) * cfg["hidden"])
    cap = cfg["cap"]
    L = (cap - 1).bit_length()
    return {
        "tree_sample": B * (L + 1) * 4 + B * 20,
        "gather": B * min(H + n, 2 * H) * F + B * ((H + n) * 4 + n * 4 + 5) + 2 * B * H * F * 4 + B * 16,
        "c51": 3 * B * A * Z * 4 + B * 20 + Z * 4 + B * A * Z * 4 + B * 8,
        "tree_update": B * 12 + B * 4 + B * L * 12,
        "noisy_resample": noisy_elems * 4,          # per net
        "sqnorm": P * 4,                            # read grad
        "clip_adam": 7 * P * 4,                     # read p,g,m,v ; write p,m,v
        "append": F * 4 + F + 13 + L * 8,
        # fused head (canonical: K1 3136, H 512): weights mu+sigma read once per launch + activations in/out
        "head_fc1": head["w1"] * 2 * 4 + 2 * B * head["K1"] * 4 + 2 * B * 2 * head["H"] * 4,            # online pass (2B rows)
        "head_fc2": head["w2"] * 2 * 4 + 2 * B * 2 * head["H"] * 4 + 2 * B * head["N2"] * 4,
        "head_bwd1": head["w1"] * 2 * 4 * 2 + B * (head["K1"] + 2 * head["H"]) * 4 + B * head["K1"] * 4,  # read mu,sigma; write both grads
        "head_dh": head["w2"] * 2 * 4 + B * (head["N2"] + 2 * 2 * head["H"]) * 4,
        "head_wgrad2": head["w2"] * 2 * 4 + B * (head["N2"] + 2 * head["H"]) * 4,
        "c51_dueling": 3 * B * head["N2"] * 4 + B * 20 + Z * 4 + B * head["N2"] * 4 + B * 4,
        "noise_factors": (head["K1"] * 2 + head["H"] * 4 + head["N2"]) * 4,
    }


def csrc_sha256(files=None):
    """sha256 over rainbow_b200/csrc/ (all .cu / .cuh, or the given file names, in sorted order)."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "rainbow_b200", "csrc")
    for fn in sorted(os.listdir(d) if files is None else files):
        if fn.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(d, fn), "rb").read())
    return h.hexdigest()


# which translation unit (+ the shared header) a kernel's DRAM-traffic capture depends on
KERNEL_SOURCES = {"head_fc1": ["rb_head_tc.cu"], "head_reduce1": ["rb_head_tc.cu"], "head_fc2": ["rb_head.cu"], "head_dh": ["rb_head.cu"],
                  "head_bwd1": ["rb_head.cu"], "head_wgrad2": ["rb_head.cu"], "bias_grad": ["rb_head.cu"], "conv_wgrad": ["rb_head.cu"],
                  "noise_factors": ["rb_head.cu"]}


def kernel_source_sha(name):
    return csrc_sha256(sorted(KERNEL_SOURCES.get(name, ["rb_kernels.cu"]) + ["rb_internal.cuh"]))


DUMP_LIMIT_BYTES = 64 << 20


def last_step_outputs(agent, mem):
    """What the last `reset_noise(); learn(mem)` left its caller, as host arrays: the per-sample losses, the tree indices
    of the batch and the priorities written back for them, and every online-net parameter after the optimiser step
    (6.9 M floats at C2 / C4)."""
    import torch
    idx = mem._last.tree_idx
    out = {"loss": agent.last_loss, "tree_idx": idx.to(torch.float64), "priority": mem.transitions.tree[idx]}
    out.update(("param." + name, p) for name, p in agent.online_net.named_parameters())
    return {k: v.detach().cpu().numpy() for k, v in out.items()}


def dump_outputs(directory, arrays):
    """--dump-outputs: DIR/<name>.npy for every array (float32, or float64 for the indices)."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(directory, name + ".npy"), a)
    log(f"dumped {len(arrays)} arrays ({total / 1e6:.1f} MB) of the last timed step to {directory}")


def ours(opts, cfg, rank, world, local):
    import torch

    from rainbow_b200 import _lib
    from rainbow_b200.agent import Agent
    from rainbow_b200.dist import GradSync, shard_seed
    from rainbow_b200.memory import ReplayMemory

    torch.backends.cudnn.allow_tf32 = False        # the reference computes in true fp32
    torch.backends.cuda.matmul.allow_tf32 = False
    # The conv algorithms cuDNN picks by timing for these shapes accumulate in a run-dependent order, and the prioritized
    # replay turns such last-bit differences into different batches within a few hundred updates.  A run whose outputs
    # are dumped therefore uses cuDNN's deterministic algorithms (heuristic choice): it reproduces bit for bit, and is
    # slower (B200 at 1000 W, C2: 485 against 323 us per update).
    deterministic = bool(opts.dump_outputs)
    torch.backends.cudnn.benchmark = not deterministic
    torch.backends.cudnn.deterministic = deterministic
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    torch.manual_seed(shard_seed(0, rank))
    np.random.seed(123 + rank)
    peer = False if (world == 1 or opts.nccl or os.environ.get("RB_PEER", "1") == "0") else (True if opts.peer_optimizer else "auto")
    args = make_args(cfg, dev, peer_optimizer=peer)
    cap, B = cfg["cap"], cfg["B"]

    # defer_appends: the e2e loop's 4 appends per update are written by ONE rb_append_batch launch that reads the frames in
    # place from the replay's pinned staging ring (SURVEY 8(f).2); the `value` loop never appends, so it is unaffected
    mem = ReplayMemory(args, cap, seed=shard_seed(17, rank), defer_appends=True)
    meta = synthetic_meta(cap, 1 + rank)
    tr = mem.transitions
    tr.load_arrays(timestep=meta["timestep"], action=meta["action"], reward=meta["reward"], nonterminal=meta["nonterminal"],
                   index=meta["head"], full=True, t_episode=int(meta["timestep"][meta["head"] - 1]) + 1)
    gen = torch.Generator(device=dev).manual_seed(1 + rank)
    for s in range(0, cap, 65536):
        e = min(cap, s + 65536)
        tr.frames[s:e] = torch.randint(0, 256, (e - s, 7056), dtype=torch.uint8, device=dev, generator=gen)
    pri = torch.from_numpy(meta["priority"]).to(dev)
    leaf = torch.arange(cap, device=dev) + tr.tree_start
    for s in range(0, cap, 1024):
        tr.update(leaf[s:s + 1024], pri[s:s + 1024])
    log("replay filled")
    agent = Agent(args, FakeEnv())
    sync = GradSync()

    def step():
        agent.reset_noise()
        agent.learn(mem)

    def barrier():
        if sync.enabled:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(k):
            fn(i)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        sync.max_(ms)
        barrier()
        return float(ms.item())

    W, K = max(3, opts.warmup), opts.steps
    for _ in range(Agent.GRAPH_WARMUP + 2):   # eager warm-up + graph capture happen here, outside any timing
        step()
    for _ in range(W):
        step()
    mem.check_last_sample()
    log("warm-up + graph capture done")
    if world > 1:
        import faulthandler
        faulthandler.cancel_dump_traceback_later()

    if opts.profile_steps:   # ncu window (use with `ncu --profile-from-start off`): numbers under a profiler are never reported
        mode = opts.profile_mode
        if mode == "eager":
            agent.use_cuda_graph = False
            step()
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        for i in range(opts.profile_steps):
            if mode == "e2e":
                for j in range(REPLAY_FREQUENCY):
                    mem.append(torch.rand(4, 84, 84).pin_memory(), j, 0.0, False)
            step()
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return

    sampler = ClockSampler(local)
    sampler.start()
    # ---- value: inputs resident in HBM, K updates --------------------------------------------------
    ms_value = timed(lambda i: step(), K)
    log(f"value region: {ms_value / K:.3f} ms/step")
    if opts.dump_outputs and rank == 0:   # before the e2e region below moves the parameters and the tree on
        dump_outputs(opts.dump_outputs, last_step_outputs(agent, mem))
    # ---- e2e: public API with host frames ------------------------------------------------------------
    host_frames = [torch.rand(4, 84, 84).pin_memory() for _ in range(8)]
    loss_host = [torch.empty(B, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_evt = [torch.cuda.Event(), torch.cuda.Event()]
    loss_seen = {"sum": 0.0, "n": 0, "pending": [False, False]}

    def consume(slot):
        if loss_seen["pending"][slot]:
            loss_evt[slot].synchronize()                 # the host really reads every step's loss ...
            loss_seen["sum"] += float(loss_host[slot].sum())
            loss_seen["n"] += 1
            loss_seen["pending"][slot] = False

    def e2e_step(i):
        for j in range(REPLAY_FREQUENCY):
            mem.append(host_frames[(i + j) % 8], (i + j) % ACTIONS, float((i % 3) - 1), (i * 4 + j) % 1000 == 999)
        step()
        slot = i & 1
        consume(slot)                                    # ... one step behind the GPU (double-buffered pinned copy),
        loss_host[slot].copy_(agent.last_loss, non_blocking=True)   # so the launch thread is not stalled every step
        loss_evt[slot].record()
        loss_seen["pending"][slot] = True

    for i in range(W):
        e2e_step(i)
    def e2e_region(i):
        e2e_step(i)
        if i == K - 1:                                   # drain inside the timed region: every loss has reached the host
            consume(0)
            consume(1)

    ms_e2e = timed(e2e_region, K)
    log(f"e2e region: {ms_e2e / K:.3f} ms/step ({loss_seen['n']} losses read back)")
    clocks = sampler.finish()
    mem.check_last_sample()
    assert np.isfinite(loss_seen["sum"]) and loss_seen["n"] >= K

    # ---- per-kernel durations: eager pass, CUDA events around every hand-written kernel -------------------
    agent.use_cuda_graph = False
    for _ in range(3):
        step()
    timed_steps = min(K, 100)   # the library keeps events for 2048 launches per kernel id (PROF_SLOTS): up to 20 per step fit
    with _lib.KernelTimer() as kt:
        for i in range(timed_steps):
            for j in range(REPLAY_FREQUENCY if i % 10 == 0 else 0):
                mem.append(host_frames[j], j, 0.0, False)
            step()
        torch.cuda.synchronize(dev)
    agent.use_cuda_graph = True
    log("kernel timing pass done")

    # ---- context only (N = 1): the same update with the documented TF32 switch for the conv body (north star: "tensor
    # cores only there").  Not the headline: the parity tests and `value` run the fp32 policy the Agent sets by default.
    tf32_ctx = None
    if world == 1 and not opts.no_cpu_baseline:
        import argparse as _ap
        a2 = Agent(_ap.Namespace(**{**vars(args), "tf32": True}), FakeEnv())     # sets the process-wide TF32 flags
        try:
            for _ in range(Agent.GRAPH_WARMUP + 4):
                a2.reset_noise()
                a2.learn(mem)

            def step_tf32(i):
                a2.reset_noise()
                a2.learn(mem)

            ms_tf32 = timed(step_tf32, K)
            tf32_ctx = {"ms_per_step": ms_tf32 / K, "value": K / (ms_tf32 * 1e-3), "unit": "updates/s",
                        "what": "Agent(args.tf32=True): cuDNN may use TF32 tensor-core kernels for the conv body (heads unchanged); outside "
                                "the 1e-5 parity bar, reported for context only"}
        finally:
            torch.backends.cudnn.allow_tf32 = False
            torch.backends.cuda.matmul.allow_tf32 = False
            del a2
        log(f"tf32 conv context: {tf32_ctx['ms_per_step']:.3f} ms/step")

    if rank != 0:
        return
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
    P = agent.optimiser.numel
    noisy = sum(m.weight_epsilon.numel() + m.bias_epsilon.numel() for m in agent.online_net.noisy_layers())
    alg = algorithmic_bytes(cfg, P, noisy)
    # launches per update of every hand-written kernel, counted in the eager pass above (appends excluded: they belong to
    # the e2e loop's actor side, not to `reset_noise(); learn(mem)`)
    launches_per_step = {k: cnt / timed_steps for k, (cnt, _) in kt.result.items() if k != "append"}
    kernels = {}
    for name, (cnt, us) in kt.result.items():
        if name in alg:
            gbs = alg[name] / (us * 1e-6) / 1e9
            kernels[name] = {"us": round(us, 2), "bytes": alg[name], "GBps": round(gbs, 1), "frac": round(gbs / peak, 4),
                             "launches_timed": cnt, "launches_per_step": round(launches_per_step.get(name, 0), 2)}
    step_kernel_us = {k: kt.result[k][1] * n for k, n in launches_per_step.items()}
    # dominant hand-written kernel = the one the step spends the most device time in (duration x launches per update);
    # the longest single launch is reported next to it
    ranked = [k for k in sorted(step_kernel_us, key=step_kernel_us.get, reverse=True) if k in kernels]
    dominant = ranked[0]
    longest = max((k for k in kernels if launches_per_step.get(k, 0)), key=lambda k: kernels[k]["us"])
    d = kernels[dominant]
    # DRAM bytes per launch come from the committed `ncu --set full` capture; they are only quoted while the kernel sources
    # are the ones that capture was taken from (sha256 of csrc/ recorded next to the numbers), otherwise null
    traffic, traffic_note = None, "no ncu --set full capture of this kernel for the current sources"
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        # the capture is quoted only while the translation unit that holds the kernel is byte-identical to the captured one
        if tj.get("source_sha256", {}).get(dominant) == kernel_source_sha(dominant):
            traffic = tj.get(opts.config, {}).get(dominant)
            traffic_note = f"dram__bytes_read.sum + dram__bytes_write.sum per launch, {tj.get('source', 'profiles/')}"
        else:
            traffic_note = "profiles/traffic.json was captured from other sources of this kernel (sha256 differs): not quoted"
    roofline = {"kernel": "k_" + dominant, "bound": "hbm", "achieved": d["GBps"], "peak": peak, "unit": "GB/s", "frac": d["frac"],
                "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": d["bytes"], "us_per_launch": d["us"],
                "selection": "largest (mean launch duration x launches per update) among the hand-written kernels",
                "us_per_step": round(step_kernel_us[dominant], 2),
                "longest_single_launch": {"kernel": "k_" + longest, "us": kernels[longest]["us"], "frac": kernels[longest]["frac"]},
                "timing": "CUDA events around each launch on its stream, eager (non-graph) replay of the same step",
                "kernels": kernels,
                "all_kernel_us": {k: round(v[1], 2) for k, v in kt.result.items()},
                "own_kernel_us_per_step": round(sum(step_kernel_us.values()), 1)}

    total_updates = K * world
    value = total_updates / (ms_value * 1e-3)
    e2e_value = total_updates / (ms_e2e * 1e-3)
    line = {"metric": "learner updates/sec (batch32, 1M buffer, 51 atoms)", "value": value,
            "unit": "updates/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_value / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(opts.config, cfg, world, P),
                           **({"gradient_exchange": ("peer-memory optimiser over NVLink: reduce-scatter by peer loads beside the conv backward, "
                                                     "sharded clip+Adam, all-gather by " + ("NVSwitch multicast stores" if agent.optimiser.peer.multicast else "peer stores"))
                               if agent.peer_optimizer else "NCCL all-reduce (head slice overlapped with the conv backward) + replicated clip+Adam"}
                              if world > 1 else {})),
            "e2e": {"value": e2e_value, "unit": "updates/s", "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": REPLAY_FREQUENCY * 84 * 84 * 4, "d2h_bytes_per_step": B * 4,
                    "what": f"per step: {REPLAY_FREQUENCY} x mem.append(host frame) -- staged in the replay's pinned ring and written by one rb_append_batch "
                            "launch that reads them in place over PCIe -- + dqn.reset_noise() + dqn.learn(mem) + per-sample loss copied to pinned host "
                            "memory and read by the host one step behind the GPU (double buffer)"},
            # our kernels launched in the timed `value` region, counted per kernel id during the eager replay of the same step
            # (C2: 2 k_noise_factors, k_tree_sample, k_gather, 2 x (k_head_fc1_tc + k_head_reduce1 + k_head_fc2), k_c51_dueling,
            # k_head_wgrad2, k_head_dh, k_head_bwd1, 2 k_bias_grad, rb_conv_wgrad (two kernels under one id), k_sqnorm, k_clip_adam,
            # k_tree_update_warp = 20 ids per step; the other graph nodes are cuDNN / ATen)
            "gpu_launches": int(round(K * sum(launches_per_step.values()))),
            "clocks": clocks, "roofline": roofline}
    if tf32_ctx is not None:
        line["tf32_conv_context"] = tf32_ctx
    if deterministic:
        line["dump_outputs"] = {"dir": opts.dump_outputs, "cudnn": "deterministic algorithms, heuristic choice: reproducible "
                                                                    "outputs, slower than a run without --dump-outputs"}
    if world == 1 and not opts.no_cpu_baseline:
        del agent, mem, tr                                  # give the 7 GB of HBM back before the reference's GPU leg
        torch.cuda.empty_cache()
        ups, dt, threads, n_cpu, kind, sample, extra = cpu_arm(cfg, opts.cpu_updates, 3, budget_s=25, also_gpu=dev)
        line["cpu_baseline"] = {"value": ups, "unit": "updates/s", "cores": threads, "kind": kind, "sample": sample}
        line.update(extra)
    emit(line)


class StdoutGuard:
    """Keeps fd 1 clean: libraries (NCCL prints its version banner there) write to stderr instead, and only the
    final JSON line goes to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.real, (text + "\n").encode())


GUARD = None


def emit(obj):
    line = json.dumps(obj)
    if GUARD is not None:
        GUARD.emit(line)
    else:
        print(line, flush=True)


def main():
    global GUARD
    GUARD = StdoutGuard()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--cpu-updates", type=int, default=150)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--peer-optimizer", action="store_true",
                    help="N>1: insist on the fused reduce-scatter + clip + Adam + all-gather over NVLink peer memory (the default tries "
                         "it and falls back to NCCL all-reduce + replicated Adam if symmetric memory cannot be set up)")
    ap.add_argument("--nccl", action="store_true", help="N>1: NCCL all-reduce + replicated Adam (no peer-memory optimiser)")
    ap.add_argument("--profile-steps", type=int, default=0, help="run this many steps inside cudaProfilerStart/Stop and exit")
    ap.add_argument("--profile-mode", default="graph", choices=["graph", "eager", "e2e"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (losses, batch tree indices, priorities "
                         "written back, online-net parameters) as DIR/<name>.npy; inputs are seeded and cuDNN runs its "
                         "deterministic algorithms, so two builds compare output for output (the timing is then slower)")
    opts = ap.parse_args()
    if opts.dump_outputs and (opts.impl != "ours" or opts.profile_steps):
        ap.error("--dump-outputs needs --impl ours and no --profile-steps")
    cfg = CONFIGS[opts.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if opts.impl == "reference":
        reference_arm(opts, cfg, rank)
        return
    if world > 1:
        # a communicator that never comes up must not eat the caller's whole time budget: dump every thread's stack and
        # exit if set-up + warm-up of the multi-rank job take longer than this (cancelled once the timed regions start)
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ.get("RB_BENCH_SETUP_TIMEOUT", "300")), exit=True, file=sys.stderr)
        from rainbow_b200.dist import init_from_env
        init_from_env("nccl")
    elif opts.gpus > 1:
        print(f"bench.py: --gpus {opts.gpus} needs torchrun (one rank per GPU); running rank 0 only on one GPU", file=sys.stderr)
    ours(opts, cfg, rank, world, local)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
