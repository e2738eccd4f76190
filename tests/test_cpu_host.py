"""CPU-only tests of the host side: the C-ABI library loads and exports every declared symbol, argument
validation answers without a GPU, the product refuses to run without CUDA (no CPU fallback), format-exchange
helpers, model layout/initialisation parity with the reference recipe, and the multi-rank gradient exchange
(world_size 2, gloo)."""
import argparse
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def make_args(**kw):
    d = dict(device=torch.device("cpu"), history_length=4, discount=0.99, multi_step=3, priority_weight=0.4,
             priority_exponent=0.5, atoms=51, V_min=-10.0, V_max=10.0, batch_size=32, norm_clip=10.0, model=None,
             learning_rate=6.25e-5, adam_eps=1.5e-4, architecture="canonical", hidden_size=512, noisy_std=0.1)
    d.update(kw)
    return argparse.Namespace(**d)


def test_abi_exports_every_declared_symbol():
    from rainbow_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "rainbow_b200.h")).read()
    declared = set(re.findall(r"^\s*(?:int|const char\*)\s+(rb_\w+)\s*\(", header, flags=re.M))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SIGNATURES), "python binding table and header disagree"
    for name in declared:
        assert hasattr(lib, name), f"librainbow_b200.so does not export {name}"
    assert lib.rb_abi_version() == 2
    assert lib.rb_clip_adam_scratch_elems() > 0


def test_abi_argument_validation_without_gpu():
    """Bad arguments are rejected on the host before any launch, with errno-style codes."""
    from rainbow_b200 import _lib
    lib = _lib.load()
    one = C.c_void_p(8)  # never dereferenced: validation fails first
    assert lib.rb_tree_update(None, 7, 8, one, one, 0.5, 0, 4, one, None, None, None) == -22
    assert b"null" in lib.rb_last_error()
    assert lib.rb_tree_update(one, 7, 7, one, one, 0.5, 0, 4, one, None, None, None) == -22          # odd size
    assert lib.rb_tree_sample(one, 7, 8, one, 3, 4, None, 0, 1, None, 4, 0.4, None, 8, one, one, one, one, one, None) == -22
    assert lib.rb_gather(one, one, one, one, one, 8, one, 4, 40, 30, one, one, one, one, one, one, None) == -34  # window > 64
    assert lib.rb_c51_loss_grad(one, one, one, one, one, one, one, one, -10.0, 10.0, 0.4, 0.97, 4, 6, 200, one, one, None,
                                None, None) == -34                                               # atoms > 128
    assert lib.rb_noisy_resample(None, None, None, None, 4, None, None, 1, None, None) == -22
    assert lib.rb_clip_adam(one, one, one, one, 0, 1.0, 10.0, 1e-4, 0.9, 0.999, 1e-4, one, one, None, None, None) == -22
    tot, n = C.c_double(), C.c_int()
    assert lib.rb_profile_collect(99, C.byref(tot), C.byref(n)) == -22
    # entry points added with ABI version 2
    assert lib.rb_q_values(one, 4, 6, 51, one, None, None, None, None) == -22                       # no output requested
    assert lib.rb_q_values(one, 4, 6, 200, one, one, None, None, None) == -34                       # atoms > RB_MAX_ATOMS
    assert lib.rb_conv_wgrad(one, one, 32, 4, 84, 84, 32, 7, 4, one, one, None, None) == -34        # kernel size not instantiated
    assert lib.rb_conv_wgrad(one, one, 32, 32, 20, 20, 64, 4, 2, one, one, None, None) == -34       # needs more than 256 threads
    assert lib.rb_conv_wgrad(one, None, 32, 4, 84, 84, 32, 8, 4, one, one, None, None) == -22
    assert lib.rb_conv_wgrad_scratch_elems(32, 4, 84, 32, 8, 4) == 32 * 7 * (32 * 4 * 8 * 8 + 32)   # 20 output rows in 7 bands of 3
    assert lib.rb_conv_wgrad_scratch_elems(32, 4, 4, 32, 8, 4) == 0
    two = (C.c_void_p * 2)(8, 8)
    assert lib.rb_peer_reduce(two, two, 2, 0, 2, 0, 64, 0.5, one, one, one, None) == -34            # segment id
    assert lib.rb_peer_reduce(two, two, 2, 0, 0, 0, 60, 0.5, one, one, one, None) == -22            # not a multiple of 4 * world
    assert lib.rb_peer_reduce(two, two, 2, 2, 0, 0, 64, 0.5, one, one, one, None) == -34            # rank >= world
    assert lib.rb_peer_reduce(two, two, 9, 0, 0, 0, 144, 0.5, one, one, one, None) == -34           # world > RB_MAX_PEERS
    beg, ln = (C.c_int64 * 2)(0, 64), (C.c_int64 * 2)(64, 60)
    assert lib.rb_peer_adam_gather(two, two, two, 2, 0, 3, beg, ln, one, one, one, 10.0, 1e-4, 0.9, 0.999, 1e-4, one, one, one,
                                   None, None, None) == -34                                        # at most two segments
    assert lib.rb_peer_adam_gather(two, two, two, 2, 0, 2, beg, ln, one, one, one, 10.0, 1e-4, 0.9, 0.999, 1e-4, one, one, one,
                                   None, None, None) == -22                                        # second segment: 60 elements
    assert lib.rb_peer_scratch_bytes() >= (2 * 592 + 2) * 8


def test_no_cpu_fallback():
    from rainbow_b200 import RainbowB200Error, _lib
    from rainbow_b200.agent import Agent
    from rainbow_b200.memory import ReplayMemory
    from rainbow_b200.model import DQN

    class Env:
        def action_space(self):
            return 6

    with pytest.raises(RainbowB200Error):
        ReplayMemory(make_args(), 1000)
    with pytest.raises(RainbowB200Error):
        Agent(make_args(), Env())
    with pytest.raises(RainbowB200Error):
        DQN(make_args(), 6).reset_noise()
    with pytest.raises(RainbowB200Error):
        _lib.ptr(torch.zeros(4))


def test_product_never_imports_the_oracle():
    for fn in os.listdir(os.path.join(ROOT, "rainbow_b200")):
        if fn.endswith(".py"):
            src = open(os.path.join(ROOT, "rainbow_b200", fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn
    cu = open(os.path.join(ROOT, "rainbow_b200", "csrc", "rb_kernels.cu")).read()
    assert "rb_oracle" not in cu


def test_model_layout_and_init_stream():
    """Same state_dict keys as the reference and -- because construction consumes the torch RNG in the same
    order (uniform_ for weight_mu, bias_mu, then two randn draws per NoisyLinear) -- a seed gives the same
    initial sigma/mu statistics recipe (model.py:25-30)."""
    from rainbow_b200.model import DQN
    torch.manual_seed(3)
    net = DQN(make_args(), 6)
    sd = net.state_dict()
    assert sd["fc_h_v.weight_mu"].shape == (512, 3136) and sd["fc_z_a.weight_mu"].shape == (6 * 51, 512)
    assert sd["convs.0.weight"].shape == (32, 4, 8, 8) and sd["convs.4.weight"].shape == (64, 64, 3, 3)
    assert torch.allclose(sd["fc_h_v.weight_sigma"], torch.full((512, 3136), 0.1 / 3136 ** 0.5))
    assert torch.allclose(sd["fc_h_v.bias_sigma"], torch.full((512,), 0.1 / 512 ** 0.5))
    assert sd["fc_h_v.weight_mu"].abs().max() <= 1 / 3136 ** 0.5
    # construction noise is rank one: eps_w = eps_out (outer) eps_in, eps_b = eps_out
    w, b = sd["fc_z_v.weight_epsilon"], sd["fc_z_v.bias_epsilon"]
    assert torch.allclose(w, torch.outer(b, w[0] / b[0]), atol=1e-6)
    q = net(torch.rand(2, 4, 84, 84))
    assert q.shape == (2, 6, 51) and torch.allclose(q.sum(2), torch.ones(2, 6), atol=1e-5)
    assert torch.allclose(net(torch.zeros(1, 4, 84, 84), log=True).exp().sum(2), torch.ones(1, 6), atol=1e-5)
    de = DQN(make_args(architecture="data-efficient", hidden_size=256), 4)
    assert de.fc_h_v.weight_mu.shape == (256, 576)
    with pytest.raises(ValueError):
        DQN(make_args(architecture="nope"), 4)


def test_reference_format_round_trip():
    from rainbow_b200.memory import Transition_dtype, reference_fields_to_ring, ring_to_reference_fields
    rs = np.random.RandomState(0)
    size = 16
    state = dict(capacity=size, index=5, full=True, max=2.5, sum_tree=rs.rand(15 + size).astype(np.float32),
                 frames=rs.randint(0, 256, (size, 7056), dtype=np.uint8), timestep=rs.randint(0, 9, size).astype(np.int32),
                 action=rs.randint(0, 6, size).astype(np.int32), reward=rs.randn(size).astype(np.float32),
                 nonterminal=rs.randint(0, 2, size).astype(np.uint8))
    ref = ring_to_reference_fields(state)
    assert ref["data"].dtype == Transition_dtype and ref["data"].dtype.itemsize == 7069  # memory.py:7 packed record
    assert ref["tree_start"] == 15 and ref["sum_tree"].shape == (31,)
    back = reference_fields_to_ring(ref, t=3)
    for k in ("frames", "timestep", "action", "reward", "nonterminal"):
        assert np.array_equal(back[k], state[k]), k
    assert back["index"] == 5 and back["full"] is True and back["max_value"] == 2.5 and back["t_episode"] == 3


def test_segment_tree_rejects_odd_sizes_before_touching_cuda():
    from rainbow_b200.memory import SegmentTree
    with pytest.raises(ValueError):
        SegmentTree(7, "cuda:0")


def test_shard_seed_and_single_process_sync():
    from rainbow_b200.dist import GradSync, shard_seed
    seeds = {shard_seed(0, r) for r in range(8)} | {shard_seed(1, r) for r in range(8)}
    assert len(seeds) == 16
    s = GradSync()
    assert not s.enabled and s.world_size == 1 and s.rank == 0
    g = torch.ones(8)
    assert s.all_reduce_(g) is g and s.broadcast_(g) is g and torch.equal(g, torch.ones(8))


_WORKER = r"""
import os, sys, torch
sys.path.insert(0, sys.argv[1])
from rainbow_b200.dist import GradSync, init_from_env, shard_seed
rank, world, local = init_from_env("gloo")
assert world == 2
sync = GradSync()
assert sync.enabled and sync.world_size == 2 and sync.rank == rank
# identical start: rank 0's parameters win
p = torch.full((1000,), float(rank + 1))
sync.broadcast_(p)
assert torch.equal(p, torch.ones(1000))
# data-parallel step: every rank has its own gradient, all ranks must end with the same averaged one
torch.manual_seed(shard_seed(0, rank))
g = torch.randn(1000)
mine = g.clone()
sync.all_reduce_(g)
torch.manual_seed(shard_seed(0, 1 - rank))
other = torch.randn(1000)
assert torch.allclose(g, mine + other)
avg = g * (1.0 / sync.world_size)          # the 1/world factor the clip+Adam kernel applies (grad_scale)
p -= 0.1 * avg
chk = p.clone()
torch.distributed.all_reduce(chk, op=torch.distributed.ReduceOp.MAX)
assert torch.equal(chk, p), "ranks diverged"
# the learner reduces the flat gradient in two slices (noisy head first, on a side stream; conv slice afterwards):
# in-place all-reduce on VIEWS of one flat buffer must equal one all-reduce of the whole buffer
torch.manual_seed(100 + rank)
flat = torch.randn(4096)
whole = flat.clone()
conv_end = 1280
sync.all_reduce_(flat[conv_end:])
sync.all_reduce_(flat[:conv_end])
sync.all_reduce_(whole)
assert torch.equal(flat, whole)
t = torch.tensor([float(rank)])
assert float(sync.max_(t)) == 1.0
torch.distributed.destroy_process_group()
sys.stdout.write(f"rank{rank}ok\n"); sys.stdout.flush()
"""


def test_two_rank_gradient_exchange_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = 29600 + os.getpid() % 300
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script), ROOT]
    env = dict(os.environ, OMP_NUM_THREADS="1")
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    assert out.stdout.count("ok") == 2, out.stdout


def test_bench_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_bench_algorithmic_bytes_match_survey():
    """The roofline numerators bench.py uses are SURVEY.md 8(d)'s per-update figures."""
    sys.path.insert(0, ROOT)
    import bench
    P, noisy = 6_868_928, 3_395_429
    c2 = bench.algorithmic_bytes(bench.CONFIGS["C2"], P, noisy)
    assert c2["tree_sample"] == 3328 and c2["gather"] == 8_807_840 and c2["c51"] == 157_772 and c2["tree_update"] == 8192
    assert c2["clip_adam"] == 7 * P * 4 and c2["sqnorm"] == P * 4 and c2["noisy_resample"] == noisy * 4
    c3 = bench.algorithmic_bytes(bench.CONFIGS["C3"], 828_842, 387_173)
    assert c3["tree_sample"] == 2944 and c3["gather"] == 9_037_984 and c3["tree_update"] == 7040
    c4 = bench.algorithmic_bytes(bench.CONFIGS["C4"], P, noisy)
    assert c4["tree_sample"] == 53_248 and c4["gather"] == 140_925_440 and c4["c51"] == 2_521_292 and c4["tree_update"] == 131_072
    assert bench.host_threads() >= 1


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs writes one float .npy per array, refuses more than 64 MB, and is refused where there is no timed
    step of ours to dump."""
    sys.path.insert(0, ROOT)
    import bench
    arrays = {"loss": np.arange(4, dtype=np.float32), "tree_idx": np.arange(4, dtype=np.float64),
              "param.fc_z_v.bias_mu": np.ones(51, np.float32)}
    bench.dump_outputs(str(tmp_path / "out"), arrays)
    assert sorted(os.listdir(tmp_path / "out")) == sorted(k + ".npy" for k in arrays)
    for k, a in arrays.items():
        back = np.load(tmp_path / "out" / (k + ".npy"))
        assert back.dtype == a.dtype and np.array_equal(back, a)
    with pytest.raises(RuntimeError):
        bench.dump_outputs(str(tmp_path / "big"), {"p": np.zeros(bench.DUMP_LIMIT_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "big").exists()
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                          str(tmp_path / "ref")], capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr and not (tmp_path / "ref").exists()


def test_stdout_guard_keeps_library_prints_off_stdout(tmp_path):
    """Only the JSON line may reach fd 1 (NCCL prints its banner there)."""
    script = tmp_path / "guard.py"
    script.write_text("import os, sys\nsys.path.insert(0, %r)\nimport bench\nbench.GUARD = bench.StdoutGuard()\n"
                      "os.write(1, b'library banner\\n')\nprint('python print')\nbench.emit({'ok': 1})\n" % ROOT)
    out = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout == '{"ok": 1}\n'
    assert "library banner" in out.stderr and "python print" in out.stderr


def test_flat_parameter_layout():
    """FusedClipAdam host logic (no kernel is launched): every parameter becomes a view of ONE flat buffer on a
    256-byte boundary, gradients likewise, conv parameters come first (conv_end), padding stays zero."""
    from rainbow_b200.agent import FusedClipAdam
    from rainbow_b200.model import DQN
    torch.manual_seed(0)
    net = DQN(make_args(architecture="data-efficient", hidden_size=64), 3)
    before = {k: v.clone() for k, v in net.state_dict().items()}
    opt = FusedClipAdam(net, lr=1e-4, eps=1e-4, max_norm=10.0)
    named = [(n, p) for n, p in net.named_parameters()]
    assert len(named) == 4 + 16 and opt.numel % 64 == 0
    base = opt.flat_param.data_ptr()
    prev_end = 0
    for (n, p), off in zip(named, opt.offsets):
        assert off % 64 == 0 and off >= prev_end
        assert p.data_ptr() == base + 4 * off and p.grad.data_ptr() == opt.flat_grad.data_ptr() + 4 * off
        assert torch.equal(p, before[n]), n                      # values survived the re-pointing
        assert not opt.flat_param[prev_end:off].any()             # alignment padding is zero
        prev_end = off + p.numel()
    first_fc = next(off for (n, _), off in zip(named, opt.offsets) if n.startswith("fc_"))
    assert opt.conv_end == first_fc and all(n.startswith("convs.") for (n, _), off in zip(named, opt.offsets) if off < first_fc)
    opt.flat_grad.fill_(1.0)
    opt.zero_conv_grad()
    assert not opt.flat_grad[:opt.conv_end].any() and opt.flat_grad[opt.conv_end:].all()
    opt.zero_grad()
    assert not opt.flat_grad.any()
    # load_state_dict writes through the views (the flat buffer follows), as update_target_net / --model rely on
    net.load_state_dict({k: v + 1 for k, v in before.items()})
    assert torch.equal(opt.flat_param[opt.offsets[0]:opt.offsets[0] + named[0][1].numel()], (before[named[0][0]] + 1).reshape(-1))


def test_save_reference_pickle_is_loaded_by_the_unmodified_reference():
    """SURVEY 8(f).3, export direction: save_reference_pickle() of a replay holding the fixture's arrays must decode to the
    same object graph as tests/golden/ref_memory.pkl.bz2, the file the UNMODIFIED reference wrote from that replay (same
    class names, attributes, types, dtypes and bits).  The reference's pickle.load builds its objects from exactly that
    graph, so it loads ours into the object whose next sample (np.random.seed(3)) is tests/golden/ref_memory.npz `tidx`."""
    import bz2
    import io
    import pickle
    from helpers import GOLD, golden
    from rainbow_b200.memory import Transition_dtype, save_reference_pickle
    g = golden("ref_memory")
    meta = g["meta"]
    size = int(meta[3])

    class HostReplay:   # stands in for a device ReplayMemory: same reference_state() contract, no GPU needed
        def reference_state(self, device="cpu"):
            data = np.zeros(size, dtype=Transition_dtype)
            data["timestep"], data["state"] = g["timestep"], g["frames"].reshape(size, 84, 84)
            data["action"], data["reward"], data["nonterminal"] = g["action"], g["reward"], g["nonterminal"].astype(np.bool_)
            mem = dict(device=torch.device(device), capacity=size, history=4, discount=0.99, n=3, priority_weight=0.4,
                       priority_exponent=0.5, t=int(meta[2]), n_step_scaling=torch.tensor([0.99 ** i for i in range(3)]))
            tree = dict(index=int(meta[0]), size=size, full=bool(meta[1]), tree_start=2 ** (size - 1).bit_length() - 1,
                        sum_tree=g["sum_tree"], data=data, max=float(g["max"]))
            return mem, tree

    buf = io.BytesIO()
    save_reference_pickle(HostReplay(), buf)
    assert "memory" not in sys.modules or "rainbow_b200" not in getattr(sys.modules["memory"], "__file__", "")

    class Decoder(pickle.Unpickler):   # the reference's classes as empty stand-ins: the graph is decoded, no code of theirs runs
        def find_class(self, module, name):
            if module == "memory":
                return type(name, (), {"__module__": "memory"})
            return super().find_class(module, name)

    ours = Decoder(io.BytesIO(buf.getvalue())).load()
    with bz2.open(os.path.join(GOLD, "ref_memory.pkl.bz2"), "rb") as f:
        theirs = Decoder(f).load()
    for a, b in ((ours, theirs), (ours.transitions, theirs.transitions)):
        assert (type(a).__module__, type(a).__name__) == (type(b).__module__, type(b).__name__)
        assert sorted(vars(a)) == sorted(vars(b)), type(b).__name__
        for k, want in vars(b).items():
            got = vars(a)[k]
            if k == "transitions":
                continue
            if isinstance(want, np.ndarray):
                assert type(got) is np.ndarray and got.dtype == want.dtype and got.shape == want.shape, k
                assert got.tobytes() == want.tobytes(), k
            elif isinstance(want, torch.Tensor):
                assert type(got) is torch.Tensor and got.dtype == want.dtype and got.device == want.device, k
                assert torch.equal(got, want), k
            elif k == "max":   # the running max: a numpy float32 once a priority was written, a Python number before
                assert isinstance(got, (float, np.floating)) and np.float32(got) == want, k
            else:
                assert type(got) is type(want) and got == want, k


def test_oracle_clip_adam_follows_the_reference_trajectory():
    """Pins oracle.clip_adam (the checker of rb_clip_adam) to the UNMODIFIED reference: the recorded gradients of the three
    consecutive C2-shaped updates (tests/golden/update_c2.npz, sub-sampled tensors) driven through the oracle's clip+Adam must
    reproduce the reference's parameters after every step to float rounding (<= 4e-9 = one ulp of the largest weights, |p| < 0.0625)."""
    import oracle
    from helpers import golden, update_case
    case, g = update_case("c2"), golden("update_c2")
    torch.manual_seed(case["seed"])
    args = make_args(batch_size=case["B"], multi_step=case["n"], architecture=case["arch"], hidden_size=case["hidden"])
    from rainbow_b200.model import DQN
    net = DQN(args, case["A"])            # same host RNG stream as the reference's Agent construction (checked by SHA below)
    import hashlib
    sd0 = torch.cat([p.detach().reshape(-1) for _, p in net.named_parameters()]).numpy()
    assert hashlib.sha256(sd0.tobytes()).hexdigest() == case["sd0_sha"]
    keys = [k for k, _ in net.named_parameters()]
    p = np.concatenate([v.detach().reshape(-1)[::case["strides"][k]].numpy() for k, v in net.named_parameters()]).astype(np.float32)
    m, v = np.zeros_like(p), np.zeros_like(p)
    worst = 0.0
    for s in range(case["steps"]):
        grad = np.concatenate([g[f"s{s}_grad.{k}"] for k in keys]).astype(np.float32)
        total = float(np.sqrt(sum(g[f"s{s}_gradsum.{k}"][1] for k in keys)))
        assert total < 10.0           # no clipping in the recorded steps: the sub-sample's own norm is below the threshold too
        oracle.clip_adam(p, grad, m, v, 10.0, 6.25e-5, 0.9, 0.999, 1.5e-4, s + 1)
        want = np.concatenate([g[f"s{s}_param.{k}"] for k in keys])
        worst = max(worst, float(np.abs(p - want).max()))
        p[:] = want                   # follow the reference exactly from here on (m, v stay the oracle's)
    assert worst <= 4e-9, worst


def test_bench_traffic_capture_is_keyed_by_kernel_source():
    """profiles/traffic.json carries, per kernel, the hash of the source file the capture was taken from; bench.py quotes a
    capture only while that file is unchanged (VERDICT r01: a stale capture must never be quoted)."""
    import json
    sys.path.insert(0, ROOT)
    import bench
    tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    assert set(tj["source_sha256"]) == set(tj["C2"])
    for name in tj["C2"]:
        assert len(bench.kernel_source_sha(name)) == 64
    # a kernel of rb_head.cu does not depend on rb_kernels.cu and the other way round
    assert bench.KERNEL_SOURCES["head_bwd1"] == ["rb_head.cu"] and "clip_adam" not in bench.KERNEL_SOURCES
    assert bench.kernel_source_sha("clip_adam") == bench.csrc_sha256(["rb_internal.cuh", "rb_kernels.cu"])
    assert bench.kernel_source_sha("clip_adam") != bench.kernel_source_sha("head_bwd1")
