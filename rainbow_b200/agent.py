"""Rainbow learner: the reference's Agent API (agent.py:12-118) over B200-native kernels.

One `learn(mem)` (agent.py:61-100) is:

    K1 rb_tree_sample + K2 rb_gather          (mem.sample, memory.py:148-155)
    3 x conv body (torch: cuDNN)              (agent.py:66,71,75 -> model.py:70-71)
    K6 rb_noisy_resample (target net)         (agent.py:74)
    fused noisy dueling heads (rb_head_forward) on the conv features -- online net on [s; s'], target on s'
    K3 rb_c51_dueling_loss_grad               (agent.py:67,72-73,76-96 + softmax halves of model.py:76-79 + model.py:75)
    rb_head_backward (16 head gradients + d conv features), torch autograd backward through the online convs
    [NCCL all-reduce of the flat gradient when world_size > 1]
    K7 rb_clip_adam                           (agent.py:97-98)
    K4 rb_tree_update                         (agent.py:100 -> memory.py:157-159)

Nothing in that chain synchronises with the host, so the whole update is captured into one CUDA graph
(`cuda_graph=True`, the default) and replayed: the update is launch-latency bound otherwise
(the reference issues ~600 ATen ops per update, SURVEY.md 2.1).
"""
import os
import warnings
import weakref

import numpy as np
import torch

from . import _lib
from .dist import GradSync
from .memory import ReplayMemory, _SampleWorkspace
from .model import DQN


def c51_loss_grad(q_online_s, q_online_ns, q_target_ns, actions, returns, nonterminals, weights, support, vmin, vmax,
                  delta_z, gamma_n, loss=None, grad=None, m_out=None, astar_out=None):
    """Launch K3 on pre-softmax logits [B,A,Z]; returns (loss[B], grad[B,A,Z])."""
    B, A, Z = q_online_s.shape
    dev = q_online_s.device
    if loss is None:
        loss = torch.empty(B, dtype=torch.float32, device=dev)
    if grad is None:
        grad = torch.empty((B, A, Z), dtype=torch.float32, device=dev)
    _lib.check(_lib.load().rb_c51_loss_grad(
        _lib.ptr(q_online_s), _lib.ptr(q_online_ns), _lib.ptr(q_target_ns), _lib.ptr(actions), _lib.ptr(returns),
        _lib.ptr(nonterminals), _lib.ptr(weights), _lib.ptr(support), float(vmin), float(vmax), float(delta_z),
        float(gamma_n), B, A, Z, _lib.ptr(loss), _lib.ptr(grad), _lib.ptr(m_out), _lib.ptr(astar_out), _lib.stream()))
    return loss, grad


def c51_dueling_loss_grad(z_online, z_target, actions_n, atoms, actions, returns, nonterminals, weights, support, vmin, vmax,
                          delta_z, gamma_n, m_out=None, astar_out=None):
    """K3 fed straight by the fused heads (rb_c51_dueling_loss_grad): z_online [2B, Z(1+A)] (s rows, then s' rows),
    z_target [B, Z(1+A)]; returns (loss[B], dz[B, Z(1+A)]) with dz = d mean(w*loss) / d (z_value | z_advantage)."""
    B = actions.shape[0]
    loss = torch.empty(B, dtype=torch.float32, device=actions.device)
    dz = torch.empty((B, atoms * (1 + actions_n)), dtype=torch.float32, device=actions.device)
    _lib.check(_lib.load().rb_c51_dueling_loss_grad(
        _lib.ptr(z_online), _lib.ptr(z_target), actions_n, atoms, _lib.ptr(actions), _lib.ptr(returns),
        _lib.ptr(nonterminals), _lib.ptr(weights), _lib.ptr(support), float(vmin), float(vmax), float(delta_z),
        float(gamma_n), B, _lib.ptr(loss), _lib.ptr(dz), _lib.ptr(m_out), _lib.ptr(astar_out), _lib.stream()))
    return loss, dz


class FusedClipAdam:
    """clip_grad_norm_ + Adam (agent.py:46,97-98) over ONE flat parameter buffer.

    The network's parameters are re-pointed at slices of `flat_param` (each slice starts on a 256-byte
    boundary; padding stays zero), their .grad at slices of `flat_grad`, so the optimiser step is two kernel
    launches (sum of squares, then clip+Adam) and the multi-GPU gradient exchange is a single all-reduce."""

    ALIGN = 64  # elements

    def __init__(self, net, lr, eps, max_norm, betas=(0.9, 0.999), peer=False):
        named = [(n, p) for n, p in net.named_parameters() if p.requires_grad]
        self.params = [p for _, p in named]
        dev = self.params[0].device
        self.offsets, off = [], 0
        self.conv_end = None  # flat offset where the first noisy-head parameter starts (convs come first)
        for n, p in named:
            if self.conv_end is None and n.startswith("fc_"):
                self.conv_end = off
            self.offsets.append(off)
            off += -(-p.numel() // self.ALIGN) * self.ALIGN
        self.numel = off
        if self.conv_end is None:
            self.conv_end = off
        self.lr, self.eps, self.max_norm, self.betas = float(lr), float(eps), float(max_norm), betas
        self.peer = None
        if peer:   # buffers in symmetric memory, optimiser fused with the gradient exchange (csrc/rb_peer.cu)
            from .peer import PeerOptimizerState
            # segment 0 = noisy head (final first, reduced while the conv backward runs), segment 1 = conv parameters
            self.peer = PeerOptimizerState(off, dev, segments=[(self.conv_end, off), (0, self.conv_end)])
            self.flat_param, self.flat_grad = self.peer.flat_param, self.peer.flat_grad
            self.exp_avg, self.exp_avg_sq = self.peer.exp_avg, self.peer.exp_avg_sq
        else:
            self.flat_param = torch.zeros(off, dtype=torch.float32, device=dev)
            self.flat_grad = torch.zeros(off, dtype=torch.float32, device=dev)
            self.exp_avg = torch.zeros(off, dtype=torch.float32, device=dev)
            self.exp_avg_sq = torch.zeros(off, dtype=torch.float32, device=dev)
        self.step_count = self.peer.step_count if self.peer is not None else torch.zeros(1, dtype=torch.int64, device=dev)
        self.grad_norm = self.peer.grad_norm if self.peer is not None else torch.zeros(1, dtype=torch.float32, device=dev)
        self._lib = _lib.load()
        self._partial = torch.zeros(self._lib.rb_clip_adam_scratch_elems(), dtype=torch.float64, device=dev)
        with torch.no_grad():
            for p, o in zip(self.params, self.offsets):
                n = p.numel()
                self.flat_param[o:o + n].copy_(p.reshape(-1))
                p.data = self.flat_param[o:o + n].view_as(p)
                p.grad = self.flat_grad[o:o + n].view_as(p)

    def zero_grad(self):
        self.flat_grad.zero_()

    def zero_conv_grad(self):
        """Only the conv parameters accumulate through autograd on the fused path; the head kernels overwrite theirs."""
        self.flat_grad[:self.conv_end].zero_()

    def step(self, grad_scale=1.0, gate=None):
        """`gate`: optional device int32 (ReplayMemory.sample_gate()); when its first element is 0 the step is skipped on
        the device (single-GPU only: data-parallel ranks must step in lock step, there a rejected batch simply contributes
        a zero gradient through its zeroed importance weights)."""
        if self.peer is not None:   # reduce-scatter + clip + Adam + all-gather over peer memory (1/world folded in)
            self.peer.step(self.max_norm, self.lr, self.betas, self.eps)
            return
        _lib.check(self._lib.rb_clip_adam(
            _lib.ptr(self.flat_param), _lib.ptr(self.flat_grad), _lib.ptr(self.exp_avg), _lib.ptr(self.exp_avg_sq),
            self.numel, float(grad_scale), self.max_norm, self.lr, self.betas[0], self.betas[1], self.eps,
            _lib.ptr(self.step_count), _lib.ptr(self._partial), _lib.ptr(self.grad_norm), _lib.ptr(gate), _lib.stream()))

    def state_dict(self):
        return dict(step=int(self.step_count.item()), exp_avg=self.exp_avg.clone(), exp_avg_sq=self.exp_avg_sq.clone(),
                    lr=self.lr, eps=self.eps, betas=self.betas, max_norm=self.max_norm)

    def load_state_dict(self, sd):
        self.step_count.fill_(int(sd["step"]))
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])


class Agent:
    def __init__(self, args, env):
        self.device = torch.device(args.device)
        if self.device.type != "cuda":
            raise _lib.RainbowB200Error(f"rainbow_b200.Agent needs a CUDA device, got '{self.device}' (no CPU fallback)")
        # Precision policy (documented switch, default = the reference's arithmetic): the learner computes in true fp32.
        # `args.tf32 = True` lets cuDNN / cuBLAS use TF32 tensor cores for the conv backward and the autograd fallback
        # (features()); the own conv forward is fp32-accurate either way.  The parity tests and bench.py run with the
        # default.  torch keeps these flags per process, so the
        # Agent sets them: what is measured is what ships.
        self.tf32 = bool(getattr(args, "tf32", False))
        torch.backends.cudnn.allow_tf32 = self.tf32
        torch.backends.cuda.matmul.allow_tf32 = self.tf32
        self.action_space = env.action_space()
        self.history = int(getattr(args, "history_length", 4))
        self.atoms = args.atoms
        self.Vmin = args.V_min
        self.Vmax = args.V_max
        self.support = torch.linspace(args.V_min, args.V_max, self.atoms).to(device=self.device)  # agent.py:18
        self.delta_z = (args.V_max - args.V_min) / (self.atoms - 1)
        self.batch_size = args.batch_size
        self.n = args.multi_step
        self.discount = args.discount
        self.norm_clip = args.norm_clip

        self.online_net = DQN(args, self.action_space).to(device=self.device)
        model_path = getattr(args, "model", None)
        if model_path:  # agent.py:26-36: pretrained weights, with the old conv key names re-mapped
            if not os.path.isfile(model_path):
                raise FileNotFoundError(model_path)
            state_dict = torch.load(model_path, map_location="cpu")
            for i, old in enumerate(("conv1", "conv2", "conv3")):
                for kind in ("weight", "bias"):
                    if f"{old}.{kind}" in state_dict:
                        state_dict[f"convs.{2 * i}.{kind}"] = state_dict.pop(f"{old}.{kind}")
            self.online_net.load_state_dict(state_dict)
            print("Loading pretrained model: " + model_path)
        self.online_net.train()
        self.online_net.lazy_noise = True   # reset_noise() is launched at its first use / on a side branch of the update

        self.target_net = DQN(args, self.action_space).to(device=self.device)
        self.sync = GradSync()  # no-op unless torch.distributed is initialised with world_size > 1
        # distinct noise streams per net and per rank
        self.online_net.noise_seed = (self.online_net.noise_seed * 2 + 1 + 7919 * self.sync.rank) & (2 ** 63 - 1)
        self.target_net.noise_seed = (self.target_net.noise_seed * 2 + 2 + 7919 * self.sync.rank) & (2 ** 63 - 1)

        # peer_optimizer: "auto" (bench.py's multi-GPU default) tries the fused NVLink optimiser (csrc/rb_peer.cu) and falls
        # back to NCCL all-reduce + replicated Adam on EVERY rank if any rank could not set up the symmetric memory;
        # True insists (raises), False / absent keeps the NCCL path
        want = getattr(args, "peer_optimizer", False)
        self.peer_optimizer = bool(want) and self.sync.enabled
        self.optimiser = None
        if self.peer_optimizer:
            err = None
            try:
                self.optimiser = FusedClipAdam(self.online_net, lr=args.learning_rate, eps=args.adam_eps, max_norm=self.norm_clip,
                                               peer=True)
            except Exception as e:   # noqa: BLE001 -- whatever went wrong, all ranks must take the same path
                err = e
            ok = torch.tensor([0 if err is not None else 1], dtype=torch.int32, device=self.device)
            torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN)
            if int(ok.item()) == 0:
                if want != "auto":
                    raise _lib.RainbowB200Error(f"peer optimiser could not be set up on some rank (this rank: {err})")
                warnings.warn(f"rainbow_b200: peer-memory optimiser unavailable ({err}); using NCCL all-reduce + replicated Adam")
                self.peer_optimizer, self.optimiser = False, None
        if self.optimiser is None:
            self.optimiser = FusedClipAdam(self.online_net, lr=args.learning_rate, eps=args.adam_eps, max_norm=self.norm_clip,
                                           peer=False)
        self.sync.broadcast_(self.optimiser.flat_param)  # identical initial parameters on every rank
        if self.peer_optimizer:
            self.sync.exchange = False   # the optimiser step does the gradient exchange itself
        self.update_target_net()
        self.target_net.train()
        for p in self.target_net.parameters():
            p.requires_grad = False

        self.use_cuda_graph = bool(getattr(args, "cuda_graph", True))
        self.use_fused_head = bool(getattr(args, "fused_head", True))
        self.batch_online_convs = bool(getattr(args, "batch_online_convs", True))
        self._step_gate = None
        self._streams = None
        self._graphs = {}         # online-noise-pending flag -> (captured update graph, its sample workspace, its loss tensor)
        self._graph_key = None    # (weakref to the memory the graph was captured for, batch size)
        self._learn_calls = 0
        self._rejected_seen = 0
        self._q_graphs = {}       # training-mode flag -> captured one-state act / evaluate_q graph
        self.last_loss = None  # per-sample losses of the most recent update (device tensor)

    # ---- acting / evaluation (agent.py:49-59,110-118) ---------------------------------------------
    def reset_noise(self):
        self.online_net.reset_noise()

    def q_select(self, states, q_out=None):
        """Greedy action and its value for a batch of states [N, history, 84, 84] (device): conv body (rb_conv_forward), fused
        noisy dueling head, then rb_q_values -- softmax over atoms, expectation over the support (agent.py:55) and the
        arg-max / max over actions in one launch.  Returns device tensors (actions int64[N], values float32[N]); nothing
        synchronises.  Falls back to plain torch ops for head shapes the fused kernels do not cover."""
        on = self.online_net
        N = states.shape[0]
        with torch.no_grad():
            if on.fused_ok(N):
                x = on.features_nograd(states).contiguous()
                z, _, _ = on.head().forward(x)
                best_a = torch.empty(N, dtype=torch.int64, device=self.device)
                best_q = torch.empty(N, dtype=torch.float32, device=self.device)
                _lib.check(_lib.load().rb_q_values(_lib.ptr(z), N, self.action_space, self.atoms, _lib.ptr(self.support),
                                                   _lib.ptr(q_out), _lib.ptr(best_a), _lib.ptr(best_q), _lib.stream()))
                return best_a, best_q
            q = (on(states) * self.support).sum(2)
            if q_out is not None:
                q_out.copy_(q)
            best_q, best_a = q.max(1)
            return best_a, best_q

    def _one_state(self, state):
        """One state through a captured CUDA graph (conv x3, fused head x2, rb_q_values): returns pinned host tensors
        (action int64[1], value float32[1]) after ONE device-to-host copy and one event wait -- the per-env-step cost of
        main.py:139,153 / test.py:26 instead of ~40 eager launches and a blocking .item()."""
        on = self.online_net
        on.flush_noise()            # a deferred reset_noise() must not be captured into (and redrawn by) the act graph
        key = bool(on.training)
        g = self._q_graphs.get(key)
        if g is None:
            g = dict(inp=torch.zeros((1, self.history, 84, 84), dtype=torch.float32, device=self.device),
                     host=torch.zeros(2, dtype=torch.float64).pin_memory(), dev=torch.zeros(2, dtype=torch.float64, device=self.device),
                     done=torch.cuda.Event(), graph=None, warm=0)
            self._q_graphs[key] = g

        def run():
            a, q = self.q_select(g["inp"])
            g["dev"][0:1].copy_(a)      # both results in one small buffer -> one D2H copy
            g["dev"][1:2].copy_(q)

        g["inp"].copy_(state.reshape(g["inp"].shape), non_blocking=True)
        if not self.use_cuda_graph:
            run()
        elif g["graph"] is None and g["warm"] < 2:
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):
                run()
            torch.cuda.current_stream(self.device).wait_stream(side)
            g["warm"] += 1
        else:
            if g["graph"] is None:
                torch.cuda.synchronize(self.device)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    run()
                g["graph"] = graph
            g["graph"].replay()
        g["host"].copy_(g["dev"], non_blocking=True)
        g["done"].record(torch.cuda.current_stream(self.device))
        g["done"].synchronize()
        return g["host"]

    def act(self, state):
        """agent.py:53-55."""
        return int(self._one_state(state)[0])

    def act_e_greedy(self, state, epsilon=0.001):
        return np.random.randint(0, self.action_space) if np.random.random() < epsilon else self.act(state)

    def evaluate_q(self, state):
        """agent.py:110-112 (one state -> float).  For many states use evaluate_q_batch / evaluate_q_memory."""
        return float(self._one_state(state)[1])

    def evaluate_q_batch(self, states):
        """max_a Q(s, a) for states [N, history, 84, 84]: device float32[N], no synchronisation."""
        return self.q_select(states)[1]

    def evaluate_q_memory(self, val_mem, chunk=64):
        """test.py:37-41 `for state in val_mem: T_Qs.append(dqn.evaluate_q(state))` as batched passes over the validation
        memory's iterator states (rb_iter_states -> conv -> fused head -> rb_q_values) and a single read-back.
        Returns the list of floats that loop would have produced."""
        outs = []
        for first in range(0, val_mem.capacity, chunk):
            count = min(chunk, val_mem.capacity - first)
            outs.append(self.q_select(val_mem.iter_states(first, count))[1])
        return torch.cat(outs).cpu().tolist() if outs else []

    def train(self):
        self.online_net.train()

    def eval(self):
        self.online_net.eval()

    def update_target_net(self):
        self.target_net.load_state_dict(self.online_net.state_dict())

    def save(self, path, name="model.pth"):
        torch.save(self.online_net.state_dict(), os.path.join(path, name))

    # ---- the update ------------------------------------------------------------------------------
    def _fused_path(self, B):
        """The fused head takes the update: online forward over [s; s'], target forward over s', backward over the batch
        (B <= 32, and the head shape within the backward kernels' limits).  Everything else takes the library path."""
        on = self.online_net
        return (self.use_fused_head and on.training and on.fused_ok(2 * B) and on.fused_ok(B, backward=True) and
                self.target_net.fused_ok(B))

    @staticmethod
    def _adjacent(states, next_states):
        """The [2B, ...] tensor whose halves are `states` and `next_states`, if they are laid out that way."""
        if (states.is_contiguous() and next_states.is_contiguous() and states.shape == next_states.shape and
                next_states.data_ptr() == states.data_ptr() + states.numel() * states.element_size() and
                states._base is not None and states._base is next_states._base):
            base = states._base
            if base.data_ptr() == states.data_ptr() and base.numel() == 2 * states.numel():
                return base.view((2 * states.shape[0],) + tuple(states.shape[1:]))
        return None

    def _side_streams(self):
        if self._streams is None:
            self._streams = (torch.cuda.Stream(device=self.device), torch.cuda.Stream(device=self.device))
        return self._streams

    def _update_fused(self, batch, target_noise=None, after_loss=None):
        """agent.py:66-98 with the fused head: torch only runs the conv bodies (forward x3, backward x1).
        The three network passes are independent until the loss, and every conv kernel of this size leaves most of the
        148 SMs idle, so they run as three concurrent branches (fork/join with events; inside the captured CUDA graph
        they become parallel branches): online(s) with autograd on the caller's stream, online(s') and the whole
        target pass (noise draw, convs, head) on two side streams."""
        idxs, states, actions, returns, next_states, nonterminals, weights = batch
        on, tg = self.online_net, self.target_net
        B = states.shape[0]
        main = torch.cuda.current_stream(self.device)
        s_ns, s_tg = self._side_streams()
        fork = torch.cuda.Event()
        fork.record(main)
        noise_done = None
        if on._noise_pending:   # the online net's deferred reset_noise(): beside the sampling / conv work, not in front of it
            with torch.cuda.stream(s_ns):
                s_ns.wait_event(fork)
                on.flush_noise()
                noise_done = torch.cuda.Event()
                noise_done.record(s_ns)
        with torch.cuda.stream(s_tg), torch.no_grad():
            s_tg.wait_event(fork)
            if target_noise is None:
                tg.reset_noise()                                            # agent.py:74
            else:
                tg.reset_noise(*target_noise)
            x_t = tg.features_nograd(next_states)
            z_t, _, _ = tg.head().forward(x_t)
            done_tg = torch.cuda.Event()
            done_tg.record(s_tg)
        manual = on.manual_conv_ok(states)
        # [s; s'] in ONE conv pass when the sampler laid both state blocks out back to back (ReplayMemory's workspaces do):
        # the online net's weights stream once, and two concurrent conv chains (online, target) share the SMs instead of three
        both = self._adjacent(states, next_states) if (manual and self.batch_online_convs) else None
        if both is not None:
            with torch.no_grad():
                acts2 = on.conv_forward_saving(both)
                acts = [a[:B] for a in acts2]              # the s half (batch-major: contiguous slices) feeds the backward
                x_both = acts2[-1].view(2 * B, -1)
                x_s, xs_d = x_both[:B], x_both[:B]
                if noise_done is not None:
                    main.wait_event(noise_done)
                z_on, h_on, p_on = on.head().forward(x_both)              # rows [0,B) = s, [B,2B) = s'
                main.wait_event(done_tg)
        else:
            with torch.cuda.stream(s_ns), torch.no_grad():
                s_ns.wait_event(fork)
                x_ns = on.features_nograd(next_states)
                done_ns = torch.cuda.Event()
                done_ns.record(s_ns)
            if manual:
                with torch.no_grad():
                    acts = on.conv_forward_saving(states)  # library kernels, backward scheduled by hand below
                x_s = acts[-1].view(B, -1)
            else:
                x_s = on.features(states)                  # autograd graph: convs only
            with torch.no_grad():
                xs_d = x_s.detach()
                main.wait_event(done_ns)
                if noise_done is not None:
                    main.wait_event(noise_done)
                x_ns.record_stream(main)
                z_on, h_on, p_on = on.head().forward(xs_d, x_ns)              # rows [0,B) = s, [B,2B) = s'
                main.wait_event(done_tg)
        with torch.no_grad():
            loss, dz = c51_dueling_loss_grad(z_on, z_t, self.action_space, self.atoms, actions, returns, nonterminals, weights,
                                             self.support, self.Vmin, self.Vmax, self.delta_z, self.discount ** self.n)
            wb_done = None
            if after_loss is not None:
                # the priority write-back (agent.py:100) needs nothing but the per-sample losses: it runs on a side
                # stream beside the whole backward instead of at the end of the critical path
                loss_ready = torch.cuda.Event()
                loss_ready.record(main)
                with torch.cuda.stream(s_ns):
                    s_ns.wait_event(loss_ready)
                    after_loss(loss)
                    wb_done = torch.cuda.Event()
                    wb_done.record(s_ns)
            dh = torch.empty((B + 32, 2 * on.hidden_size), dtype=torch.float32, device=self.device)   # dh, then its transpose
            dx = torch.empty_like(xs_d)
            if manual:
                # dx comes back already masked by the last conv layer's ReLU; conv gradients are overwritten.
                # The layer-2 weight gradient feeds nothing but the optimiser: it runs beside the dh -> layer-1 chain.
                hd = on.head()
                dz_ready = torch.cuda.Event()
                dz_ready.record(main)
                with torch.cuda.stream(s_tg):
                    s_tg.wait_event(dz_ready)
                    hd.backward(p_on, xs_d, h_on[:B], dz, dh, dx, parts=hd.BWD_WGRAD2)
                    w2_done = torch.cuda.Event()
                    w2_done.record(s_tg)
                hd.backward(p_on, xs_d, h_on[:B], dz, dh, dx, relu_mask_x=True, parts=hd.BWD_DH | hd.BWD_LAYER1)
                main.wait_event(w2_done)
                head_ready = None
                if self.sync.enabled:
                    # 99 % of the gradient bytes (the noisy head) are final here: start their exchange on a side
                    # stream so it overlaps the conv backward; the conv slice (a few hundred KB) follows afterwards.
                    # Peer optimiser: reduce-scatter by NVLink peer loads (rb_peer_reduce); else NCCL all-reduce.
                    head_ready = torch.cuda.Event()
                    head_ready.record(main)
                    with torch.cuda.stream(s_tg):
                        s_tg.wait_event(head_ready)
                        if self.optimiser.peer is not None:
                            self.optimiser.peer.reduce_segment(0)
                        else:
                            self.sync.all_reduce_(self.optimiser.flat_grad[self.optimiser.conv_end:])
                        head_reduced = torch.cuda.Event()
                        head_reduced.record(s_tg)
                # (a separate stream for the first layer's own weight-gradient kernel was tried and lost: it then overlaps
                # cuDNN's wgrad of the layer above and both slow down -- r02e vs r02f timelines)
                grads_done = on.conv_backward_into_grads(acts, dx.view_as(acts[-1]), s_ns)
                main.wait_event(grads_done)
                if self.sync.enabled:
                    self.sync.all_reduce_(self.optimiser.flat_grad[:self.optimiser.conv_end])
                    main.wait_event(head_reduced)
            else:
                self.optimiser.zero_conv_grad()
                on.head().backward(p_on, xs_d, h_on[:B], dz, dh, dx)       # writes the 16 head gradients + dx
        if not manual:
            x_s.backward(dx)
            self.sync.all_reduce_(self.optimiser.flat_grad)
        self.optimiser.step(grad_scale=1.0 / self.sync.world_size, gate=self._step_gate)
        if wb_done is not None:
            main.wait_event(wb_done)
        return loss

    def _update_from_batch(self, batch, target_noise=None, after_loss=None, gate=None):
        """agent.py:66-98 on an already sampled batch; returns per-sample losses (device).  `after_loss(loss)`, if
        given, is called as soon as the losses exist (the fused path runs it on a side stream).  `gate`: the sample's
        status words; a rejected batch leaves the parameters untouched (world 1)."""
        self._step_gate = gate if self.sync.world_size == 1 else None
        if self._fused_path(batch[1].shape[0]):
            return self._update_fused(batch, target_noise, after_loss)
        idxs, states, actions, returns, next_states, nonterminals, weights = batch
        q_s = self.online_net.logits(states)
        with torch.no_grad():
            q_ns = self.online_net.logits(next_states)
            if target_noise is None:
                self.target_net.reset_noise()
            else:
                self.target_net.reset_noise(*target_noise)
            q_t = self.target_net.logits(next_states)
            loss, grad = c51_loss_grad(q_s.detach(), q_ns, q_t, actions, returns, nonterminals, weights, self.support,
                                       self.Vmin, self.Vmax, self.delta_z, self.discount ** self.n)
        self.optimiser.zero_grad()
        q_s.backward(grad)
        self.sync.all_reduce_(self.optimiser.flat_grad)
        self.optimiser.step(grad_scale=1.0 / self.sync.world_size, gate=self._step_gate)
        if after_loss is not None:
            after_loss(loss)
        return loss

    def _learn_eager(self, mem):
        batch = mem.sample(self.batch_size)
        if isinstance(mem, ReplayMemory):
            gate = mem.sample_gate()
            return self._update_from_batch(batch, after_loss=lambda loss: mem.update_priorities(batch[0], loss, gate=gate),
                                           gate=gate)
        loss = self._update_from_batch(batch)
        mem.update_priorities(batch[0], loss.detach().cpu().numpy())  # a foreign (reference-style, host) memory: agent.py:100
        return loss

    def _capture(self, mem):
        """Record one whole update (sample -> ... -> priority write-back) into a CUDA graph.  Capturing does
        not execute; the caller replays."""
        ws = _SampleWorkspace(self.batch_size, mem.history, self.device)
        mem.flush_appends()
        mem.push_beta()  # outside the capture: a captured fill_ would freeze beta at today's value
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            batch = mem.sample_into(ws)
            loss = self._update_from_batch(batch, after_loss=lambda l: mem.update_priorities(batch[0], l, gate=ws.status),
                                           gate=ws.status)
        return graph, ws, loss

    @property
    def _graph(self):
        """Any captured update graph (None before the first capture)."""
        return next(iter(self._graphs.values()))[0] if self._graphs else None

    GRAPH_WARMUP = 2  # eager updates before capture (cuDNN/cuBLAS plan selection, autograd buffers)

    def learn(self, mem):
        """agent.py:61-100.  Exactly one update per call: the first GRAPH_WARMUP calls run eagerly on a side
        stream (torch's documented warm-up recipe for whole-step capture), the next call captures the graph and
        every call from then on is one graph launch."""
        # the captured graph bakes in: this memory's buffers, the batch size and training-mode (noisy) weights
        graphable = (self.use_cuda_graph and isinstance(mem, ReplayMemory) and mem.rng == "philox" and
                     self.online_net.training)
        # weak reference: the agent must not keep a dropped 7 GB replay alive; a dead or different referent, or another
        # batch size, invalidates the captured graph (a recycled id() can never alias a dead memory's graph)
        if graphable and (self._graph_key is None or self._graph_key[0]() is not mem or self._graph_key[1] != self.batch_size):
            self._graphs, self._graph_key, self._warm = {}, (weakref.ref(mem), self.batch_size), 0
        if not graphable:
            self.last_loss = self._learn_eager(mem)
        elif not self._graphs and self._warm < self.GRAPH_WARMUP:
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):
                self.last_loss = self._learn_eager(mem)
            torch.cuda.current_stream(self.device).wait_stream(side)
            self._warm += 1
        else:
            # two variants of the graph: with the online net's deferred reset_noise() as a side branch (the usual
            # `reset_noise(); learn()` pair) and without it (an act() in between has already launched the draw)
            pending = bool(self.online_net._noise_pending)
            if pending not in self._graphs:
                self._graphs[pending] = self._capture(mem)
            graph, ws, loss = self._graphs[pending]
            mem.flush_appends()   # no-op unless the memory defers its appends
            mem.push_beta()
            graph.replay()
            self.online_net._noise_pending = False
            self.online_net._eps_stale = self.online_net._eps_stale or pending
            self.last_loss, mem._last = loss, ws
        self._learn_calls += 1
        if self._learn_calls % 4096 == 0 and isinstance(mem, ReplayMemory):
            # diagnostics only (the device already skipped such updates): how many batches stayed invalid after
            # max_attempts redraws -- a ring that is too empty around the write head, or zero-priority leaves
            rejected = mem.rejected_batches()
            if rejected > self._rejected_seen:
                warnings.warn(f"rainbow_b200: {rejected - self._rejected_seen} sampled batches were rejected "
                              f"{mem.max_attempts} times in a row and skipped (no update, no priority write-back)")
            self._rejected_seen = rejected
