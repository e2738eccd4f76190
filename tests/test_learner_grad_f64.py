"""The learner's gradients against a float64 model of one update, and the head kernels at their edges against float64.

The model (Net64, c51_f64) is written here from the update's definition: the convs, noisy layers composed from the net's
factor vectors (W = mu + sigma * outer(f_out, f_in); mu only in eval mode), the dueling combination, softmax / log_softmax,
the C51 target with the double-DQN arg-max and the l / u projection including its l == u fix-up, loss = mean(w * loss_i),
parameter gradients from torch autograd in float64.

Two discontinuities would otherwise make a correct fp32 learner disagree with float64:
 * a ReLU whose pre-activation is within rounding of zero: its mask may differ between fp32 and float64, which moves a whole
   activation's gradient (~1e-6) in or out of the layers below.  The model's backward therefore takes the masks of the
   gradient-carrying pass (online net on s) from the GPU forward, and a separate assertion requires the forced masks to agree
   with float64's own signs everywhere except where |pre-activation| <= 1e-5 * the layer's max;
 * the double-DQN arg-max: every fixture is seeded on the CPU (parameters from torch.manual_seed at construction, noise
   injected as raw normals, batch from a CPU generator), and a CPU test requires every sample's top-two online q(s', .) to
   be at least 1e-4 apart in float64.

The CPU tests check the model itself against the reference's recorded values (tests/golden/learn.npz: loss, projection,
arg-max and logit gradient of 5 cases; tests/golden/model_step.npz: one whole update of a data-efficient net).
Observed maxima are recorded with test_gpu_update.record, beside those of the other parity tests."""
import ctypes as C
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import golden, manifest
from test_gpu_parity import FakeEnv, make_args

DEV = "cuda:0"
F64 = torch.float64

# Bounds of the comparisons, about 4x above the worst a B200 showed (DESIGN.md, "Learner gradients against float64").
# Relative to the reference tensor: max |got - ref| / max |ref| and ||got - ref||_2 / ||ref||_2.
GRAD_MAX, GRAD_L2 = 7e-6, 7e-6          # whole update, noisy-head tensors (observed 1.6e-6 / 1.6e-6)
CONV_MAX, CONV_L2 = 2e-5, 2e-5          # whole update, conv tensors: sums over up to 400 B signed terms behind three fp32
                                        # data-gradient layers (observed 5.2e-6 / 4.4e-6, conv 0 of canonical at B 7)
LOSS_ABS = 6e-6                         # whole update, per-sample loss, absolute (observed 1.4e-6)
FWD_MAX, FWD_L2 = 4e-6, 4e-6            # rb_head_forward h and z (observed 1.1e-6 / 0.9e-6)
BWD_MAX, BWD_L2 = 1e-5, 1e-5            # rb_head_backward gradients and dx (observed 2.4e-6 / 2.2e-6, dx at A*Z = 1062)
LOGIT_ABS = 5e-6                        # rb_head_logits, absolute, logits of unit scale (observed 1.2e-6)
QV_ABS = 2.5e-5                         # rb_q_values / q_select, absolute, q within [-10, 10] (observed 5.6e-6)
BIAS_SUM = 2e-7                         # rb_bias_grad: |got - ref| <= BIAS_SUM * sum |terms| per channel (observed 5.3e-8)
NEAR_ZERO = 1e-5                        # ReLU units with |pre| <= NEAR_ZERO * layer max may flip between fp32 and float64
ARGMAX_GAP = 1e-4


def record(name, values):
    from test_gpu_update import record as rec
    rec(name, values)


# ------------------------------------------------------------------------------------------------------------------------
# the float64 model
def relu_forced(y, mask):
    return torch.relu(y) if mask is None else y * mask.to(y.dtype)


class Net64:
    """float64 copy of a DQN: its parameters (leaves with requires_grad) and, in training mode, its current noise factors."""

    def __init__(self, net, noisy=True, device=None):
        dev = device if device is not None else next(net.parameters()).device
        self.p = {k: v.detach().to(dev, F64).clone().requires_grad_(True) for k, v in net.named_parameters()}
        self.strides = [m.stride[0] for m in net.conv_layers()]
        self.f = {k: (fi.detach().to(dev, F64), fo.detach().to(dev, F64)) for k, (fi, fo) in net.noise_factors().items()} \
            if noisy else None
        self.A, self.Z, self.H = net.action_space, net.atoms, net.hidden_size

    def linear(self, name, x):
        w, b = self.p[name + ".weight_mu"], self.p[name + ".bias_mu"]
        if self.f is not None:
            fi, fo = self.f[name]
            w = w + self.p[name + ".weight_sigma"] * torch.outer(fo, fi)
            b = b + self.p[name + ".bias_sigma"] * fo
        return x @ w.t() + b

    def features(self, x, masks=None, pre=None):
        a = x.to(F64)
        for i, s in enumerate(self.strides):
            y = F.conv2d(a, self.p[f"convs.{2 * i}.weight"], self.p[f"convs.{2 * i}.bias"], stride=s)
            if pre is not None:
                pre.append(y.detach())
            a = relu_forced(y, None if masks is None else masks[i])
        return a.reshape(a.shape[0], -1)

    def head(self, f, h_mask=None, pre=None):
        """conv features [M, K1] -> (z = (z_value | z_advantage) [M, Z(1+A)], h [M, 2H])"""
        hp = torch.cat([self.linear("fc_h_v", f), self.linear("fc_h_a", f)], 1)
        if pre is not None:
            pre.append(hp.detach())
        h = relu_forced(hp, h_mask)
        z = torch.cat([self.linear("fc_z_v", h[:, :self.H]), self.linear("fc_z_a", h[:, self.H:])], 1)
        return z, h

    def logits(self, x, masks=None, pre=None):
        """x [B, C, 84, 84] -> q [B, A, Z].  masks: forced ReLU masks (conv layers..., head hidden [B, 2H]) or None."""
        L = len(self.strides)
        f = self.features(x, None if masks is None else masks[:L], pre)
        z, _ = self.head(f, None if masks is None else masks[L], pre)
        return dueling(z, self.A, self.Z)


def dueling(z, A, Z):
    v, a = z[:, :Z].reshape(-1, 1, Z), z[:, Z:].reshape(-1, A, Z)
    return v + a - a.mean(1, keepdim=True)


def c51_f64(q_s, q_ns, q_t, actions, returns, nonterm, weights, support, vmin, vmax, delta_z, gamma_n):
    """The C51 update on logits [B, A, Z] (all float64): per-sample loss, mean(w * loss), projected target m, a*."""
    B, A, Z = q_s.shape
    rows = torch.arange(B, device=q_s.device)
    with torch.no_grad():
        astar = (F.softmax(q_ns, 2) * support).sum(2).argmax(1)                 # double DQN: online net picks a*
        p_t = F.softmax(q_t, 2)[rows, astar]
        Tz = (returns.reshape(B, 1) + nonterm.reshape(B, 1) * gamma_n * support.reshape(1, Z)).clamp(vmin, vmax)
        b = (Tz - vmin) / delta_z
        lo, up = b.floor().long(), b.ceil().long()
        lo[(up > 0) & (lo == up)] -= 1                                           # b integral: keep the mass
        up[(lo < Z - 1) & (lo == up)] += 1
        m = torch.zeros(B, Z, dtype=F64, device=q_s.device)
        m.scatter_add_(1, lo, p_t * (up.to(F64) - b))
        m.scatter_add_(1, up, p_t * (b - lo.to(F64)))
    loss = -(m * F.log_softmax(q_s, 2)[rows, actions]).sum(1)
    return loss, (weights * loss).mean(), m, astar


def rel_err(got, ref):
    """(max |got - ref| / max |ref|, ||got - ref|| / ||ref||) in float64; NaN anywhere in `got` gives NaN."""
    got, ref = got.detach().to(F64), ref.detach().to(got.device, F64)
    d = got - ref
    return float(d.abs().max() / ref.abs().max().clamp_min(1e-300)), float(d.norm() / ref.norm().clamp_min(1e-300))


def within(got, ref, max_tol, l2_tol):
    e_max, e_l2 = rel_err(got, ref)
    return e_max <= max_tol and e_l2 <= l2_tol       # False for NaN


def grad_bounds(name):
    return (CONV_MAX, CONV_L2) if name.startswith("convs") else (GRAD_MAX, GRAD_L2)


def grad_excess(errs):
    return [f"{k}: max {e[0]:.2e} l2 {e[1]:.2e}" for k, e in errs.items()
            if not (e[0] <= grad_bounds(k)[0] and e[1] <= grad_bounds(k)[1])]


def mask_disagreements(gpu_mask, pre64):
    """Forced masks vs float64's signs: (units that disagree beyond the near-zero band, units inside the band)."""
    band = pre64.abs() <= NEAR_ZERO * float(pre64.abs().max())
    differ = gpu_mask.to(pre64.device) != (pre64 > 0)
    return int((differ & ~band).sum()), int(band.sum())


# ------------------------------------------------------------------------------------------------------------------------
# seeded fixtures
UpdateCase = SimpleNamespace
UPDATE_CASES = [
    # fused path (B <= 32, head within the backward kernels' limits)
    UpdateCase(id="c_512_a6_z51_b1", arch="canonical", hidden=512, A=6, Z=51, B=1, seed=11, fused=True),
    UpdateCase(id="c_512_a6_z51_b7", arch="canonical", hidden=512, A=6, Z=51, B=7, seed=12, fused=True),
    UpdateCase(id="c_512_a6_z51_b32", arch="canonical", hidden=512, A=6, Z=51, B=32, seed=113, fused=True),
    UpdateCase(id="de_256_a18_z51_b5", arch="data-efficient", hidden=256, A=18, Z=51, B=5, seed=14, fused=True),
    UpdateCase(id="de_256_a18_z51_b31", arch="data-efficient", hidden=256, A=18, Z=51, B=31, seed=115, fused=True),
    UpdateCase(id="de_64_a3_z101_b17", arch="data-efficient", hidden=64, A=3, Z=101, B=17, seed=16, fused=True),
    UpdateCase(id="c_128_a18_z59_b32", arch="canonical", hidden=128, A=18, Z=59, B=32, seed=17, fused=True),  # A*Z = 1062
    # library path for the online pass on s (B > 32)
    UpdateCase(id="c_512_a6_z51_b512", arch="canonical", hidden=512, A=6, Z=51, B=512, seed=218, fused=False),   # C4
    UpdateCase(id="de_256_a6_z51_b33", arch="data-efficient", hidden=256, A=6, Z=51, B=33, seed=19, fused=False),
]
# shapes around the head kernels' limits: learn() must route them to a path that runs and stays correct
ROUTING_CASES = [
    UpdateCase(id="de_128_a18_z59_b32", arch="data-efficient", hidden=128, A=18, Z=59, B=32, seed=121, fused=True),
    UpdateCase(id="de_128_a18_z60_b32", arch="data-efficient", hidden=128, A=18, Z=60, B=32, seed=22, fused=False),
    UpdateCase(id="de_128_a18_z128_b32", arch="data-efficient", hidden=128, A=18, Z=128, B=32, seed=23, fused=False),
    UpdateCase(id="de_1024_a6_z51_b32", arch="data-efficient", hidden=1024, A=6, Z=51, B=32, seed=124, fused=True),
    UpdateCase(id="de_1088_a6_z51_b32", arch="data-efficient", hidden=1088, A=6, Z=51, B=32, seed=125, fused=False),
]


def case_args(c, **kw):
    return make_args(architecture=c.arch, hidden_size=c.hidden, atoms=c.Z, batch_size=c.B, multi_step=3, cuda_graph=False, **kw)


def noisy_sizes(net):
    layers = net.noisy_layers()
    return sum(m.in_features for m in layers), sum(m.out_features for m in layers)


def factors(x):
    return x.sign() * x.abs().sqrt()


def make_inputs(c, n_in, n_out):
    """Raw noise normals (online, target) and the batch, from a CPU generator.  Returns and terminal flags include the
    clamps at V_min and V_max (exactly and beyond) and one zero importance weight."""
    g = torch.Generator().manual_seed(1000 + c.seed)
    noise = [torch.randn(n, generator=g) for n in (n_in, n_out, n_in, n_out)]
    B = c.B
    both = torch.randint(0, 256, (2 * B, 4, 84, 84), generator=g).float() / 255
    actions = torch.randint(0, c.A, (B,), generator=g)
    returns = torch.rand(B, generator=g) * 6 - 3
    nonterm = torch.ones(B, 1)
    weights = torch.rand(B, generator=g) * 0.9 + 0.1
    i = torch.arange(B)
    returns[i % 6 == 0], nonterm[i % 6 == 0] = 10.0, 0.0      # Tz = V_max exactly
    returns[i % 6 == 1], nonterm[i % 6 == 1] = -10.0, 0.0     # Tz = V_min exactly
    returns[i % 6 == 3] = 25.0                                 # every atom clamps to V_max
    returns[i % 6 == 4] = -25.0                                # ... to V_min
    weights[i % 6 == 2] = 0.0
    return noise, both, actions, returns, nonterm, weights


def cpu_fixture(c):
    """The online net exactly as Agent builds it under torch.manual_seed(c.seed) (its parameters are drawn first), with the
    injected online noise, on the CPU; plus the batch."""
    from rainbow_b200.model import DQN
    torch.manual_seed(c.seed)
    net = DQN(case_args(c, device=torch.device("cpu")), c.A)
    n_in, n_out = noisy_sizes(net)
    noise, both, actions, returns, nonterm, weights = make_inputs(c, n_in, n_out)
    with torch.no_grad():
        net._f_in.copy_(factors(noise[0]))
        net._f_out.copy_(factors(noise[1]))
    return net, noise, both, actions, returns, nonterm, weights


def top_two_gap(q):
    """q [B, A] -> gap between the largest and second-largest value per row (inf for one action)."""
    if q.shape[1] < 2:
        return torch.full((q.shape[0],), math.inf, dtype=q.dtype)
    t = q.topk(2, 1).values
    return t[:, 0] - t[:, 1]


# ------------------------------------------------------------------------------------------------------------------------
# CPU: the model against the reference's recorded values, and the fixtures' arg-max margins
@pytest.mark.parametrize("case", manifest()["learn_cases"], ids=lambda c: c["name"])
def test_f64_c51_against_reference_golden(case):
    g = golden("learn")
    p = case["name"] + "_"
    d = lambda k: torch.from_numpy(np.ascontiguousarray(g[p + k])).to(F64)
    q_s = d("q_s").requires_grad_(True)
    loss, total, m, astar = c51_f64(q_s, d("q_ns"), d("q_t"), torch.from_numpy(g[p + "actions"]), d("returns"), d("nonterm"),
                                    d("weights"), d("support"), case["V_min"], case["V_max"], case["delta_z"],
                                    case["discount"] ** case["n"])
    grad, = torch.autograd.grad(total, q_s)
    assert np.array_equal(astar.numpy(), g[p + "astar"])
    # the reference computed in fp32: its b = (Tz - V_min) / dz carries ~ulp(50) into m (observed <= 4.5e-6)
    np.testing.assert_allclose(m.numpy(), g[p + "m"], rtol=0, atol=1e-5)
    np.testing.assert_allclose(loss.detach().numpy(), g[p + "loss"], rtol=4e-6, atol=4e-6)
    np.testing.assert_allclose(grad.numpy(), g[p + "grad"], rtol=0, atol=5e-7)
    np.testing.assert_allclose(m.sum(1).numpy(), 1.0, rtol=0, atol=1e-12)


def test_f64_update_against_reference_golden():
    """One whole update of the unmodified reference (tests/golden/model_step.npz: data-efficient / 64, B 4, A 3, CPU fp32)
    through Net64 + c51_f64: the model's convs, noisy layers, dueling head, target and autograd are those of the update."""
    from rainbow_b200.model import DQN
    g = golden("model_step")
    B, A = 4, 3
    net = DQN(make_args(batch_size=B, architecture="data-efficient", hidden_size=64, device=torch.device("cpu")), A)
    net.load_state_dict({k[4:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd0.")})   # recovers the factors
    tgt = DQN(make_args(batch_size=B, architecture="data-efficient", hidden_size=64, device=torch.device("cpu")), A)
    tgt.load_state_dict({k[4:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd0.")})
    with torch.no_grad():
        tgt._f_in.copy_(factors(torch.from_numpy(np.concatenate([g[f"target_randn{2 * i}"] for i in range(4)]))))
        tgt._f_out.copy_(factors(torch.from_numpy(np.concatenate([g[f"target_randn{2 * i + 1}"] for i in range(4)]))))
    on64, tg64 = Net64(net), Net64(tgt)
    s = torch.from_numpy(g["states_u8"]).to(F64) / 255
    ns = torch.from_numpy(g["nstates_u8"]).to(F64) / 255
    support = torch.linspace(-10, 10, 51).to(F64)
    q_s = on64.logits(s)
    with torch.no_grad():
        q_ns, q_t = on64.logits(ns), tg64.logits(ns)
    f = lambda k: torch.from_numpy(g[k]).to(F64)
    loss, total, _, _ = c51_f64(q_s, q_ns, q_t, torch.from_numpy(g["actions"]), f("returns"), f("nonterm"), f("weights"),
                                support, -10.0, 10.0, 0.4, 0.99 ** 3)
    grads = torch.autograd.grad(total, list(on64.p.values()))
    np.testing.assert_allclose(loss.detach().numpy(), g["loss"], rtol=0, atol=2e-6)
    for (k, _), gr in zip(on64.p.items(), grads):
        ref = torch.from_numpy(g["grad." + k])
        assert within(gr, ref, 2e-5, 2e-6), (k, rel_err(gr, ref))


def test_head_supported_at_the_limits():
    """rb_head_supported (host only) on either side of each limit of the head kernels."""
    from rainbow_b200 import _lib
    q = _lib.load().rb_head_supported
    assert q(3136, 512, 51, 6, 64, 0) == 0 and q(3136, 512, 51, 6, 32, 1) == 0
    assert q(3136, 512, 51, 6, 33, 1) == -34                                          # backward: B <= 32
    assert q(3136, 128, 59, 18, 32, 1) == 0 and q(3136, 128, 60, 18, 32, 1) == -34     # dh kernel: A * Z <= 1065
    assert q(3136, 128, 60, 18, 64, 0) == 0                                           # ... the forward takes it
    assert q(3136, 1024, 51, 6, 32, 1) == 0 and q(3136, 1088, 51, 6, 32, 1) == -34     # layer-1 backward: hidden <= 1024
    assert q(576, 64, 128, 18, 2048, 0) == 0 and q(576, 64, 128, 18, 4096, 0) == -34   # forward tile count
    assert q(576, 1088, 51, 6, 64, 0) == 0 and q(576, 1088, 51, 6, 4096, 0) == -34
    assert q(576, 64, 128, 3, 8, 0) == 0 and q(576, 64, 129, 3, 8, 0) == -34           # RB_MAX_ATOMS
    assert q(560, 64, 51, 6, 8, 0) == -34 and q(576, 96, 51, 6, 8, 0) == -34           # conv_features % 32, hidden % 64
    assert q(576, 64, 51, 6, 0, 0) == -22


@pytest.mark.parametrize("c", UPDATE_CASES + ROUTING_CASES, ids=lambda c: c.id)
def test_fixture_argmax_margin(c):
    """The double-DQN arg-max of every fixture sample is clear by ARGMAX_GAP in float64, so fp32 cannot pick another a*."""
    net, _, both, *_ = cpu_fixture(c)
    with torch.no_grad():
        q = Net64(net).logits(both[c.B:])
        support = torch.linspace(-10, 10, c.Z).to(F64)
        gap = top_two_gap((F.softmax(q, 2) * support).sum(2))
    assert float(gap.min()) >= ARGMAX_GAP, f"seed {c.seed}: smallest top-two gap {float(gap.min()):.2e}"


# ------------------------------------------------------------------------------------------------------------------------
# GPU: the whole update against the float64 model
def gpu_update(c, adjacent=True, fused_head=True):
    """Agent under torch.manual_seed(c.seed), online noise injected, optimiser step replaced by a no-op, flat gradient
    filled with NaN; runs Agent._update_from_batch on the fixture batch.  Returns what the comparison needs."""
    from rainbow_b200.agent import Agent
    torch.manual_seed(c.seed)
    ag = Agent(case_args(c, batch_online_convs=adjacent, fused_head=fused_head), FakeEnv(c.A))
    on, tg = ag.online_net, ag.target_net
    n_in, n_out = noisy_sizes(on)
    noise, both, actions, returns, nonterm, weights = make_inputs(c, n_in, n_out)
    on.reset_noise(noise[0].to(DEV), noise[1].to(DEV))
    both = both.to(DEV)
    if adjacent:
        states, next_states = both[:c.B], both[c.B:]
        assert ag._adjacent(states, next_states) is not None
    else:
        states, next_states = both[:c.B].clone(), both[c.B:].clone()
    batch = (torch.arange(c.B, device=DEV), states, actions.to(DEV), returns.to(DEV), next_states, nonterm.to(DEV),
             weights.to(DEV))
    ag.optimiser.step = lambda *a, **k: None            # flat_grad keeps exactly what Adam would have seen
    ag.optimiser.flat_grad.fill_(float("nan"))
    fused = ag._fused_path(c.B)
    loss = ag._update_from_batch(batch, target_noise=(noise[2].to(DEV), noise[3].to(DEV)))
    torch.cuda.synchronize()
    # the ReLU masks of the gradient-carrying pass, from the same kernels on the same input
    with torch.no_grad():
        if fused and on.manual_conv_ok(states):
            acts = on.conv_forward_saving(both if adjacent else states)[1:]
            if adjacent:
                _, h, _ = on.head().forward(acts[-1].reshape(2 * c.B, -1))
            else:
                _, h, _ = on.head().forward(acts[-1].reshape(c.B, -1), on.features_nograd(next_states).contiguous())
            acts = [a[:c.B] for a in acts]
            h = h[:c.B].clone()
        else:
            a, acts = states, []
            for i in range(0, len(on.convs), 2):
                a = on.convs[i + 1](on.convs[i](a))
                acts.append(a)
            feats = a.reshape(c.B, -1)
            on.materialise_noise()
            h = torch.cat([on.fc_h_v(feats), on.fc_h_a(feats)], 1)
        masks = [a > 0 for a in acts] + [h > 0]
    return ag, fused, loss.clone(), states, next_states, batch, masks


def compare_update(c, ag, loss, states, next_states, batch, masks, noisy=True):
    """Float64 model of the update that ran: per-sample loss error, per-tensor gradient errors, mask statistics."""
    on, tg = ag.online_net, ag.target_net
    on64, tg64 = Net64(on, noisy=noisy), Net64(tg, noisy=noisy)
    pre = []
    q_s = on64.logits(states, masks=masks, pre=pre)
    with torch.no_grad():
        q_ns, q_t = on64.logits(next_states), tg64.logits(next_states)
    _, _, actions, returns, _, nonterm, weights = batch
    support = ag.support.to(F64)
    loss64, total, _, astar = c51_f64(q_s, q_ns, q_t, actions, returns.to(F64), nonterm.to(F64), weights.to(F64), support,
                                      ag.Vmin, ag.Vmax, ag.delta_z, ag.discount ** ag.n)
    names = list(on64.p)
    grads = torch.autograd.grad(total, [on64.p[k] for k in names], allow_unused=True)     # sigma unused in eval mode
    grads = {k: torch.zeros_like(on64.p[k]) if g is None else g for k, g in zip(names, grads)}
    # the forced masks may only differ from float64's own signs inside the near-zero band
    flips, near = [], []
    for m, p in zip(masks, pre):
        f, n = mask_disagreements(m, p)
        flips.append(f)
        near.append(n)
    errs = {k: rel_err(dict(on.named_parameters())[k].grad, grads[k]) for k in names}
    loss_err = float((loss.to(F64) - loss64.detach()).abs().max())
    return dict(loss=loss_err, errs=errs, flips=flips, near=near, grads=grads)


UPDATE_PARAMS = [pytest.param(c, adj, id=f"{c.id}-{'adjacent' if adj else 'separate'}")
                 for c in UPDATE_CASES for adj in ((True, False) if c.fused else (True,))]


@pytest.mark.gpu
@pytest.mark.parametrize("c,adjacent", UPDATE_PARAMS)
def test_update_gradient_vs_float64(c, adjacent):
    """Agent._update_from_batch: every parameter's full gradient tensor and the per-sample loss against float64."""
    old = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True      # the non-fused path's masks are recomputed through the same cuDNN calls
    obs = {}
    try:
        ag, fused, loss, states, next_states, batch, masks = gpu_update(c, adjacent)
        assert fused == c.fused, "fixture routed to the other path"
        for k, p in ag.online_net.named_parameters():
            assert bool(torch.isfinite(p.grad).all()), f"{k}: gradient not (fully) written"
        r = compare_update(c, ag, loss, states, next_states, batch, masks)
        worst = max(r["errs"], key=lambda k: r["errs"][k][0])
        obs = dict(loss=r["loss"], grad_max=max(e[0] for e in r["errs"].values()),
                   grad_l2=max(e[1] for e in r["errs"].values()), worst_tensor=worst, near_zero_relu=r["near"],
                   mask_flips_outside_band=r["flips"], by_tensor={k: [round(e[0], 10), round(e[1], 10)] for k, e in r["errs"].items()})
        assert r["flips"] == [0] * len(masks), f"GPU ReLU masks differ from float64 outside the near-zero band: {r['flips']}"
        assert r["loss"] <= LOSS_ABS, f"loss off by {r['loss']:.2e}"
        bad = grad_excess(r["errs"])
        assert not bad, "\n".join(bad)
        # negative control: one element moved by twice the bound is caught
        k = worst
        g = dict(ag.online_net.named_parameters())[k].grad.clone()
        ref = r["grads"][k]
        g.view(-1)[int(ref.abs().argmax())] += 2 * grad_bounds(k)[0] * float(ref.abs().max())
        assert not within(g, ref, *grad_bounds(k))
    finally:
        torch.backends.cudnn.deterministic = old
        record(f"f64_update_{c.id}_{'adjacent' if adjacent else 'separate'}", obs)


@pytest.mark.gpu
def test_update_comparison_rejects_eval_weights():
    """Negative control: the same update compared with a model that uses eval-mode (mu only) weights must fail."""
    c = UPDATE_CASES[3]
    ag, _, loss, states, next_states, batch, masks = gpu_update(c)
    r = compare_update(c, ag, loss, states, next_states, batch, masks, noisy=False)
    assert grad_excess(r["errs"]), "eval-mode weights passed the comparison"


@pytest.mark.gpu
@pytest.mark.parametrize("c", ROUTING_CASES, ids=lambda c: c.id)
def test_learn_routes_unsupported_head_shapes(c):
    """Shapes around the head kernels' limits (actions * atoms vs the dh kernel, hidden <= 1024): learn() picks a path that
    runs, and the update matches float64."""
    from rainbow_b200 import _lib
    from rainbow_b200.agent import Agent
    from test_gpu_parity import synthetic_ring
    lib = _lib.load()
    K1 = 576 if c.arch == "data-efficient" else 3136
    assert (lib.rb_head_supported(K1, c.hidden, c.Z, c.A, c.B, 1) == 0) == c.fused
    # through the public API once: sample, update, Adam step, priority write-back
    torch.manual_seed(c.seed)
    ag = Agent(case_args(c), FakeEnv(c.A))
    mem, _ = synthetic_ring(1024, seed=c.seed, args=dict())
    ag.reset_noise()
    ag.learn(mem)
    torch.cuda.synchronize()
    assert torch.isfinite(ag.last_loss).all() and int(ag.optimiser.step_count.item()) == 1
    # and against the float64 model on the fixture batch
    old = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        ag, fused, loss, states, next_states, batch, masks = gpu_update(c)
        assert fused == c.fused
        r = compare_update(c, ag, loss, states, next_states, batch, masks)
    finally:
        torch.backends.cudnn.deterministic = old
    record(f"f64_routing_{c.id}", dict(loss=r["loss"], grad_max=max(e[0] for e in r["errs"].values()),
                                       grad_l2=max(e[1] for e in r["errs"].values()), near_zero_relu=r["near"],
                                       worst_tensor=max(r["errs"], key=lambda k: r["errs"][k][0])))
    assert r["flips"] == [0] * len(masks)
    assert r["loss"] <= LOSS_ABS
    bad = grad_excess(r["errs"])
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,A,Z", [(64, 18, 128), (1088, 6, 51), (64, 6, 51)])
def test_q_select_routes_unsupported_row_counts(hidden, A, Z):
    """q_select over 4096 states: where the forward's tile count refuses the head (A18 x Z128, hidden 1088) the library path
    answers; either way the greedy action and value match float64."""
    from rainbow_b200 import _lib
    from rainbow_b200.agent import Agent
    N = 4096
    torch.manual_seed(31)
    ag = Agent(make_args(architecture="data-efficient", hidden_size=hidden, atoms=Z, cuda_graph=False), FakeEnv(A))
    on = ag.online_net
    n_in, n_out = noisy_sizes(on)
    g = torch.Generator().manual_seed(32)
    on.reset_noise(torch.randn(n_in, generator=g).to(DEV), torch.randn(n_out, generator=g).to(DEV))
    states = (torch.randint(0, 256, (N, 4, 84, 84), generator=g).float() / 255).to(DEV)
    supported = _lib.load().rb_head_supported(576, hidden, Z, A, N, 0) == 0
    assert supported == (hidden == 64 and Z == 51)
    q_out = torch.empty(N, A, device=DEV)
    best_a, best_q = ag.q_select(states, q_out=q_out)
    torch.cuda.synchronize()
    with torch.no_grad():
        q64 = (F.softmax(Net64(on).logits(states), 2) * ag.support.to(F64)).sum(2)
    np.testing.assert_allclose(q_out.cpu().numpy(), q64.cpu().numpy(), rtol=0, atol=QV_ABS)
    np.testing.assert_allclose(best_q.cpu().numpy(), q64.max(1).values.cpu().numpy(), rtol=0, atol=QV_ABS)
    clear = (top_two_gap(q64.cpu()) > 2 * QV_ABS).numpy()
    assert np.array_equal(best_a.cpu().numpy()[clear], q64.argmax(1).cpu().numpy()[clear])


# ------------------------------------------------------------------------------------------------------------------------
# GPU: the head kernels at their edges, against float64
def head_net(arch, hidden, A, Z, seed=0):
    from rainbow_b200.model import DQN
    torch.manual_seed(seed)
    net = DQN(make_args(architecture=arch, hidden_size=hidden, atoms=Z), A).to(DEV)
    with torch.no_grad():                   # sigma well away from its initial value, so the noise terms matter
        for m in net.noisy_layers():
            m.weight_sigma.mul_(torch.empty_like(m.weight_sigma).uniform_(0.5, 3.0))
            m.bias_sigma.mul_(torch.empty_like(m.bias_sigma).uniform_(0.5, 3.0))
    net.reset_noise()
    return net


GUARD = 4096


def raw_forward(net, x_lo, x_hi, noisy):
    """rb_head_forward into h / z buffers followed by GUARD sentinel elements."""
    from rainbow_b200 import _lib
    hd = net.head()
    M = x_lo.shape[0] + (0 if x_hi is None else x_hi.shape[0])
    H, ncols = net.hidden_size, hd.ncols
    buf = hd._buffers(M, x_lo.device)             # split-K scratch and the tickets
    h = torch.full((M * 2 * H + GUARD,), 777.0, device=DEV)
    z = torch.full((M * ncols + GUARD,), 777.0, device=DEV)
    p = hd.params(noisy)
    _lib.check(hd.lib.rb_head_forward(C.byref(p), _lib.ptr(x_lo), x_lo.shape[0], _lib.ptr(x_hi), M - x_lo.shape[0],
                                      _lib.ptr(buf["part1"]), _lib.ptr(buf["part2"]), _lib.ptr(hd._tickets), _lib.ptr(h),
                                      _lib.ptr(z), _lib.stream()))
    return h, z, M


@pytest.mark.gpu
@pytest.mark.parametrize("hidden,A,Z", [(64, 1, 2), (64, 18, 101), (64, 18, 128), (1024, 1, 128), (1024, 18, 51), (1024, 18, 2)])
@pytest.mark.parametrize("rows", [1, 8, 31, 33, 65, 512, 4096])
def test_head_forward_vs_float64(hidden, A, Z, rows):
    """rb_head_forward (h and z) against float64 in training and eval mode, with every row split the learner and the act
    paths use: all rows in x_lo, m_lo % 8 != 0 with m_hi > 0 (FFMA layer 1), m_lo % 8 == 0 with m_hi > 0 (tensor cores), and
    the FFMA layer 1 forced.  Guard elements past h / z stay untouched, the tickets return to zero, and a second launch is
    bit-identical.  Shapes the kernel refuses must be refused cleanly, as rb_head_supported says."""
    from rainbow_b200 import _lib
    lib = _lib.load()
    net = head_net("data-efficient", hidden, A, Z, seed=rows)
    torch.manual_seed(rows + 1)
    x = torch.randn(rows, 576, device=DEV).relu()
    if lib.rb_head_supported(576, hidden, Z, A, rows, 0) != 0:
        with pytest.raises(_lib.RainbowB200Error, match="too many rows"):
            raw_forward(net, x, None, True)
        return
    splits = [("lo", rows)]
    if rows > 1:
        splits += [("odd", (rows // 2) | 1 if (rows // 2) % 8 else rows // 2 + 1), ("tc8", max(8, (rows // 2) // 8 * 8))]
    splits = [(n, m) for n, m in splits if m == rows or 0 < m < rows]
    obs = {}
    for noisy in (True, False):
        net.train(noisy)
        n64 = Net64(net, noisy=noisy)
        with torch.no_grad():
            z64, h64 = n64.head(x.to(F64))
        for name, m_lo in splits + [("ffma", rows)]:
            x_lo, x_hi = x[:m_lo].contiguous(), (x[m_lo:].contiguous() if m_lo < rows else None)
            try:
                lib.rb_head_debug(4 if name == "ffma" else 0)
                h, z, M = raw_forward(net, x_lo, x_hi, noisy)
                h2, z2, _ = raw_forward(net, x_lo, x_hi, noisy)
            finally:
                lib.rb_head_debug(0)
            torch.cuda.synchronize()
            hb, zb = h[:M * 2 * hidden].view(M, -1), z[:M * net.head().ncols].view(M, -1)
            assert bool((h[M * 2 * hidden:] == 777.0).all()) and bool((z[M * net.head().ncols:] == 777.0).all()), "wrote past the end"
            assert int(net.head()._tickets.abs().sum()) == 0, "split-K tickets are self-resetting"
            assert torch.equal(h, h2) and torch.equal(z, z2), "second launch differs"
            eh, ez = rel_err(hb, h64), rel_err(zb, z64)
            obs[f"{name}_{'train' if noisy else 'eval'}"] = [eh[0], eh[1], ez[0], ez[1]]
            assert within(hb, h64, FWD_MAX, FWD_L2), (name, noisy, "h", eh)
            assert within(zb, z64, FWD_MAX, FWD_L2), (name, noisy, "z", ez)
            if noisy and name == "lo":   # negative control: eval-mode weights are not the noisy answer
                with torch.no_grad():
                    z_eval, _ = Net64(net, noisy=False).head(x.to(F64))
                assert not within(zb, z_eval, FWD_MAX, FWD_L2)
    net.train()
    record(f"f64_head_forward_h{hidden}_a{A}_z{Z}_m{rows}", dict(worst=max(max(v) for v in obs.values()), by_split=obs))


@pytest.mark.gpu
@pytest.mark.parametrize("A,Z", [(1, 2), (1, 128), (6, 51), (18, 51), (18, 101), (18, 128)])
def test_head_logits_and_q_values_vs_float64(A, Z):
    """rb_head_logits (dueling combination) and rb_q_values (softmax expectation, arg-max, max) against float64."""
    from rainbow_b200 import _lib
    lib = _lib.load()
    M = 257
    torch.manual_seed(A * 1000 + Z)
    z = torch.randn(M, Z * (1 + A), device=DEV) * 2
    support = torch.linspace(-10, 10, Z).to(DEV)
    q = torch.full((M * A * Z + GUARD,), 777.0, device=DEV)
    _lib.check(lib.rb_head_logits(_lib.ptr(z), M, A, Z, _lib.ptr(q), _lib.stream()))
    qv = torch.full((M, A), 777.0, device=DEV)
    best_a = torch.full((M,), -1, dtype=torch.int64, device=DEV)
    best_q = torch.full((M,), 777.0, device=DEV)
    _lib.check(lib.rb_q_values(_lib.ptr(z), M, A, Z, _lib.ptr(support), _lib.ptr(qv), _lib.ptr(best_a), _lib.ptr(best_q),
                               _lib.stream()))
    torch.cuda.synchronize()
    logits64 = dueling(z.to(F64), A, Z)
    q64 = (F.softmax(logits64, 2) * support.to(F64)).sum(2)
    assert bool((q[M * A * Z:] == 777.0).all())
    e_logit = float((q[:M * A * Z].view(M, A, Z).to(F64) - logits64).abs().max())
    e_q = float((qv.to(F64) - q64).abs().max())
    e_best = float((best_q.to(F64) - q64.max(1).values).abs().max())
    record(f"f64_q_values_a{A}_z{Z}", dict(logits=e_logit, q=e_q, best_q=e_best))
    assert e_logit <= LOGIT_ABS and e_q <= QV_ABS and e_best <= QV_ABS, (e_logit, e_q, e_best)
    clear = top_two_gap(q64) > 2 * QV_ABS
    assert bool(clear.any())
    assert torch.equal(best_a[clear], q64.argmax(1)[clear])


HEAD_PARAM_NAMES = [f"{l}.{k}" for l in ("fc_h_v", "fc_h_a", "fc_z_v", "fc_z_a")
                    for k in ("weight_mu", "weight_sigma", "bias_mu", "bias_sigma")]


def head_backward_case(arch, hidden, A, Z, B, relu_mask_x=True):
    """The learner's head backward: forward on x (about half exactly 0), then BWD_WGRAD2 as its own launch and
    BWD_DH | BWD_LAYER1.  Returns (gpu results, float64 reference, dh scratch guard intact)."""
    net = head_net(arch, hidden, A, Z, seed=B)
    hd = net.head()
    K1 = net.conv_output_size
    torch.manual_seed(100 + B)
    x = torch.randn(B, K1, device=DEV).relu()
    dz = torch.randn(B, Z * (1 + A), device=DEV) * 0.1
    params = dict(net.named_parameters())
    for k in HEAD_PARAM_NAMES:
        params[k].grad = torch.full_like(params[k], float("nan"))      # overwritten, not accumulated
    n = (B + 32) * 2 * hidden
    scratch = torch.full((n + GUARD,), 777.0, device=DEV)
    dx = torch.full((B, K1), float("nan"), device=DEV)
    with torch.no_grad():
        _, h, p = hd.forward(x)
        h = h[:B].clone()
        hd.backward(p, x, h, dz, scratch, dx, relu_mask_x=relu_mask_x, parts=hd.BWD_WGRAD2)
        hd.backward(p, x, h, dz, scratch, dx, relu_mask_x=relu_mask_x, parts=hd.BWD_DH | hd.BWD_LAYER1)
    torch.cuda.synchronize()
    guard_ok = bool((scratch[n:] == 777.0).all())
    n64 = Net64(net)
    x64 = x.to(F64).requires_grad_(True)
    z64, _ = n64.head(x64, h_mask=h > 0)
    names = HEAD_PARAM_NAMES
    ref = torch.autograd.grad(z64, [x64] + [n64.p[k] for k in names], dz.to(F64))
    got = [dx] + [params[k].grad for k in names]
    ref = [ref[0] * (x > 0)] + list(ref[1:])              # dx w.r.t. the pre-activation of the ReLU that produced x
    return ["dx"] + names, got, ref, guard_ok


@pytest.mark.gpu
@pytest.mark.parametrize("arch,hidden,A,Z", [("data-efficient", 256, 3, 51), ("canonical", 512, 18, 59)], ids=["az153", "az1062"])
@pytest.mark.parametrize("B", [1, 2, 31, 32])
def test_head_backward_production_mode_vs_float64(arch, hidden, A, Z, B):
    names, got, ref, guard_ok = head_backward_case(arch, hidden, A, Z, B)
    assert guard_ok, "dh scratch written past (B + 32) * 2H"
    errs = {k: rel_err(g, r) for k, g, r in zip(names, got, ref)}
    record(f"f64_head_backward_{arch}_a{A}_z{Z}_b{B}", dict(worst_max=max(e[0] for e in errs.values()),
                                                            worst_l2=max(e[1] for e in errs.values())))
    bad = [f"{k}: {e}" for k, e in errs.items() if not (e[0] <= BWD_MAX and e[1] <= BWD_L2)]
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_head_backward_comparison_rejects_unmasked_dx():
    """Negative controls of the head-gradient comparison: dx computed with relu_mask_x=0 (x has exact zeros), and one
    gradient element moved by twice the bound, must both fail."""
    names, got, ref, _ = head_backward_case("data-efficient", 256, 3, 51, 7, relu_mask_x=False)
    assert not within(got[0], ref[0], BWD_MAX, BWD_L2)
    assert all(within(g, r, BWD_MAX, BWD_L2) for g, r in zip(got[1:], ref[1:]))     # only dx depends on the flag
    g = got[1].clone()
    g.view(-1)[int(ref[1].abs().argmax())] += 2 * BWD_MAX * float(ref[1].abs().max())
    assert not within(g, ref[1], BWD_MAX, BWD_L2)


@pytest.mark.gpu
@pytest.mark.parametrize("B,Ch,HW", [(32, 64, 81), (32, 64, 49), (32, 64, 25), (7, 64, 1), (32, 1, 81), (512, 64, 49),
                                     (512, 32, 400)])
def test_bias_grad_vs_float64(B, Ch, HW):
    """rb_bias_grad (conv bias gradients of the manual conv backward) against a float64 sum, at the learner's shapes
    ([B,64,9,9], [B,64,7,7], [B,64,5,5]) and at HW = 1, C = 1 and B = 512."""
    from rainbow_b200 import _lib
    torch.manual_seed(B * 7 + Ch + HW)
    g = torch.randn(B, Ch, HW, device=DEV) * (torch.rand(B, Ch, HW, device=DEV) > 0.4)
    out = torch.full((Ch + GUARD,), float("nan"), device=DEV)
    _lib.check(_lib.load().rb_bias_grad(_lib.ptr(g), B, Ch, HW, _lib.ptr(out), _lib.stream()))
    torch.cuda.synchronize()
    ref = g.to(F64).sum((0, 2))
    scale = g.to(F64).abs().sum((0, 2)).clamp_min(1e-30)
    err = float(((out[:Ch].to(F64) - ref).abs() / scale).max())
    record(f"f64_bias_grad_b{B}_c{Ch}_hw{HW}", dict(err_over_abs_sum=err))
    assert bool(torch.isnan(out[Ch:]).all()), "wrote past C"
    assert err <= BIAS_SUM, err
