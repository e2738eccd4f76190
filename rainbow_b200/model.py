"""Dueling distributional network with factorised-noise linear layers.

API and state_dict layout follow the reference's model.py (NoisyLinear model.py:10-46, DQN
model.py:49-85) so checkpoints interchange: convs.{0,2,4}.{weight,bias} and
fc_{h_v,h_a,z_v,z_a}.{weight_mu,weight_sigma,bias_mu,bias_sigma,weight_epsilon,bias_epsilon}.

The conv body's parameters, layout, autograd path (features()) and backward stay torch / cuDNN.  What is ours:
  * the conv body's forward on the learner, act and evaluation paths (conv_forward_saving / features_nograd): one
    rb_conv_forward launch per layer (csrc/rb_head.cu k_conv_fwd, conv + bias + ReLU as an implicit GEMM on the tensor cores,
    error-compensated TF32 = fp32-accurate whatever allow_tf32 says).  It replaced cuDNN's fused conv + ReLU, whose fp32
    kernels were the largest block on the update's critical path and take as long at 64 rows as at 32;
  * noise lives as FACTOR VECTORS f(eps_in), f(eps_out) per layer (model.py:36-38); reset_noise() is one tiny
    rb_noise_factors launch (device Philox + Box-Muller) instead of the reference's ~52 ATen ops and 13.6 MB of
    weight_epsilon writes per net.  The weight_epsilon / bias_epsilon buffers of the state_dict are materialised
    lazily (rb_noisy_outer) only when somebody looks at them (state_dict(), the library-GEMM fallback path);
  * the noisy dueling head (model.py:69-75 after the convs) runs through the fused head kernels
    (rb_head_forward / rb_head_logits, csrc/rb_head.cu), which compose W = mu + sigma*eps on the fly;
  * logits(): the pre-softmax dueling combination (model.py:75), which the fused C51 kernel consumes.

Autograd: when gradients are being recorded (an external caller training through forward()), logits() uses the
plain torch path (composed weights + F.linear) so autograd works as in the reference; the learner in
rainbow_b200.agent drives the fused forward AND backward kernels itself.
"""
import ctypes as C
import math

import torch
from torch import nn
from torch.nn import functional as F

from . import _lib

RB_ERR_RANGE = -34   # include/rainbow_b200.h: shape outside what a kernel instantiates

_ARCH = {
    # name: (conv specs (out_channels, kernel, stride), flattened conv output size)   model.py:55-63
    "canonical": (((32, 8, 4), (64, 4, 2), (64, 3, 1)), 3136),
    "data-efficient": (((32, 5, 5), (64, 5, 5)), 576),
}


class NoisyLinear(nn.Module):
    """y = x (mu_w + sigma_w * eps_w)^T + (mu_b + sigma_b * eps_b) in training mode, mu only in eval mode."""

    def __init__(self, in_features, out_features, std_init=0.5):
        super().__init__()
        self.in_features, self.out_features, self.std_init = in_features, out_features, std_init
        self.weight_mu = nn.Parameter(torch.empty(out_features, in_features))
        self.weight_sigma = nn.Parameter(torch.empty(out_features, in_features))
        self.register_buffer("weight_epsilon", torch.zeros(out_features, in_features))
        self.bias_mu = nn.Parameter(torch.empty(out_features))
        self.bias_sigma = nn.Parameter(torch.empty(out_features))
        self.register_buffer("bias_epsilon", torch.zeros(out_features))
        self.reset_parameters()
        self._construction_noise()

    def _construction_noise(self):
        """Construction-time only (host, before the module is moved to the GPU): the reference draws one
        noise sample in __init__ (model.py:23).  Doing the same keeps the torch RNG stream -- and therefore
        every later layer's initial weights -- identical to the reference for the same seed.  The learner
        never uses this path: DQN.reset_noise() is a CUDA kernel."""
        with torch.no_grad():
            x_in, x_out = torch.randn(self.in_features), torch.randn(self.out_features)
            self._f_in, self._f_out = x_in.sign() * x_in.abs().sqrt(), x_out.sign() * x_out.abs().sqrt()
            self.weight_epsilon.copy_(torch.outer(self._f_out, self._f_in))
            self.bias_epsilon.copy_(self._f_out)

    def reset_parameters(self):  # model.py:25-30
        bound = 1.0 / math.sqrt(self.in_features)
        with torch.no_grad():
            self.weight_mu.uniform_(-bound, bound)
            self.bias_mu.uniform_(-bound, bound)
            self.weight_sigma.fill_(self.std_init / math.sqrt(self.in_features))
            self.bias_sigma.fill_(self.std_init / math.sqrt(self.out_features))

    def forward(self, x):
        if self.training:  # model.py:43-44
            w = torch.addcmul(self.weight_mu, self.weight_sigma, self.weight_epsilon)
            b = torch.addcmul(self.bias_mu, self.bias_sigma, self.bias_epsilon)
            return F.linear(x, w, b)
        return F.linear(x, self.weight_mu, self.bias_mu)


def _layer_arrays(layers):
    n = len(layers)
    return ((C.c_void_p * n)(*[_lib.ptr(m.weight_epsilon) for m in layers]),
            (C.c_void_p * n)(*[_lib.ptr(m.bias_epsilon) for m in layers]),
            (C.c_int * n)(*[m.in_features for m in layers]), (C.c_int * n)(*[m.out_features for m in layers]), n)


def resample_noise(layers, seed, rng_counter, x_in=None, x_out=None):
    """One rb_noisy_resample launch (K6) over `layers`: draws AND materialises weight_epsilon / bias_epsilon.
    x_in / x_out: optional injected raw normals (parity mode), concatenated over layers."""
    w, b, fin, fout, n = _layer_arrays(layers)
    _lib.check(_lib.load().rb_noisy_resample(w, b, fin, fout, n, _lib.ptr(x_in), _lib.ptr(x_out), seed,
                                             _lib.ptr(rng_counter), _lib.stream()))


class FusedHead:
    """Launcher of the fused noisy dueling head kernels for one DQN (csrc/rb_head.cu)."""

    MAX_ROWS = 4096

    def __init__(self, net):
        self.net = net
        self.lib = _lib.load()
        s1, s2 = C.c_int(), C.c_int()
        _lib.check(self.lib.rb_head_splits(net.conv_output_size, net.hidden_size, C.byref(s1), C.byref(s2)))
        self.s1, self.s2 = s1.value, s2.value
        self.ncols = net.atoms * (1 + net.action_space)
        self._scratch = {}
        self._tickets = None

    @staticmethod
    def supported(net, rows, backward=False):
        """Whether the kernels take this net's head at `rows` rows (and, with `backward`, its backward at a batch of `rows`):
        the library's own limits (rb_head_supported), so a shape they refuse is routed elsewhere instead of raising."""
        if not next(net.parameters()).is_cuda:
            return False
        rc = _lib.load().rb_head_supported(net.conv_output_size, net.hidden_size, net.atoms, net.action_space, rows,
                                           1 if backward else 0)
        if rc not in (0, RB_ERR_RANGE):
            _lib.check(rc)
        return rc == 0

    def params(self, noisy=None):
        net = self.net
        noisy = net.training if noisy is None else noisy
        p = _lib.HeadParams()
        (hv, ha), (zv, za) = (net.fc_h_v, net.fc_h_a), (net.fc_z_v, net.fc_z_a)
        for s, (l1, l2) in enumerate(((hv, zv), (ha, za))):
            p.w1_mu[s], p.w1_sigma[s] = _lib.ptr(l1.weight_mu), _lib.ptr(l1.weight_sigma)
            p.b1_mu[s], p.b1_sigma[s] = _lib.ptr(l1.bias_mu), _lib.ptr(l1.bias_sigma)
            p.w2_mu[s], p.w2_sigma[s] = _lib.ptr(l2.weight_mu), _lib.ptr(l2.weight_sigma)
            p.b2_mu[s], p.b2_sigma[s] = _lib.ptr(l2.bias_mu), _lib.ptr(l2.bias_sigma)
        if noisy:
            f = net.noise_factors()  # {layer name: (f_in, f_out)}
            for s, (n1, n2) in enumerate((("fc_h_v", "fc_z_v"), ("fc_h_a", "fc_z_a"))):
                p.eps_in1[s], p.eps_out1[s] = _lib.ptr(f[n1][0]), _lib.ptr(f[n1][1])
                p.eps_in2[s], p.eps_out2[s] = _lib.ptr(f[n2][0]), _lib.ptr(f[n2][1])
        p.conv_features, p.hidden, p.atoms, p.actions = net.conv_output_size, net.hidden_size, net.atoms, net.action_space
        return p

    def grads(self):
        """rb_head_grads pointing at the .grad storage of the 16 head parameters (must exist)."""
        net = self.net
        g = _lib.HeadGrads()
        for s, (l1, l2) in enumerate(((net.fc_h_v, net.fc_z_v), (net.fc_h_a, net.fc_z_a))):
            g.w1_mu[s], g.w1_sigma[s] = _lib.ptr(l1.weight_mu.grad), _lib.ptr(l1.weight_sigma.grad)
            g.b1_mu[s], g.b1_sigma[s] = _lib.ptr(l1.bias_mu.grad), _lib.ptr(l1.bias_sigma.grad)
            g.w2_mu[s], g.w2_sigma[s] = _lib.ptr(l2.weight_mu.grad), _lib.ptr(l2.weight_sigma.grad)
            g.b2_mu[s], g.b2_sigma[s] = _lib.ptr(l2.bias_mu.grad), _lib.ptr(l2.bias_sigma.grad)
        return g

    def _buffers(self, M, dev):
        if M not in self._scratch:
            H = self.net.hidden_size
            f32 = torch.float32
            self._scratch[M] = dict(part1=torch.empty((self.s1, M, 2 * H), dtype=f32, device=dev),
                                    part2=torch.empty((self.s2, M, self.ncols), dtype=f32, device=dev),
                                    h=torch.empty((M, 2 * H), dtype=f32, device=dev),
                                    z=torch.empty((M, self.ncols), dtype=f32, device=dev))
        if self._tickets is None:
            self._tickets = torch.zeros(self.lib.rb_head_ticket_count(), dtype=torch.int32, device=dev)
        return self._scratch[M]

    def forward(self, x_lo, x_hi=None, noisy=None):
        """x_lo [m_lo, K1] (+ x_hi [m_hi, K1]) -> (z [M, Z(1+A)], h [M, 2H], params); buffers are reused per M."""
        m_lo = x_lo.shape[0]
        m_hi = 0 if x_hi is None else x_hi.shape[0]
        buf = self._buffers(m_lo + m_hi, x_lo.device)
        p = self.params(noisy)
        _lib.check(self.lib.rb_head_forward(C.byref(p), _lib.ptr(x_lo), m_lo, _lib.ptr(x_hi), m_hi, _lib.ptr(buf["part1"]),
                                            _lib.ptr(buf["part2"]), _lib.ptr(self._tickets), _lib.ptr(buf["h"]),
                                            _lib.ptr(buf["z"]), _lib.stream()))
        return buf["z"], buf["h"], p

    def logits(self, z):
        M = z.shape[0]
        q = torch.empty((M, self.net.action_space, self.net.atoms), dtype=torch.float32, device=z.device)
        _lib.check(self.lib.rb_head_logits(_lib.ptr(z), M, self.net.action_space, self.net.atoms, _lib.ptr(q), _lib.stream()))
        return q

    BWD_WGRAD2, BWD_DH, BWD_LAYER1, BWD_ALL = 1, 2, 4, 7

    def backward(self, p, x, h, dz, dh_scratch, dx, relu_mask_x=False, parts=7):
        g = self.grads()
        _lib.check(self.lib.rb_head_backward(C.byref(p), C.byref(g), _lib.ptr(x), _lib.ptr(h), _lib.ptr(dz), x.shape[0],
                                             _lib.ptr(dh_scratch), _lib.ptr(dx), 1 if relu_mask_x else 0, parts,
                                             _lib.stream()))
        return dx


class DQN(nn.Module):
    def __init__(self, args, action_space):
        super().__init__()
        self.atoms = args.atoms
        self.action_space = action_space
        self.hidden_size = args.hidden_size
        if args.architecture not in _ARCH:
            raise ValueError(f"unknown architecture '{args.architecture}'")
        specs, self.conv_output_size = _ARCH[args.architecture]
        mods, c_in = [], args.history_length
        for c_out, k, s in specs:
            mods += [nn.Conv2d(c_in, c_out, k, stride=s, padding=0), nn.ReLU()]
            c_in = c_out
        self.convs = nn.Sequential(*mods)
        self.fc_h_v = NoisyLinear(self.conv_output_size, args.hidden_size, std_init=args.noisy_std)
        self.fc_h_a = NoisyLinear(self.conv_output_size, args.hidden_size, std_init=args.noisy_std)
        self.fc_z_v = NoisyLinear(args.hidden_size, self.atoms, std_init=args.noisy_std)
        self.fc_z_a = NoisyLinear(args.hidden_size, action_space * self.atoms, std_init=args.noisy_std)
        self.noise_seed = int(torch.initial_seed()) & (2 ** 63 - 1)
        self.register_buffer("_noise_counter", torch.zeros(1, dtype=torch.int64), persistent=False)
        # factor vectors of all layers back to back, in reset order: f(eps_in) | f(eps_out)
        layers = self.noisy_layers()
        self.register_buffer("_f_in", torch.cat([m._f_in for m in layers]), persistent=False)
        self.register_buffer("_f_out", torch.cat([m._f_out for m in layers]), persistent=False)
        self._noise_queue = []   # parity facility: injected raw normals consumed by the next reset_noise() calls
        # lazy_noise (set by the learner for its online net): an argument-less reset_noise() only marks the draw as pending;
        # it is launched by flush_noise() right before its first use (act / evaluate / state_dict), or by the learner on a
        # side branch of the update instead of serially in front of it.  Same draws, same order, nothing skipped.
        self.lazy_noise = False
        self._noise_pending = False
        self._eps_stale = False  # weight_epsilon / bias_epsilon buffers currently equal the outer product of the factors
        self._head = None
        self.use_fused_head = True
        self.use_own_wgrad = True     # first conv layer's weight gradient through rb_conv_wgrad (else cuDNN)

    # ---- noise ---------------------------------------------------------------------------------------
    def noisy_layers(self):
        """Layers in the reference's reset order (named_children containing 'fc', model.py:83-85)."""
        return [m for name, m in self.named_children() if "fc" in name]

    def noise_factors(self):
        self.flush_noise()
        out, oi, oo = {}, 0, 0
        for name, m in self.named_children():
            if "fc" in name:
                out[name] = (self._f_in[oi:oi + m.in_features], self._f_out[oo:oo + m.out_features])
                oi, oo = oi + m.in_features, oo + m.out_features
        return out

    def reset_noise(self, x_in=None, x_out=None):
        """model.py:82-85: new factor vectors for every NoisyLinear, one launch.  x_in / x_out: optional injected
        raw normals (parity).  Needs the network on a CUDA device."""
        if not self._f_in.is_cuda:
            raise _lib.RainbowB200Error("DQN.reset_noise needs the network on a CUDA device (no CPU fallback)")
        if x_in is None and self._noise_queue:
            x_in, x_out = self._noise_queue.pop(0)
        if x_in is None and self.lazy_noise and not torch.cuda.is_current_stream_capturing():
            self._noise_pending = True
            return
        self._noise_pending = False
        _lib.check(_lib.load().rb_noise_factors(_lib.ptr(self._f_in), self._f_in.numel(), _lib.ptr(self._f_out),
                                                self._f_out.numel(), _lib.ptr(x_in), _lib.ptr(x_out), self.noise_seed,
                                                _lib.ptr(self._noise_counter), _lib.stream()))
        self._eps_stale = True

    def flush_noise(self):
        """Launch a reset_noise() that was deferred (lazy_noise)."""
        if self._noise_pending:
            self._noise_pending = False
            lazy, self.lazy_noise = self.lazy_noise, False
            try:
                self.reset_noise()
            finally:
                self.lazy_noise = lazy

    def queue_noise(self, x_in, x_out):
        """Parity testing: the next argument-less reset_noise() uses these raw standard normals (device float32, all
        layers back to back: eps_in draws / eps_out draws, model.py:37-38) instead of the device Philox stream, so the
        public reset_noise(); learn(mem) sequence can be fed the reference's recorded torch.randn draws."""
        self._noise_queue.append((x_in.contiguous(), x_out.contiguous()))

    def materialise_noise(self):
        """Bring weight_epsilon / bias_epsilon (model.py:39-40) up to date with the factor vectors."""
        self.flush_noise()
        if self._eps_stale:
            w, b, fin, fout, n = _layer_arrays(self.noisy_layers())
            _lib.check(_lib.load().rb_noisy_outer(w, b, fin, fout, n, _lib.ptr(self._f_in), _lib.ptr(self._f_out),
                                                  _lib.stream()))
            self._eps_stale = False

    def _factors_from_buffers(self):
        """After load_state_dict: recover the rank-one factors from the loaded epsilon buffers
        (eps_out = bias_epsilon; eps_in = the weight_epsilon row of the largest |eps_out| divided by it)."""
        with torch.no_grad():
            fi, fo = [], []
            for m in self.noisy_layers():
                b = m.bias_epsilon
                o = int(b.abs().argmax())
                fo.append(b.clone())
                fi.append(m.weight_epsilon[o] / b[o] if float(b[o]) != 0.0 else torch.zeros_like(m.weight_epsilon[0]))
            self._f_in.copy_(torch.cat(fi))
            self._f_out.copy_(torch.cat(fo))
        self._eps_stale = False

    def state_dict(self, *args, **kwargs):
        if self._f_in.is_cuda:
            self.flush_noise()
        if self._eps_stale and self._f_in.is_cuda:
            self.materialise_noise()
        return super().state_dict(*args, **kwargs)

    def load_state_dict(self, state_dict, *args, **kwargs):
        out = super().load_state_dict(state_dict, *args, **kwargs)
        self._noise_pending = False          # the loaded epsilon buffers supersede a deferred draw
        self._factors_from_buffers()
        return out

    # ---- forward -------------------------------------------------------------------------------------
    def head(self):
        if self._head is None:
            self._head = FusedHead(self)
        return self._head

    def fused_ok(self, rows, backward=False):
        return self.use_fused_head and rows <= FusedHead.MAX_ROWS and FusedHead.supported(self, rows, backward)

    def features(self, x):
        return self.convs(x).view(-1, self.conv_output_size)

    # ---- conv body with a hand-scheduled backward (library kernels, our schedule) -------------------------
    def conv_layers(self):
        return [m for m in self.convs if isinstance(m, nn.Conv2d)]

    def manual_conv_ok(self, x):
        return x.is_cuda and torch.backends.cudnn.enabled

    def _own_conv_body(self, x):
        """[a0 = x, a1, ..., aL] through rb_conv_forward (csrc/rb_head.cu k_conv_fwd: conv + bias + ReLU, one launch per layer),
        or None when the input is not a contiguous fp32 CUDA tensor or the kernel does not instantiate a layer's shape."""
        if not (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 4):
            return None
        lib = _lib.load()
        acts = [x]
        for m in self.conv_layers():
            a = acts[-1]
            if (m.padding != (0, 0) or m.dilation != (1, 1) or m.groups != 1 or m.kernel_size[0] != m.kernel_size[1] or
                    m.stride[0] != m.stride[1] or not (m.weight.is_contiguous() and m.bias.is_contiguous())):
                return None
            k, s = m.kernel_size[0], m.stride[0]
            y = torch.empty((a.shape[0], m.out_channels, (a.shape[2] - k) // s + 1, (a.shape[3] - k) // s + 1),
                            dtype=torch.float32, device=a.device)
            rc = lib.rb_conv_forward(_lib.ptr(a), _lib.ptr(m.weight), _lib.ptr(m.bias), a.shape[0], a.shape[1], a.shape[2], a.shape[3],
                                     m.out_channels, k, s, _lib.ptr(y), _lib.stream())
            if rc == RB_ERR_RANGE:
                return None
            _lib.check(rc)
            acts.append(y)
        return acts

    def conv_forward_saving(self, x):
        """Conv body keeping every layer's input for the manual backward: [a0 = x, a1, ..., aL] (aL = ReLU(conv_L(...)), the
        conv features).  Own tensor-core kernel per layer; shapes it does not cover go through the modules of features()."""
        acts = self._own_conv_body(x)
        if acts is None:
            acts = [x]
            for i in range(0, len(self.convs), 2):
                acts.append(self.convs[i + 1](self.convs[i](acts[-1])))
        return acts

    def _own_wgrad_ok(self, m, a_in):
        k, s = m.kernel_size, m.stride
        return (self.use_own_wgrad and k[0] == k[1] and s[0] == s[1] and k[0] in (3, 4, 5, 8) and tuple(m.padding) == (0, 0) and
                tuple(m.dilation) == (1, 1) and m.groups == 1 and a_in.is_contiguous() and m.weight.grad.is_contiguous() and
                m.in_channels * k[0] * ((m.out_channels + 3) // 4) <= 256 and
                _lib.load().rb_conv_wgrad_scratch_elems(a_in.shape[0], m.in_channels, a_in.shape[2], m.out_channels, k[0], s[0]) > 0)

    def _wgrad_scratch(self, m, a_in):
        n = _lib.load().rb_conv_wgrad_scratch_elems(a_in.shape[0], m.in_channels, a_in.shape[2], m.out_channels, m.kernel_size[0], m.stride[0])
        buf = getattr(self, "_wgrad_buf", None)
        if buf is None or buf.numel() < n or buf.device != a_in.device:
            buf = torch.empty(n, dtype=torch.float32, device=a_in.device)
            self._wgrad_buf = buf
        return buf

    def conv_backward_into_grads(self, acts, g_last, side_stream, first_layer_stream=None):
        """Backward of the conv body given g_last = d loss / d (pre-activation of the last conv layer).
        The data-gradient chain (dgrad -> ReLU mask -> dgrad ...) runs on the current stream; the weight and bias
        gradients, which nothing downstream waits for except the optimiser, run on `side_stream` and are written
        straight into the parameters' .grad storage.  Returns the event the optimiser has to wait for."""
        lib = _lib.load()
        main = torch.cuda.current_stream(g_last.device)
        layers = self.conv_layers()
        g = g_last
        extra_done = None
        for li in range(len(layers) - 1, -1, -1):
            m, a_in = layers[li], acts[li]
            ready = torch.cuda.Event()
            ready.record(main)
            own = li == 0 and self._own_wgrad_ok(m, a_in)
            # the first layer's gradient is the last thing the chain produces: it gets its own stream so that it does not
            # queue behind the (independent) weight gradients of the layers above on `side_stream`
            st = first_layer_stream if (own and first_layer_stream is not None) else side_stream
            with torch.cuda.stream(st):
                st.wait_event(ready)
                g.record_stream(st)
                if own:
                    # first layer: no data gradient follows, so this launch sits alone on the critical path -> own kernel
                    # (csrc/rb_head.cu k_conv_wgrad_first; weight AND bias gradient from one pass over g)
                    _lib.check(lib.rb_conv_wgrad(_lib.ptr(g), _lib.ptr(a_in), a_in.shape[0], a_in.shape[1], a_in.shape[2], a_in.shape[3],
                                                 m.out_channels, m.kernel_size[0], m.stride[0], _lib.ptr(self._wgrad_scratch(m, a_in)),
                                                 _lib.ptr(m.weight.grad), _lib.ptr(m.bias.grad), st.cuda_stream))
                else:   # bias first (it only needs g), then the library's weight gradient
                    _lib.check(lib.rb_bias_grad(_lib.ptr(g), g.shape[0], g.shape[1], g.shape[2] * g.shape[3],
                                                _lib.ptr(m.bias.grad), st.cuda_stream))
                    _, gw, _ = torch.ops.aten.convolution_backward(g, a_in, m.weight, None, m.stride, m.padding, m.dilation, False,
                                                                   [0, 0], m.groups, [False, True, False])
                    m.weight.grad.copy_(gw)
                if st is not side_stream:
                    extra_done = torch.cuda.Event()
                    extra_done.record(st)
            if li > 0:
                gin, _, _ = torch.ops.aten.convolution_backward(g, a_in, m.weight, None, m.stride, m.padding, m.dilation, False,
                                                                [0, 0], m.groups, [True, False, False])
                g = torch.ops.aten.threshold_backward(gin, a_in, 0.0)      # ReLU of the layer below (a_in = its output)
        if extra_done is not None:
            side_stream.wait_event(extra_done)
        done = torch.cuda.Event()
        done.record(side_stream)
        return done

    def features_nograd(self, x):
        """Inference-only conv body: the own conv + bias + ReLU kernel per layer (fp32-accurate, see _own_conv_body);
        features() for inputs or shapes it does not cover."""
        acts = self._own_conv_body(x)
        if acts is None:
            return self.features(x)
        return acts[-1].view(-1, self.conv_output_size)

    def logits(self, x):
        """Pre-softmax q [B, A, Z] (model.py:69-75)."""
        feats = self.features(x)
        recording = torch.is_grad_enabled() and (feats.requires_grad or self.fc_h_v.weight_mu.requires_grad)
        if not recording and self.fused_ok(feats.shape[0]):
            z, _, _ = self.head().forward(feats.contiguous())
            return self.head().logits(z)
        if self._eps_stale:
            self.materialise_noise()
        v = self.fc_z_v(F.relu(self.fc_h_v(feats))).view(-1, 1, self.atoms)
        a = self.fc_z_a(F.relu(self.fc_h_a(feats))).view(-1, self.action_space, self.atoms)
        return v + a - a.mean(1, keepdim=True)

    def forward(self, x, log=False):
        q = self.logits(x)
        return F.log_softmax(q, dim=2) if log else F.softmax(q, dim=2)
