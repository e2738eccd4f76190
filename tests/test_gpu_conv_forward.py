"""rb_conv_forward (csrc/rb_head.cu k_conv_fwd): the conv body's forward, conv + bias + ReLU per layer, on the tensor cores
with the error-compensated TF32 product -- fp32-accurate against float64 torch, deterministic, every output written."""
import argparse

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
RB_ERR_RANGE = -34

# (IC, IH, OC, K, S) of every conv layer of model.py::_ARCH
LAYERS = {
    "canonical0": (4, 84, 32, 8, 4), "canonical1": (32, 20, 64, 4, 2), "canonical2": (64, 9, 64, 3, 1),
    "data_efficient0": (4, 84, 32, 5, 5), "data_efficient1": (32, 16, 64, 5, 5),
}


def make_args(**kw):
    d = dict(device=torch.device(DEV), history_length=4, atoms=51, architecture="canonical", hidden_size=512, noisy_std=0.1)
    d.update(kw)
    return argparse.Namespace(**d)


def launch(x, w, b, S, out):
    from rainbow_b200 import _lib
    return _lib.load().rb_conv_forward(x.data_ptr(), w.data_ptr(), b.data_ptr(), x.shape[0], x.shape[1], x.shape[2], x.shape[3],
                                       w.shape[0], w.shape[2], S, out.data_ptr(), torch.cuda.current_stream().cuda_stream)


def layer_inputs(name, rows, seed=0):
    IC, IH, OC, K, S = LAYERS[name]
    g = torch.Generator(device=DEV).manual_seed(seed + rows)
    if name.endswith("0"):
        x = torch.rand(rows, IC, IH, IH, device=DEV, generator=g)                        # states in [0, 1)
    else:
        x = torch.relu(torch.randn(rows, IC, IH, IH, device=DEV, generator=g))           # post-ReLU activations
    bound = 1.0 / (IC * K * K) ** 0.5                                                     # nn.Conv2d's default init range
    w = (torch.rand(OC, IC, K, K, device=DEV, generator=g) * 2 - 1) * bound
    b = (torch.rand(OC, device=DEV, generator=g) * 2 - 1) * bound
    return x, w, b, S


@pytest.mark.parametrize("rows", [1, 7, 32, 64])
@pytest.mark.parametrize("name", sorted(LAYERS))
def test_conv_forward_matches_float64(name, rows):
    from rainbow_b200 import _lib
    x, w, b, S = layer_inputs(name, rows)
    ref = F.relu(F.conv2d(x.double(), w.double(), b.double(), stride=S))
    out = torch.full(ref.shape, float("nan"), device=DEV)          # every element must be written
    _lib.check(launch(x, w, b, S, out))
    assert not torch.isnan(out).any()
    scale = float(ref.abs().max())
    np.testing.assert_allclose(out.cpu().numpy(), ref.cpu().numpy(), rtol=0, atol=2e-6 * scale)
    out2 = torch.full(ref.shape, float("nan"), device=DEV)
    _lib.check(launch(x, w, b, S, out2))
    assert torch.equal(out, out2), "second launch differs"


def test_conv_forward_saving_agrees_with_cudnn():
    """The learner's 64-row [s; s'] pass against the cuDNN formulation it replaced (conv + bias + ReLU per layer).
    cuDNN's fp32 kernels are themselves further from float64 than 2e-6 x max|ref| on the last layer (its activations are
    small after the default init), so each layer is checked against float64 at that tolerance and against cuDNN within the
    tolerance plus cuDNN's own measured deviation from float64."""
    from rainbow_b200.model import DQN
    torch.manual_seed(0)
    torch.backends.cudnn.allow_tf32 = False
    net = DQN(make_args(), 6).to(DEV)
    x = torch.rand(64, 4, 84, 84, device=DEV)
    with torch.no_grad():
        acts = net.conv_forward_saving(x)
        ref = [x]
        for m in net.conv_layers():
            ref.append(torch.cudnn_convolution_relu(ref[-1], m.weight, m.bias, m.stride, m.padding, m.dilation, m.groups))
        feats = net.features_nograd(x)
    assert len(acts) == len(ref)
    for a_in, a, r, m in zip(acts[:-1], acts[1:], ref[1:], net.conv_layers()):
        assert a.shape == r.shape
        with torch.no_grad():
            exact = F.relu(F.conv2d(a_in.double(), m.weight.double(), m.bias.double(), stride=m.stride))
        tol = 2e-6 * float(exact.abs().max())
        np.testing.assert_allclose(a.cpu().numpy(), exact.cpu().numpy(), rtol=0, atol=tol)
        cudnn_dev = float((r.double() - exact).abs().max())
        np.testing.assert_allclose(a.cpu().numpy(), r.cpu().numpy(), rtol=0, atol=tol + cudnn_dev)
    assert torch.equal(feats, acts[-1].view(64, -1))


def test_unsupported_shapes_are_refused_and_the_model_falls_back():
    from rainbow_b200 import _lib
    from rainbow_b200.model import DQN
    x = torch.rand(2, 4, 84, 84, device=DEV)
    for OC, K, S in ((32, 6, 3), (24, 8, 4)):                     # (kernel, stride) not instantiated; OC % 32 != 0
        w, b = torch.rand(OC, 4, K, K, device=DEV), torch.rand(OC, device=DEV)
        out = torch.full((2, OC, (84 - K) // S + 1, (84 - K) // S + 1), 7.0, device=DEV)
        assert launch(x, w, b, S, out) == RB_ERR_RANGE
        assert bool((out == 7.0).all()), "a refused shape must not launch anything"
    torch.manual_seed(0)
    net = DQN(make_args(), 6).to(DEV)
    net.convs[0] = torch.nn.Conv2d(4, 32, 8, stride=3).to(DEV)   # stride 3: not instantiated -> features()
    net.conv_output_size = 64 * 10 * 10                          # 84 -> 26 -> 12 -> 10
    with torch.no_grad():
        ref = net.features(x)
        assert torch.equal(net.features_nograd(x), ref)
        acts = net.conv_forward_saving(x)
    assert torch.equal(acts[-1].view(2, -1), ref)
