"""Probe (GPU): time the conv body's forward inside CUDA graphs.
First arm: the own kernel (rb_conv_forward) per layer at the learner's exact shapes -- online [s; s'] pass (64 rows, online
weights), target pass (32 rows, target weights), canonical and data-efficient nets -- next to the same layer through cuDNN's
fused conv + ReLU, with the achieved rate and the max |difference| against float64.  Then library formulations of the
canonical body at batch B (argv[1], default 32).  Not part of the product; informs what rainbow_b200.model uses."""
import argparse
import os
import sys
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

dev = "cuda"
torch.manual_seed(0)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
torch.backends.cudnn.allow_tf32 = False
FFMA_TFLOPS = 74.0   # 148 SMs x 128 FP32 lanes x 2 FLOP x 1.965 GHz: the plain-FFMA figure, not a tensor-core peak


def graph_us(fn, reps=50, iters=20):
    """Mean µs of one fn() call, replayed from a CUDA graph of `reps` calls (warm-up outside the graph)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (iters * reps)


def own_arm():
    from rainbow_b200 import _lib
    from rainbow_b200.model import DQN
    lib = _lib.load()
    print(f"{torch.cuda.get_device_name()}: own rb_conv_forward vs cuDNN cudnn_convolution_relu (fp32, allow_tf32=False), "
          f"CUDA graphs; rate as a fraction of the {FFMA_TFLOPS:.0f} TFLOP/s plain-FFMA figure")
    print(f"{'net':15s} {'pass':7s} {'rows':>4s} {'layer':24s} {'own us':>8s} {'cudnn us':>8s} {'GFLOP':>7s} "
          f"{'own TFLOP/s':>11s} {'of FFMA':>7s} {'max|d| own':>10s} {'max|d| cudnn':>12s}")
    for arch in ("canonical", "data-efficient"):
        args = argparse.Namespace(device=torch.device(dev), history_length=4, atoms=51, architecture=arch, hidden_size=512,
                                  noisy_std=0.1)
        torch.manual_seed(1)
        online = DQN(args, 6).to(dev)
        torch.manual_seed(2)
        target = DQN(args, 6).to(dev)
        for pname, net, rows in (("online", online, 64), ("target", target, 32)):
            x = torch.rand(rows, 4, 84, 84, device=dev)
            tot_own = tot_cudnn = 0.0
            for m in net.conv_layers():
                k, s = m.kernel_size[0], m.stride[0]
                oh = (x.shape[2] - k) // s + 1
                y = torch.empty(rows, m.out_channels, oh, oh, device=dev)
                args_ = (x.data_ptr(), m.weight.data_ptr(), m.bias.data_ptr(), rows, x.shape[1], x.shape[2], x.shape[3],
                         m.out_channels, k, s, y.data_ptr())
                own = graph_us(lambda: _lib.check(lib.rb_conv_forward(*args_, _lib.stream())))
                ref_fn = lambda: torch.cudnn_convolution_relu(x, m.weight, m.bias, m.stride, m.padding, m.dilation, m.groups)
                cud = graph_us(ref_fn)
                with torch.no_grad():
                    ref = F.relu(F.conv2d(x.double(), m.weight.double(), m.bias.double(), stride=s))
                    d_own = float((y.double() - ref).abs().max())
                    d_cud = float((ref_fn().double() - ref).abs().max())
                flop = 2.0 * rows * m.out_channels * oh * oh * x.shape[1] * k * k
                tflops = flop / (own * 1e-6) / 1e12
                layer = f"{x.shape[1]}->{m.out_channels} k{k} s{s} {x.shape[2]}->{oh}"
                print(f"{arch:15s} {pname:7s} {rows:4d} {layer:24s} {own:8.2f} {cud:8.2f} {flop / 1e9:7.3f} {tflops:11.2f} "
                      f"{tflops / FFMA_TFLOPS:7.3f} {d_own:10.2e} {d_cud:12.2e}")
                tot_own, tot_cudnn = tot_own + own, tot_cudnn + cud
                x = y
            print(f"{arch:15s} {pname:7s} {rows:4d} {'whole body (serial sum)':24s} {tot_own:8.2f} {tot_cudnn:8.2f}")


own_arm()
specs = [(4, 32, 8, 4), (32, 64, 4, 2), (64, 64, 3, 1)]
ws = [torch.randn(co, ci, k, k, device=dev) * 0.05 for ci, co, k, s in specs]
bs = [torch.randn(co, device=dev) * 0.05 for ci, co, k, s in specs]
x0 = torch.rand(B, 4, 84, 84, device=dev)


def timeit(fn, name, reps=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    try:
        with torch.cuda.graph(g):
            for _ in range(reps):
                out = fn()
    except Exception as e:
        print(f"{name:45s} capture failed: {str(e)[:80]}")
        torch.cuda.synchronize()
        return None
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (5 * reps)
    print(f"{name:45s} {us:8.1f} us per 3-conv pass")
    return out


def fwd_plain(x=x0):
    for (ci, co, k, s), w, b in zip(specs, ws, bs):
        x = F.relu(F.conv2d(x, w, b, stride=s))
    return x


def fwd_fused(x=x0):
    for (ci, co, k, s), w, b in zip(specs, ws, bs):
        x = torch.cudnn_convolution_relu(x, w, b, (s, s), (0, 0), (1, 1), 1)
    return x


def fwd_unfold(x=x0):
    for (ci, co, k, s), w, b in zip(specs, ws, bs):
        n, c, h, wd = x.shape
        ho, wo = (h - k) // s + 1, (wd - k) // s + 1
        cols = F.unfold(x, k, stride=s)                       # [n, c*k*k, ho*wo]
        y = torch.baddbmm(b.view(1, -1, 1), w.view(1, co, -1).expand(n, -1, -1), cols)
        x = F.relu(y).view(n, co, ho, wo)
    return x


for tf32 in (False, True):
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    for bench in (False, True):
        torch.backends.cudnn.benchmark = bench
        tag = f"tf32={int(tf32)} bench={int(bench)}"
        ref = timeit(fwd_plain, f"conv2d+relu NCHW           {tag}")
        o = timeit(fwd_fused, f"cudnn_convolution_relu NCHW {tag}")
        if o is not None and ref is not None:
            print("     max abs diff vs plain:", float((o - ref).abs().max()))
        xcl = x0.contiguous(memory_format=torch.channels_last)
        wcl = [w.contiguous(memory_format=torch.channels_last) for w in ws]

        def fwd_cl():
            x = xcl
            for (ci, co, k, s), w, b in zip(specs, wcl, bs):
                x = F.relu(F.conv2d(x, w, b, stride=s))
            return x
        timeit(fwd_cl, f"conv2d+relu channels_last   {tag}")
    timeit(fwd_unfold, f"unfold+baddbmm              tf32={int(tf32)}")

# backward (plain autograd) for reference
for tf32 in (False, True):
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cudnn.benchmark = True
    wr = [w.clone().requires_grad_(True) for w in ws]
    br = [b.clone().requires_grad_(True) for b in bs]
    gout = torch.randn(B, 64, 7, 7, device=dev)
    for p in wr + br:
        p.grad = torch.zeros_like(p)

    def fb():
        x = x0
        for (ci, co, k, s), w, b in zip(specs, wr, br):
            x = F.relu(F.conv2d(x, w, b, stride=s))
        x.backward(gout)
        return x
    timeit(fb, f"fwd+bwd autograd            tf32={int(tf32)}", reps=5)
