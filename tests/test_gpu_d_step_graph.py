"""-m gpu: the graphed discriminator step (IRFDDiscriminatorStep(use_cuda_graph=True)) and the spectral-norm kernels it
runs on: kernels vs a float64 power iteration, native vs torch-hook sequences, replay vs its eager twin, graph vs the
eager step, interleaving with the graphed G step, recapture triggers and data parallelism."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

pytestmark = pytest.mark.gpu


def _rel(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float((a - b).norm() / b.norm())


def _disc(dev, seed=0):
    from speak_hack_b200.discriminator import StyleDiscriminator

    torch.manual_seed(seed)
    return StyleDiscriminator().to(dev).train()


def test_spectral_norm_kernels_vs_float64(cuda_device):
    """Every D layer shape, same start u / v: u, v, sigma and W_sn (train and eval mode) and dW_orig against float64."""
    from speak_hack_b200 import ops

    D = _disc(cuda_device)
    mods = D._sn_modules()
    ws = [m.weight_orig.detach() for m in mods]
    u0 = [m.weight_u.clone() for m in mods]
    v0 = [m.weight_v.clone() for m in mods]
    g = torch.Generator(device=cuda_device).manual_seed(3)
    worst = {}
    for train in (True, False):
        us, vs = [u.clone() for u in u0], [v.clone() for v in v0]
        outs, u_s, v_s, sigma = ops.spectral_norm_fwd(ws, us, vs, train)
        gs = [torch.randn(w.shape, generator=g, device=cuda_device) for w in ws]
        dws = ops.spectral_norm_bwd(gs, outs, u_s, v_s, sigma)
        torch.cuda.synchronize()
        ro = co = 0
        for i, w in enumerate(ws):
            W = w.double().reshape(w.shape[0], -1)
            u, v = u0[i].double(), v0[i].double()
            if train:
                v = torch.nn.functional.normalize(W.t() @ u, dim=0, eps=1e-12)
                u = torch.nn.functional.normalize(W @ v, dim=0, eps=1e-12)
            Wr = W.clone().requires_grad_(True)
            sig = u @ (Wr @ v)
            (Wr / sig).backward(gs[i].double().reshape(W.shape))
            r, c = W.shape
            errs = {"u": _rel(u_s[ro: ro + r], u), "v": _rel(v_s[co: co + c], v),
                    "sigma": _rel(sigma[i: i + 1], sig.detach().reshape(1)),
                    "W_sn": _rel(outs[i], W / sig.detach()), "dW": _rel(dws[i], Wr.grad)}
            if train:
                errs["u_buf"], errs["v_buf"] = _rel(us[i], u), _rel(vs[i], v)
            else:
                assert torch.equal(us[i], u0[i]) and torch.equal(vs[i], v0[i])   # eval: buffers untouched
            for k, e in errs.items():
                key = (train, k)
                if e > worst.get(key, (0.0, None))[0]:
                    worst[key] = (e, tuple(w.shape))
            ro, co = ro + r, co + c
    print("[sn] worst relative errors vs float64: " +
          ", ".join(f"{'train' if t else 'eval'} {k} {e:.2e} {s}" for (t, k), (e, s) in sorted(worst.items())))
    assert all(e < 1e-5 for e, _ in worst.values()), worst


def test_spectral_norm_kernels_are_deterministic(cuda_device):
    from speak_hack_b200 import ops

    D = _disc(cuda_device)
    mods = D._sn_modules()
    ws = [m.weight_orig.detach() for m in mods]
    res = []
    for _ in range(2):
        us, vs = [m.weight_u.clone() for m in mods], [m.weight_v.clone() for m in mods]
        outs, u_s, v_s, sigma = ops.spectral_norm_fwd(ws, us, vs, True)
        dws = ops.spectral_norm_bwd([o * 0.5 + 1.0 for o in outs], outs, u_s, v_s, sigma)
        res.append([t.clone() for t in outs + dws + [u_s, v_s, sigma]])
    assert all(torch.equal(a, b) for a, b in zip(*res))


def test_six_native_calls_follow_the_torch_hook(cuda_device):
    """Six power iterations on the kernels leave u and v where six calls of torch's spectral-norm hook leave them."""
    from speak_hack_b200 import ops
    from speak_hack_b200.discriminator import _normalized_weight

    D = _disc(cuda_device)
    mods = D._sn_modules()
    ws = [m.weight_orig.detach() for m in mods]
    us, vs = [m.weight_u.clone() for m in mods], [m.weight_v.clone() for m in mods]
    for _ in range(6):
        ops.spectral_norm_fwd(ws, us, vs, True)
    with torch.no_grad():
        for _ in range(6):
            for m in mods:
                _normalized_weight(m)
    torch.cuda.synchronize()
    eu = max(_rel(a, m.weight_u) for a, m in zip(us, mods))
    ev = max(_rel(a, m.weight_v) for a, m in zip(vs, mods))
    print(f"[sn] after 6 calls, native vs torch hook: u {eu:.2e}, v {ev:.2e}")
    assert eu < 1e-5 and ev < 1e-5


# ---------------------------------------------------------------------------------------------------- the graphed step
def _net(dev, seed=None, state=None):
    import irfd_oracle as O
    import speak_hack_b200 as P

    torch.manual_seed(O.WEIGHT_SEED if seed is None else seed)
    net = P.IRFD().to(dev).train()
    if state is not None:
        net.load_state_dict(state)
    return net


def _converged(dev, xs):
    """A model whose spectral-norm power iterations have converged (fresh u / v give weights ~1e3 too large), and its
    state_dict, so several identical copies can be made."""
    net = _net(dev)
    with torch.no_grad():
        for _ in range(6):
            net.D(xs)
    return net, {k: v.clone() for k, v in net.state_dict().items()}


def _pair(dev, b=2):
    import irfd_oracle as O

    x_s, x_t = O.synthetic_pair(b)
    return x_s.to(dev), x_t.to(dev)


def _d_state(net, ds):
    enc = [bf for e in (net.Ei, net.Ee, net.Ep) for bf in e.buffers()]
    return [ds.flat, ds.m, ds.v] + list(net.D.buffers()) + enc


def test_replay_equals_its_eager_twin(cuda_device):
    """Same state, same CPU and CUDA seeds, 3 steps: losses, D's parameters / Adam moments / u, v and the encoders'
    BatchNorm buffers are bit-identical between the replay and step_static_eager; two replays from one state too."""
    from speak_hack_b200.trainer import IRFDDiscriminatorStep

    dev = cuda_device
    xs, xt = _pair(dev)
    _, sd = _converged(dev, xs)
    runs = {}
    for graph in (True, False):
        net = _net(dev, state=sd)
        ds = IRFDDiscriminatorStep(net, use_cuda_graph=graph)
        torch.manual_seed(21)
        torch.cuda.manual_seed(22)
        seq = []
        for _ in range(3):
            loss = ds.step(xs, xt) if graph else ds.step_static_eager(xs, xt)
            seq.append(torch.stack([loss] + list(ds.last)).clone())
        torch.cuda.synchronize()
        runs[graph] = (seq, [t.clone() for t in _d_state(net, ds)])
        if graph:
            assert ds.captures == 1 and ds.step_count == 3 and ds.graph_launches > 0
            g_net, g_ds = net, ds
    print(f"[d-graph] replay losses {[s.tolist() for s in runs[True][0]]}")
    for a, b in zip(runs[True][0], runs[False][0]):
        assert torch.equal(a, b), (a, b)
    assert all(torch.isfinite(s).all() for s in runs[True][0])
    for a, b in zip(runs[True][1], runs[False][1]):
        assert torch.equal(a, b)
    # two replays from the same state
    state = _d_state(g_net, g_ds)
    snap = [t.clone() for t in state]
    step, cpu, cud = g_ds.step_count, torch.get_rng_state(), torch.cuda.get_rng_state(dev)
    outs = []
    for _ in range(2):
        for t, c in zip(state, snap):
            t.copy_(c)
        g_ds.step_count = step
        g_ds.step_dev.fill_(step)
        torch.set_rng_state(cpu)
        torch.cuda.set_rng_state(cud, dev)
        loss = g_ds.step(xs, xt)
        outs.append([torch.stack([loss] + list(g_ds.last)).clone()] + [t.clone() for t in state])
    torch.cuda.synchronize()
    assert g_ds.captures == 1
    assert all(torch.equal(a, b) for a, b in zip(*outs))


def test_graph_step_matches_eager_step(cuda_device):
    """noise_std = 0, zero generator noise weights, no style mixing: both paths are deterministic, so one graphed step
    and one eager step from the same state agree up to summation order (native vs ATen spectral norm, one stacked vs two
    generator calls)."""
    from speak_hack_b200.trainer import IRFDDiscriminatorStep

    dev = cuda_device
    xs, xt = _pair(dev)
    _, sd = _converged(dev, xs)
    res = {}
    for graph in (False, True):
        net = _net(dev, state=sd)
        net.Gd.style_mixing_prob = 0.0
        with torch.no_grad():
            for n, p in net.Gd.named_parameters():
                if "noise" in n:
                    p.zero_()
        ds = IRFDDiscriminatorStep(net, noise_std=0.0, use_cuda_graph=graph)
        torch.manual_seed(31)
        torch.cuda.manual_seed(32)
        loss = ds.step(xs, xt)
        torch.cuda.synchronize()
        bn = [bf.clone() for e in (net.Ei, net.Ee, net.Ep) for bf in e.buffers()]
        res[graph] = (float(loss), [float(t) for t in ds.last], ds.gflat.clone(), bn)
    e_loss = abs(res[True][0] - res[False][0]) / abs(res[False][0])
    e_grad = _rel(res[True][2], res[False][2])
    print(f"[d-graph] graph vs eager: loss {res[True][0]:.6e} vs {res[False][0]:.6e} (rel {e_loss:.2e}), "
          f"real/fake/R1 {res[True][1]} vs {res[False][1]}, D gradient rel {e_grad:.2e}")
    # Measured on a B200: loss rel 2.3e-5 (real-image BCE bit-identical, fake BCE 4.5e-5 apart: the stacked generator
    # call's images differ from the two separate calls' in summation order), D gradient rel 3.0e-2.  The gradient bound
    # is loose because the gradient is ill-conditioned at this state: D's logits are ~0 for every image (loss_real =
    # ln 2), so the real and fake BCE gradients, -0.4 dD/dW and +0.4 dD/dW, nearly cancel (for dense1's bias exactly
    # up to the logit differences) and the image differences above are amplified in what is left.
    assert e_loss < 1e-3 and e_grad < 6e-2
    assert all(torch.equal(a, b) for a, b in zip(res[True][3], res[False][3]))


def test_interleaved_with_graphed_g_step(cuda_device):
    """G replay, D replay, G replay, D replay: each D replay sees the Gd weights the G step just wrote — it equals a D
    graph captured fresh after every G step, bit for bit."""
    from speak_hack_b200.trainer import IRFDDiscriminatorStep, IRFDTrainer

    dev = cuda_device
    xs, xt = _pair(dev)
    _, sd = _converged(dev, xs)
    runs = {}
    for fresh in (False, True):
        net = _net(dev, state=sd)
        tr = IRFDTrainer(net, use_cuda_graph=True)
        ds = IRFDDiscriminatorStep(net, use_cuda_graph=True)
        torch.manual_seed(41)
        torch.cuda.manual_seed(42)
        seq = []
        for _ in range(2):
            tr.train_step(xs, xt)
            if fresh:
                ds.graph = None
            seq.append(torch.stack([ds.step(xs, xt)] + list(ds.last)).clone())
        torch.cuda.synchronize()
        runs[fresh] = (seq, ds.flat.clone(), tr.flat.clone(), ds.captures)
    assert runs[False][3] == 1 and runs[True][3] == 2
    print(f"[d-graph] interleaved D losses {[s.tolist() for s in runs[False][0]]}")
    assert torch.equal(runs[False][2], runs[True][2])
    for a, b in zip(runs[False][0], runs[True][0]):
        assert torch.equal(a, b), (a, b)
    assert torch.equal(runs[False][1], runs[True][1])


def test_cpu_rng_stream_matches_eager_step(cuda_device):
    """The graphed step draws the swap and style-mixing decisions from the CPU generator exactly as model(x_s, x_t)
    does in the eager step (style mixing on, so both rand and randint are drawn)."""
    from speak_hack_b200.trainer import IRFDDiscriminatorStep

    dev = cuda_device
    xs, xt = _pair(dev)
    _, sd = _converged(dev, xs)
    states = {}
    for graph in (False, True):
        net = _net(dev, state=sd)
        assert net.Gd.style_mixing_prob > 0
        ds = IRFDDiscriminatorStep(net, use_cuda_graph=graph)
        torch.manual_seed(51)
        for _ in range(4):
            ds.step(xs, xt)
        torch.cuda.synchronize()
        states[graph] = torch.get_rng_state()
    assert torch.equal(states[False], states[True])


def test_recapture_triggers(cuda_device):
    from speak_hack_b200.trainer import IRFDDiscriminatorStep

    dev = cuda_device
    xs, xt = _pair(dev)
    net, _ = _converged(dev, xs)
    ds = IRFDDiscriminatorStep(net, use_cuda_graph=True)
    ds.step(xs, xt)
    ds.step(xs, xt)
    assert ds.captures == 1
    ds.r1_weight = 2.0
    ds.step(xs, xt)
    assert ds.captures == 2
    ds.lr = 1e-4
    ds.step(xs, xt)
    assert ds.captures == 3
    xs4, xt4 = _pair(dev, 4)
    ds.step(xs4, xt4)
    assert ds.captures == 4
    ds.step(xs4, xt4)
    assert ds.captures == 4
    net.load_state_dict({k: v.clone() for k, v in net.state_dict().items()})
    loss = ds.step(xs4, xt4)
    torch.cuda.synchronize()
    assert ds.captures == 5 and torch.isfinite(loss) and ds.step_count == 7


def _dp_worker(rank, world, port, out):
    import torch.distributed as dist

    from speak_hack_b200.trainer import IRFDDiscriminatorStep

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        xs, xt = _pair(dev)
        xs, xt = xs + 0.01 * rank, xt - 0.01 * rank   # different shards, so unaveraged gradients would differ
        net, _ = _converged(dev, xs)
        ds = IRFDDiscriminatorStep(net, use_cuda_graph=True)
        for _ in range(3):
            ds.step(xs, xt)
        torch.cuda.synchronize()
        parts = [torch.empty_like(ds.flat) for _ in range(world)]
        dist.all_gather(parts, ds.flat)
        if rank == 0:
            torch.save([p.cpu() for p in parts], out)
    finally:
        dist.destroy_process_group()


def test_data_parallel_ranks_stay_identical(cuda_device, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip(f"data-parallel check needs >= 2 GPUs, this machine has {torch.cuda.device_count()}")
    import socket

    import torch.multiprocessing as mp

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    out = str(tmp_path / "flat.pt")
    mp.spawn(_dp_worker, args=(2, port, out), nprocs=2, join=True)
    a, b = torch.load(out)
    assert torch.equal(a, b)
