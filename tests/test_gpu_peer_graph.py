"""The peer-window gradient exchange with a device-held epoch (csrc/peer.cu: tp_peer_stage + tp_peer_allreduce_mean_dev) and
`PeerGradExchange(capturable=True)`: the exchange captured in CUDA graphs and replayed must give, on every replay, the same bits as
the rank-order mean computed on the CPU -- i.e. no epoch or parity buffer is frozen at capture.  Covered: several "ranks" of one
process, each replaying its own graph on its own stream; a missing peer (bounded wait, status word, NaN); the guard against
capturing a non-capturable exchange; the whole texture-learner step inside `GraphedStep` at world 1; two processes through real
CUDA IPC handles."""
import os
import socket
import time

import pytest
import torch
import torch.distributed as dist

from texpose_b200 import _C, compute_box, parallel, synth
from texpose_b200.config import AttrDict, adapt_gan_opt
from texpose_b200.model.base import summarize_loss
from texpose_b200.model.nerf_adapt_st_gan import Graph
from texpose_b200.train_graph import GraphedStep

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rank_order_mean(grads, dev):
    want = grads[0].cpu()
    for gr in grads[1:]:
        want = want + gr.cpu()
    return (want / len(grads)).to(dev)       # IEEE division as on the CPU (torch's CUDA `/ scalar` multiplies by 1/world)


@pytest.mark.parametrize("n", [7, 1000, 421385])
@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_captured_ranks_of_one_process_bit_exact(world, n):
    dev = torch.device(DEV)
    grid = 4            # small grids: every rank's waiting CTAs fit on the one device together
    n4 = (n + 3) // 4 * 4
    wins = [parallel.PeerWindow(n, dev) for _ in range(world)]
    ptrs = [w.ptr for w in wins]
    inputs = [torch.zeros(n, device=dev) for _ in range(world)]           # the graphs' static inputs
    staging = [torch.zeros(n4, device=dev) for _ in range(world)]
    outs = [torch.full((n4,), -7.0, device=dev) for _ in range(world)]
    streams = [torch.cuda.Stream(dev) for _ in range(world)]
    gen = torch.Generator(device=dev).manual_seed(n + world)

    def exchange(r):        # on the current stream
        staging[r][:n].copy_(inputs[r])
        parallel.peer_stage(ptrs[r], n, staging[r])
        parallel.peer_allreduce_mean_dev(ptrs, r, n, outs[r], grid_ctas=grid, timeout_ms=5000)

    def step(i, run):
        grads = [torch.randn(n, device=dev, generator=gen) * (10.0 ** (r % 3)) for r in range(world)]
        for r in range(world):
            inputs[r].copy_(grads[r])
        torch.cuda.synchronize()
        for r in (range(world) if i % 2 else reversed(range(world))):     # launch order must not matter
            with torch.cuda.stream(streams[r]):
                run(r)
        torch.cuda.synchronize()
        want = _rank_order_mean(grads, dev)
        for r in range(world):
            assert torch.equal(outs[r][:n], want), (world, n, i, r)

    graphs = []
    try:
        step(1, exchange)                                  # eager: device epoch 1, and every kernel is loaded before the capture
        for r in range(world):
            graphs.append(torch.cuda.CUDAGraph())
            with torch.cuda.graph(graphs[r], stream=streams[r]):
                exchange(r)
        replay = lambda r: graphs[r].replay()
        for i in range(2, 5):
            step(i, replay)
        step(5, exchange)                                  # an eager exchange between two replays advances the same counter
        for i in range(6, 9):
            step(i, replay)
        for w in wins:
            assert w.status() == 0
    finally:
        torch.cuda.synchronize()
        del graphs
        for w in wins:
            w.close()


def test_missing_peer_device_epoch_times_out_and_reports():
    dev = torch.device(DEV)
    n = 4096
    wins = [parallel.PeerWindow(n, dev) for _ in range(2)]
    ptrs = [w.ptr for w in wins]
    srcs = [torch.full((n,), 1.0 + r, device=dev) for r in range(2)]
    outs = [torch.full((n,), 3.0, device=dev) for _ in range(2)]
    streams = [torch.cuda.Stream(dev) for _ in range(2)]
    try:
        for _ in range(2):                                 # device epochs 1 and 2 with both ranks present
            for r in range(2):
                with torch.cuda.stream(streams[r]):
                    parallel.peer_stage(ptrs[r], n, srcs[r])
                    parallel.peer_allreduce_mean_dev(ptrs, r, n, outs[r], grid_ctas=4, timeout_ms=5000)
            torch.cuda.synchronize()
            assert all(bool((o == 1.5).all()) for o in outs)
        parallel.peer_stage(ptrs[0], n, srcs[0])           # epoch 3: rank 1 never shows up
        parallel.peer_allreduce_mean_dev(ptrs, 0, n, outs[0], grid_ctas=4, timeout_ms=50)
        torch.cuda.synchronize()
        assert wins[0].status() == 3 and wins[1].status() == 0
        assert torch.isnan(outs[0]).all()
    finally:
        for w in wins:
            w.close()


def test_device_epoch_argument_errors():
    dev = torch.device(DEV)
    w = parallel.PeerWindow(64, dev)
    try:
        src, out = torch.zeros(64, device=dev), torch.zeros(64, device=dev)
        with pytest.raises(RuntimeError):
            parallel.peer_stage(w.ptr, 64, src[1:])                              # too small
        with pytest.raises(RuntimeError):
            parallel.peer_stage(w.ptr, 8, src[1:])                               # misaligned
        with pytest.raises(RuntimeError):
            parallel.peer_stage(w.ptr + 16, 8, src)                              # not a window base
        with pytest.raises(RuntimeError):
            parallel.peer_allreduce_mean_dev([w.ptr], 1, 64, out)                # rank outside the world
        with pytest.raises(RuntimeError):
            parallel.peer_allreduce_mean_dev([w.ptr], 0, 64, out[1:])            # too small / misaligned
    finally:
        w.close()


@pytest.fixture
def world1_group():
    """A single-process gloo process group over an in-memory store (no sockets)."""
    assert not dist.is_initialized()
    dist.init_process_group("gloo", store=dist.HashStore(), rank=0, world_size=1)
    yield
    dist.destroy_process_group()


def test_capture_guard(world1_group):
    lin = torch.nn.Linear(37, 19).to(DEV)
    params = list(lin.parameters())
    grads = [torch.randn(p.shape, device=DEV) for p in params]
    want = torch.cat([g.reshape(-1) for g in grads])

    plain = parallel.PeerGradExchange(params)
    try:
        for p, g in zip(params, grads):
            p.grad = g
        probe = torch.zeros(1, device=DEV)
        with pytest.raises(RuntimeError, match="capturable=True"):
            with torch.cuda.graph(torch.cuda.CUDAGraph()):
                probe.add_(1.0)
                plain.allreduce_mean()
        plain.allreduce_mean()                                                   # eagerly it still works
        assert torch.equal(torch.cat([p.grad.reshape(-1) for p in params]), want)
        plain.check()
    finally:
        plain.close()

    ex = parallel.PeerGradExchange(params, capturable=True)
    try:
        static = [torch.zeros_like(p) for p in params]
        for p, s in zip(params, static):
            p.grad = s
        ex.allreduce_mean()                                                      # eager warm-up: device epoch 1
        for p, s in zip(params, static):
            p.grad = s
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            ex.allreduce_mean()
        for i in range(3):
            fresh = [torch.randn(p.shape, device=DEV) for p in params]
            for s, f in zip(static, fresh):
                s.copy_(f)
            graph.replay()
            torch.cuda.synchronize()
            assert torch.equal(torch.cat([p.grad.reshape(-1) for p in params]), torch.cat([f.reshape(-1) for f in fresh])), i
        ex.check()
    finally:
        ex.close()


# ---- the whole texture-learner step (the shape of tests/test_gpu_train_graph.py, jitter off) -----------------------------------
B, P, N, HW = 4, 8, 32, 64


def _train_setup(dev, exchange: bool):
    opt = adapt_gan_opt(H=HW, W=HW, sample_intvs=N, device=dev)
    opt.batch_size = B
    opt.nerf.sample_stratified = False            # no jitter: the runs need no common random stream
    opt.b200 = AttrDict(mlp="bf16", rng="torch")
    torch.manual_seed(0)
    g = Graph(opt, n_train_images=B).to(dev).train()
    optim = torch.optim.Adam([dict(params=g.nerf.parameters(), lr=1.e-3)], capturable=True)
    optim.add_param_group(dict(params=g.latent_vars_light.parameters(), lr=1.e-3))
    optim.add_param_group(dict(params=g.latent_vars_trans.parameters(), lr=1.e-3))
    ex = parallel.PeerGradExchange([p for p in g.parameters() if p.requires_grad], capturable=True) if exchange else None
    pose = synth.poses(list(range(B))).to(dev)
    K = torch.tensor([[286.2, 0, 32 - 286.2 * 0.3 / 8], [0, 286.8, 32 + 286.8 * 0.2 / 8], [0, 0, 1]])
    intr = K.repeat(B, 1, 1).to(dev)
    lo, hi = [t.to(dev) for t in synth.padded_aabb()]
    zn, zf = compute_box.box_range(pose, intr, lo, hi, HW, HW, *synth.BG_RANGE)
    static = dict(coords=torch.zeros(B, P, P, 2, device=dev), image=torch.zeros(B, 3, HW, HW, device=dev),
                  mask=torch.zeros(B, HW, HW, device=dev))
    idx = torch.arange(B, device=dev)

    def fn():
        ret = g.render(opt, pose, intr=intr, ray_idx=static["coords"], depth_range=(zn[:, :, None], zf[:, :, None]),
                       sample_idx=idx, mode="train")
        var = AttrDict(idx=idx, image=static["image"], obj_mask=static["mask"], ray_idx=static["coords"])
        var.update(ret)
        total = summarize_loss(opt, var, g.compute_loss(opt, var, mode="train"))["all"]
        total.backward()
        if ex is not None:
            ex.allreduce_mean()
        return total

    return g, optim, static, fn, ex


def _batch(i, dev, rank=0):
    gen = torch.Generator().manual_seed(100 + i + 1000 * rank)
    return dict(coords=synth.patch_coords(B, P, seed=50 + i + 1000 * rank)[0].to(dev),
                image=torch.rand(B, 3, HW, HW, generator=gen).to(dev),
                mask=(torch.rand(B, HW, HW, generator=gen) > 0.3).float().to(dev))


def _eager_run(dev, exchange, warm, steps, rank=0):
    g, optim, static, fn, ex = _train_setup(dev, exchange)
    losses = []
    for i in [0] * warm + list(range(1, steps + 1)):
        for k, v in _batch(i, dev, rank).items():
            static[k].copy_(v)
        optim.zero_grad(set_to_none=True)
        losses.append(fn().detach().clone())
        optim.step()
    if ex is not None:
        ex.check()
        ex.close()
    return losses[warm:], [p.detach().clone() for p in g.parameters()]


def _graphed_run(dev, warm, steps, rank=0):
    g, optim, static, fn, ex = _train_setup(dev, True)
    for k, v in _batch(0, dev, rank).items():
        static[k].copy_(v)
    step = GraphedStep(fn, optim, static=static, warmup=warm)        # the warm-up exchanges are eager: device epochs 1..warm
    losses = [step(**_batch(i, dev, rank)).detach().clone() for i in range(1, steps + 1)]
    torch.cuda.synchronize()
    ex.check()
    params = [p.detach().clone() for p in g.parameters()]
    del step
    ex.close()
    return losses, params


def test_graphed_step_with_capturable_exchange_equals_eager(world1_group):
    warm, steps = 2, 4
    losses_e, params_e = _eager_run(DEV, True, warm, steps)
    losses_g, params_g = _graphed_run(DEV, warm, steps)
    losses_0, params_0 = _eager_run(DEV, False, warm, steps)          # the mean over one rank is exact: same as no exchange
    assert len({float(x) for x in losses_g}) == steps
    for a, b, c in zip(losses_e, losses_g, losses_0):
        assert torch.equal(a, b) and torch.equal(a, c), (float(a), float(b), float(c))
    for i, (a, b, c) in enumerate(zip(params_e, params_g, params_0)):
        assert torch.equal(a, b) and torch.equal(a, c), i


# ---- two processes through CUDA IPC ---------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _exchange_worker(rank, world, port, ret):
    """Exchange-only graph: small parameters, the captured exchange against the gloo all_gather of the same gradients."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank % torch.cuda.device_count())
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ex = None
    try:
        torch.manual_seed(0)
        lin = torch.nn.Linear(37, 19).to(dev)
        emb = torch.nn.Embedding(5, 3).to(dev)
        params = list(lin.parameters()) + list(emb.parameters())
        ex = parallel.PeerGradExchange(params, timeout_ms=20000, capturable=True)
        static = [torch.zeros_like(p) for p in params]
        graph = torch.cuda.CUDAGraph()
        ok = True
        for step in range(6):
            g = torch.Generator(device=dev).manual_seed(100 * step + rank)
            grads = [torch.randn(p.shape, device=dev, generator=g) for p in params]
            for s, gr in zip(static, grads):
                s.copy_(gr)
            flat = torch.cat([gr.reshape(-1) for gr in grads])
            parts = [torch.empty_like(flat).cpu() for _ in range(world)]
            dist.all_gather(parts, flat.cpu())
            want = _rank_order_mean(parts, dev)
            if step in (0, 1, 3):          # the calls that read .grad from Python: eager exchanges and the capture
                for p, s in zip(params, static):
                    p.grad = s
            if step in (0, 3):             # eager exchanges: the first one loads the kernels, the other sits between replays
                ex.allreduce_mean()
            else:
                if step == 1:
                    with torch.cuda.graph(graph):
                        ex.allreduce_mean()
                graph.replay()             # reads `static`, and the .grad views of the reduced buffer are the captured ones
            torch.cuda.synchronize()
            ex.check()
            ok = ok and torch.equal(torch.cat([p.grad.reshape(-1) for p in params]), want)
        ret[rank] = bool(ok)
    finally:
        if ex is not None:
            ex.close()
        dist.destroy_process_group()


def _train_worker(rank, world, port, ret):
    """The whole graphed training step, one GPU per process, each rank on its own batches."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = f"cuda:{rank}"
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        warm, steps = 2, 4
        losses_e, params_e = _eager_run(dev, True, warm, steps, rank)
        losses_g, params_g = _graphed_run(dev, warm, steps, rank)
        ok = all(torch.equal(a, b) for a, b in zip(losses_e, losses_g))
        ok = ok and all(torch.equal(a, b) for a, b in zip(params_e, params_g))
        mine = torch.cat([p.reshape(-1) for p in params_g]).cpu()
        theirs = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(theirs, mine)
        ret[rank] = bool(ok and all(torch.equal(mine, t) for t in theirs))
    finally:
        dist.destroy_process_group()


def _spawn(worker, world=2, timeout_s=240):
    import torch.multiprocessing as mp
    _C.build()
    ret = mp.Manager().dict()
    ctx = mp.spawn(worker, args=(world, _free_port(), ret), nprocs=world, join=False)
    deadline = time.time() + timeout_s
    done = False
    while not done and time.time() < deadline:
        done = ctx.join(timeout=5)          # True once every worker has exited; raises if one failed
    if not done:
        for p in ctx.processes:
            if p.is_alive():
                p.terminate()
        pytest.fail(f"{worker.__name__} processes did not finish")
    assert all(ret.get(r) for r in range(world)), dict(ret)


def test_two_processes_captured_exchange():
    _spawn(_exchange_worker)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="two full training steps on one device would starve each other's waits")
def test_two_processes_graphed_training_step():
    _spawn(_train_worker, timeout_s=480)
