"""`train_graph.GraphedStep` around the pre-training step of `model.nerf_pretrain.Graph` (reference model/nerf_pretrain.py:513-586):
render(mode='train') -> compute_loss -> backward -> Adam(capturable) -> the weight re-pack, with the whole plain model (trunk and
head) training.  The replayed run must equal the eager run of the same steps bit for bit in both training precisions (bf16, and
the <= 1e-4 mode on the tensor cores), with the view matrices built inside the graph or handed in as static inputs; stratified
jitter is drawn afresh on every replay; what decides on the host refuses to be captured; and the step captures with the
device-epoch peer exchange (parallel.PeerGradExchange(capturable=True)) over the whole model's gradients, for ranks of one
process and for two processes."""
import os
import time

import pytest
import torch
import torch.distributed as dist

from texpose_b200 import _C, camera, compute_box, parallel, synth
from texpose_b200.config import AttrDict, env_opt
from texpose_b200.model.nerf_pretrain import Graph
from texpose_b200.train_graph import GraphedStep

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B, HW, N, RAYS = 2, 64, 64, 512
K = torch.tensor([[286.2, 0, 32 - 286.2 * 0.3 / 8], [0, 286.8, 32 + 286.8 * 0.2 / 8], [0, 0, 1]])
MODES = dict(bf16=AttrDict(mlp="bf16"), fp32_tc=AttrDict(mlp="fp32", fp32_engine="tc"))
ROUTE = dict(bf16=("tp_tc32_forward", "tp_tc_chain_backward"), fp32_tc=("tp_tc32_forward_split_save", "tp_tc_chain_backward_split"))
STATIC = dict(ray_idx=((B, RAYS // B), torch.long), image=((B, 3, HW, HW), torch.float32), obj_mask=((B, HW, HW), torch.float32),
              depth_gt=((B, HW, HW), torch.float32), pose=((B, 3, 4), torch.float32), intr=((B, 3, 3), torch.float32),
              z_near=((B, HW * HW), torch.float32), z_far=((B, HW * HW), torch.float32))
VIEW = dict(kinv=((B, 3, 3), torch.float32), pinv=((B, 3, 4), torch.float32))


def pretrain_setup(mode, dev=DEV, stratified=False, static_view=False, lr=1e-3, exchange=None, **b200):
    """-> (opt, graph, optimizer, static buffers, fn): fn is one pre-training step on the static buffers (no optimizer step).
    static_view: K^-1 / pose^-1 are static inputs too (camera.view_matrices, computed eagerly by `batch`)."""
    opt = env_opt(H=HW, W=HW, sample_intvs=N, device=dev)
    opt.nerf.rand_rays = RAYS
    opt.nerf.sample_stratified = stratified
    opt.loss_weight = AttrDict(render=0, mask=-1, depth=-1)
    opt.data.erode_mask_loss = False
    opt.b200 = AttrDict(MODES[mode], rng="torch", **b200)
    torch.manual_seed(0)
    g = Graph(opt).to(dev).train()
    optim = torch.optim.Adam(g.nerf.parameters(), lr=lr, capturable=True)
    static = {k: torch.zeros(*shape, dtype=dt, device=dev) for k, (shape, dt) in
              dict(STATIC, **(VIEW if static_view else {})).items()}
    idx = torch.arange(B, device=dev)

    def fn():
        var = AttrDict(idx=idx, **{k: static[k] for k in STATIC})
        view = (static["kinv"], static["pinv"]) if static_view else None
        var.update(g.render(opt, var.pose, intr=var.intr, ray_idx=var.ray_idx, depth_range=(var.z_near[:, :, None], var.z_far[:, :, None]),
                            mode="train", view=view))
        loss = g.compute_loss(opt, var, mode="train")
        total = sum(10 ** float(opt.loss_weight[k]) * loss[k] for k in loss)
        total.backward()
        if exchange is not None:
            exchange(g)
        return total

    return opt, g, optim, static, fn


def batch(opt, i, dev=DEV, rank=0, static_view=False):
    """Batch i of rank `rank`: its own views, frame, masks and depth ranges, and the ray subset `Graph.get_ray_idx` draws --
    eagerly, with the reference's torch.randperm (seeded here so that every run sees the same subsets)."""
    s = 100 + i + 1000 * rank
    gen = torch.Generator().manual_seed(s)
    pose = synth.poses([(s + b) % 13 for b in range(B)]).to(dev)
    intr = K.repeat(B, 1, 1).to(dev)
    lo, hi = [t.to(dev) for t in synth.padded_aabb()]
    zn, zf = compute_box.box_range(pose, intr, lo, hi, HW, HW, *synth.BG_RANGE)
    torch.manual_seed(s)
    var = Graph.get_ray_idx(opt, AttrDict(idx=list(range(B))))
    out = dict(ray_idx=var.ray_idx, image=torch.rand(B, 3, HW, HW, generator=gen).to(dev), obj_mask=(zf < 29).view(B, HW, HW).float(),
               depth_gt=(7.5 + torch.rand(B, HW, HW, generator=gen)).to(dev), pose=pose, intr=intr, z_near=zn, z_far=zf)
    if static_view:
        out["kinv"], out["pinv"] = camera.view_matrices(pose, intr, one_launch=camera.one_launch_matrices(opt))
    return out


def _fill(static, values):
    for k, v in values.items():
        static[k].copy_(v)


@pytest.mark.parametrize("mode,static_view", [("bf16", False), ("fp32_tc", False), ("fp32_tc", True)])
def test_graphed_pretrain_run_equals_the_eager_run_bit_for_bit(mode, static_view):
    warm, steps = 2, 4
    # ---- eager: warm-up steps on batch 0, then batches 1..steps
    opt_a, g_a, optim_a, static_a, fn_a = pretrain_setup(mode)
    losses_a = []
    for j, i in enumerate([0] * warm + list(range(1, steps + 1))):
        _fill(static_a, batch(opt_a, i))
        optim_a.zero_grad(set_to_none=True)
        _C.launch_counts.clear()
        losses_a.append(fn_a().detach().clone())
        optim_a.step()
        if j == 0:
            fwd, bwd = ROUTE[mode]
            assert _C.launch_counts.get(fwd) == 1 and _C.launch_counts.get(bwd) == 1, _C.launch_counts
            assert "tp_linear_forward" not in _C.launch_counts
    # ---- graph: the same weights, batch 0 in the static buffers during warm-up and capture
    opt_b, g_b, optim_b, static_b, fn_b = pretrain_setup(mode, static_view=static_view)
    _fill(static_b, batch(opt_b, 0, static_view=static_view))
    step = GraphedStep(fn_b, optim_b, static=static_b, warmup=warm)
    feeds = [batch(opt_b, i, static_view=static_view) for i in range(1, steps + 1)]      # eager: randperm, (view matrices)
    _C.launch_counts.clear()
    losses_b = [step(**f).detach().clone() for f in feeds]
    assert not _C.launch_counts, "a replay must not issue C-ABI launches from Python"
    assert step.replays == steps
    for a, b in zip(losses_a[warm:], losses_b):
        assert torch.equal(a, b), (float(a), float(b))
    assert len({float(x) for x in losses_b}) == steps                 # every replay saw its own batch
    for (n, pa), (_, pb) in zip(g_a.named_parameters(), g_b.named_parameters()):
        assert torch.equal(pa, pb), n
    torch.manual_seed(0)
    fresh = Graph(opt_b).to(DEV)
    for (n, p0), (_, pb) in zip(fresh.named_parameters(), g_b.named_parameters()):
        assert float((p0 - pb).detach().abs().max()) > 1e-5, n                 # every layer trained inside the graph, the trunk too


def test_stratified_jitter_is_drawn_afresh_on_every_replay():
    opt, g, optim, static, fn = pretrain_setup("bf16", stratified=True, lr=0.0)      # lr 0: only the jitter can change the loss
    _fill(static, batch(opt, 0))
    step = GraphedStep(fn, optim, static=static, warmup=2)
    before = [p.detach().clone() for p in g.parameters()]
    a = float(step().detach().clone())
    b = float(step().detach().clone())
    assert a == a and b == b and abs(a) < float("inf") and abs(b) < float("inf"), (a, b)
    assert a != b, "the same batch replayed twice must see two jitter draws"
    for p, q in zip(before, g.parameters()):
        assert torch.equal(p, q)


def test_version_keyed_caches_see_the_replayed_weights():
    """An eager render between replays must render the weights the replays wrote (NeRF._tc32_parameters is keyed by _version)."""
    opt, g, optim, static, fn = pretrain_setup("fp32_tc")
    _fill(static, batch(opt, 0))
    step = GraphedStep(fn, optim, static=static, warmup=2)
    f = batch(opt, 1)

    def frame(model):
        with torch.no_grad():
            return model.render(opt, f["pose"], intr=f["intr"], ray_idx=f["ray_idx"],
                                depth_range=(f["z_near"][:, :, None], f["z_far"][:, :, None]), mode="val").rgb.clone()

    step(**f)
    first = frame(g)
    step(**f)
    second = frame(g)
    g_ref = Graph(opt).to(DEV)
    g_ref.load_state_dict(g.state_dict())                             # a model that never saw a replay: fresh packs
    assert not torch.equal(first, second)
    assert torch.equal(second, frame(g_ref))


@pytest.mark.parametrize("what,b200,match", [("nan_guard", dict(nan_guard=True), "nan_guard"),
                                             ("host matrices", dict(), "HOST_MATRICES")])
def test_host_decisions_refuse_to_be_captured(what, b200, match):
    mode = "fp32_tc"
    opt, g, optim, static, fn = pretrain_setup(mode, **b200)
    _fill(static, batch(opt, 0))
    host = camera.HOST_MATRICES
    camera.HOST_MATRICES = what == "host matrices"
    try:
        with pytest.raises(RuntimeError, match=match):
            GraphedStep(fn, optim, static=static, warmup=1)            # the eager warm-up runs; the capture raises
    finally:
        camera.HOST_MATRICES = host
    torch.cuda.synchronize()
    _C.launch_counts.clear()
    fn()                                                             # eagerly the same step still runs
    assert _C.launch_counts


# ---- data-parallel: the whole model's gradients through the device-epoch peer exchange --------------------------------------
def _rank_order_mean(parts):
    want = parts[0].cpu()
    for p in parts[1:]:
        want = want + p.cpu()
    return want / len(parts)


def _local_exchanges(models, grid_ctas=4, timeout_ms=20000):
    """PeerGradExchange(capturable=True) for `world` ranks that live in this process on one device (one window each, opened
    directly instead of through IPC handles): the exchange path of the multi-process set-up, without a process group."""
    dev = torch.device(DEV)
    exs = []
    for m in models:
        ex = parallel.PeerGradExchange.__new__(parallel.PeerGradExchange)
        parallel.GradBucket.__init__(ex, [p for p in m.parameters() if p.requires_grad])
        ex.n = ex.flat.numel()
        ex.window = parallel.PeerWindow(ex.n, dev)
        ex.flat = torch.zeros((ex.n + 3) // 4 * 4, device=dev)
        ex.staging = torch.zeros_like(ex.flat)
        ex.epoch, ex.grid_ctas, ex.timeout_ms, ex.capturable, ex.group = 0, grid_ctas, timeout_ms, True, None
        exs.append(ex)
    for r, ex in enumerate(exs):
        ex.rank, ex.world, ex.ptrs = r, len(exs), [e.window.ptr for e in exs]
    torch.cuda.synchronize()
    return exs


@pytest.mark.parametrize("world", [2, 3])
def test_graphed_pretrain_step_with_the_peer_exchange_ranks_of_one_process(world):
    """Each rank replays its own captured step (its own batches) on its own stream; the peer exchange inside every graph averages
    the whole model's gradients, so all ranks keep identical weights, and every exchanged bucket is the rank-order mean."""
    warm, steps = 2, 3
    ranks = []
    exchanges, on = {}, [False]
    for r in range(world):
        opt, g, optim, static, fn = pretrain_setup("bf16", exchange=lambda m: exchanges[id(m)].allreduce_mean() if on[0] else None)
        ranks.append(dict(opt=opt, g=g, optim=optim, static=static, fn=fn, stream=torch.cuda.Stream(DEV)))
    exs = _local_exchanges([rk["g"] for rk in ranks])
    for rk, ex in zip(ranks, exs):
        exchanges[id(rk["g"])] = ex
    n = exs[0].n
    print(f"pre-training bucket: {n} floats ({4 * n / 2 ** 20:.2f} MiB), world {world}")
    # every batch is made up front: while one rank's exchange waits for the others, the host only copies and launches
    feeds = [[batch(rk["opt"], i, rank=r) for i in range(steps + 1)] for r, rk in enumerate(ranks)]
    shared = batch(ranks[0]["opt"], 0)
    graphs = []
    try:
        def one(r, values):
            rk = ranks[r]
            with torch.cuda.stream(rk["stream"]):
                _fill(rk["static"], values)
                rk["optim"].zero_grad(set_to_none=True)
                rk["fn"]()
                rk["optim"].step()

        torch.cuda.synchronize()
        for r in range(world):              # no exchange yet: lazy set-up (tables, optimizer state, cached blocks) on the same batch
            one(r, shared)
        torch.cuda.synchronize()
        on[0] = True
        for _ in range(warm):               # eager exchanges, every rank: device epochs 1..warm
            for r in range(world):
                one(r, feeds[r][0])
        torch.cuda.synchronize()
        for rk in ranks:
            rk["optim"].zero_grad(set_to_none=True)
            graphs.append(torch.cuda.CUDAGraph())
            with torch.cuda.graph(graphs[-1], stream=rk["stream"]):
                rk["fn"]()
                rk["optim"].step()
        _C.launch_counts.clear()
        for i in range(1, steps + 1):
            for r in (range(world) if i % 2 else reversed(range(world))):      # launch order must not matter
                rk = ranks[r]
                with torch.cuda.stream(rk["stream"]):
                    _fill(rk["static"], feeds[r][i])
                    graphs[r].replay()
            torch.cuda.synchronize()
            want = _rank_order_mean([ex.staging[:n] for ex in exs])   # staging = each rank's own gradients of this step
            assert len({float(ex.staging[:n].abs().sum()) for ex in exs}) == world     # the ranks saw different batches
            for r, ex in enumerate(exs):
                assert torch.equal(ex.flat[:n].cpu(), want), (world, i, r)
        assert not _C.launch_counts
        for ex in exs:
            assert ex.window.status() == 0
        params = [torch.cat([p.detach().reshape(-1) for p in rk["g"].parameters()]) for rk in ranks]
        for r in range(1, world):
            assert torch.equal(params[0], params[r]), r
        torch.manual_seed(0)
        fresh = torch.cat([p.detach().reshape(-1) for p in Graph(ranks[0]["opt"]).to(DEV).parameters()])
        assert not torch.equal(fresh, params[0])
    finally:
        torch.cuda.synchronize()
        del graphs
        for ex in exs:
            ex.window.close()


def _free_port():
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _train_worker(rank, world, port, ret):
    """The graphed pre-training step, one GPU per process, each rank on its own batches; eager run with the same exchange."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = f"cuda:{rank}"
    torch.cuda.set_device(dev)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        warm, steps = 2, 4
        runs = []
        for graphed in (False, True):
            box = {}
            opt, g, optim, static, fn = pretrain_setup("bf16", dev=dev, exchange=lambda m: box["ex"].allreduce_mean())
            box["ex"] = ex = parallel.PeerGradExchange([p for p in g.parameters() if p.requires_grad], capturable=True)
            if graphed:
                _fill(static, batch(opt, 0, dev, rank))
                step = GraphedStep(fn, optim, static=static, warmup=warm)
                losses = [step(**batch(opt, i, dev, rank)).detach().clone() for i in range(1, steps + 1)]
            else:
                losses = []
                for i in [0] * warm + list(range(1, steps + 1)):
                    _fill(static, batch(opt, i, dev, rank))
                    optim.zero_grad(set_to_none=True)
                    losses.append(fn().detach().clone())
                    optim.step()
                losses = losses[warm:]
            torch.cuda.synchronize()
            ex.check()
            runs.append((losses, [p.detach().clone() for p in g.parameters()]))
            step = None
            ex.close()
        (le, pe), (lg, pg) = runs
        ok = all(torch.equal(a, b) for a, b in zip(le, lg)) and all(torch.equal(a, b) for a, b in zip(pe, pg))
        mine = torch.cat([p.reshape(-1) for p in pg]).cpu()
        theirs = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(theirs, mine)
        ret[rank] = bool(ok and all(torch.equal(mine, t) for t in theirs))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="two processes need two GPUs (one device would starve the waits)")
def test_two_processes_graphed_pretrain_step():
    import torch.multiprocessing as mp
    _C.build()
    world = 2
    ret = mp.Manager().dict()
    ctx = mp.spawn(_train_worker, args=(world, _free_port(), ret), nprocs=world, join=False)
    deadline = time.time() + 480
    done = False
    while not done and time.time() < deadline:
        done = ctx.join(timeout=5)
    if not done:
        for p in ctx.processes:
            if p.is_alive():
                p.terminate()
        pytest.fail("the training processes did not finish")
    assert all(ret.get(r) for r in range(world)), dict(ret)
