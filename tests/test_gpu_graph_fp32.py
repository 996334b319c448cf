"""`train_graph.GraphedStep` in the <= 1e-4 mode on the tensor cores (opt.b200.mlp = 'fp32', fp32_engine = 'tc'): the adaptation
step (split save -> heads_backward_staged(split)) replayed equals its eager run bit for bit, with the view matrices built inside
the graph (torch.linalg.inv_ex) or handed in as static inputs; the pre-training step captured with the CPU-inverted view matrices
of the parity fixtures as static inputs meets, on its first replay, the tolerances the eager step is held to against the real
reference; and the host decisions of the adaptation engine (rng 'philox', nan_guard) and mlp_tc32.check_range refuse capture."""
import pytest
import torch

from texpose_b200 import _C, camera, compute_box, mlp_tc32, synth
from texpose_b200.config import AttrDict, adapt_gan_opt, env_opt
from texpose_b200.model.base import summarize_loss
from texpose_b200.model.nerf_adapt_st_gan import Graph
from texpose_b200.train_graph import GraphedStep
from tests.test_gpu_fp32_train import REL_GRAPH, TOL, _check_grads

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B, P, N, HW = 4, 8, 32, 64
TC = dict(mlp="fp32", fp32_engine="tc")


def _adapt_setup(static_view=False, stratified=False, **b200):
    opt = adapt_gan_opt(H=HW, W=HW, sample_intvs=N, device=DEV)
    opt.batch_size = B
    opt.nerf.sample_stratified = stratified
    opt.b200 = AttrDict(TC, rng="torch")
    opt.b200.update(b200)
    torch.manual_seed(0)
    g = Graph(opt, n_train_images=B).to(DEV).train()
    optim = torch.optim.Adam([dict(params=g.nerf.parameters(), lr=1.e-3)], capturable=True)
    optim.add_param_group(dict(params=g.latent_vars_light.parameters(), lr=1.e-3))
    optim.add_param_group(dict(params=g.latent_vars_trans.parameters(), lr=1.e-3))
    static = dict(coords=torch.zeros(B, P, P, 2, device=DEV), image=torch.zeros(B, 3, HW, HW, device=DEV),
                  mask=torch.zeros(B, HW, HW, device=DEV), pose=torch.zeros(B, 3, 4, device=DEV), intr=torch.zeros(B, 3, 3, device=DEV),
                  z_near=torch.zeros(B, HW * HW, device=DEV), z_far=torch.zeros(B, HW * HW, device=DEV))
    if static_view:
        static.update(kinv=torch.zeros(B, 3, 3, device=DEV), pinv=torch.zeros(B, 3, 4, device=DEV))
    idx = torch.arange(B, device=DEV)

    def fn():
        view = (static["kinv"], static["pinv"]) if static_view else None
        ret = g.render(opt, static["pose"], intr=static["intr"], ray_idx=static["coords"],
                       depth_range=(static["z_near"][:, :, None], static["z_far"][:, :, None]), sample_idx=idx, mode="train", view=view)
        var = AttrDict(idx=idx, image=static["image"], obj_mask=static["mask"], ray_idx=static["coords"])
        var.update(ret)
        total = summarize_loss(opt, var, g.compute_loss(opt, var, mode="train"))["all"]
        total.backward()
        return total

    return opt, g, optim, static, fn


def _batch(i, static_view=False):
    gen = torch.Generator().manual_seed(100 + i)
    pose = synth.poses([(i + b) % 11 for b in range(B)]).to(DEV)
    K = torch.tensor([[286.2, 0, 32 - 286.2 * 0.3 / 8], [0, 286.8, 32 + 286.8 * 0.2 / 8], [0, 0, 1]])
    intr = K.repeat(B, 1, 1).to(DEV)
    lo, hi = [t.to(DEV) for t in synth.padded_aabb()]
    zn, zf = compute_box.box_range(pose, intr, lo, hi, HW, HW, *synth.BG_RANGE)
    out = dict(coords=synth.patch_coords(B, P, seed=50 + i)[0].to(DEV), image=torch.rand(B, 3, HW, HW, generator=gen).to(DEV),
               mask=(torch.rand(B, HW, HW, generator=gen) > 0.3).float().to(DEV), pose=pose, intr=intr, z_near=zn, z_far=zf)
    if static_view:
        out["kinv"], out["pinv"] = camera.view_matrices(pose, intr)
    return out


@pytest.mark.parametrize("static_view", [False, True])
def test_graphed_adaptation_fp32_tc_run_equals_the_eager_run_bit_for_bit(static_view):
    warm, steps = 2, 4
    opt_a, g_a, optim_a, static_a, fn_a = _adapt_setup()
    losses_a = []
    for j, i in enumerate([0] * warm + list(range(1, steps + 1))):
        for k, v in _batch(i).items():
            static_a[k].copy_(v)
        optim_a.zero_grad(set_to_none=True)
        _C.launch_counts.clear()
        losses_a.append(fn_a().detach().clone())
        optim_a.step()
        if j == 0:
            c = _C.launch_counts
            assert c.get("tp_tc32_forward_split_save") == 1 and c.get("tp_tc_chain_backward_split") == 2, c
            assert "tp_linear_forward" not in c
    opt_b, g_b, optim_b, static_b, fn_b = _adapt_setup(static_view)
    for k, v in _batch(0, static_view).items():
        static_b[k].copy_(v)
    step = GraphedStep(fn_b, optim_b, static=static_b, warmup=warm)
    feeds = [_batch(i, static_view) for i in range(1, steps + 1)]
    _C.launch_counts.clear()
    losses_b = [step(**f).detach().clone() for f in feeds]
    assert not _C.launch_counts, "a replay must not issue C-ABI launches from Python"
    for a, b in zip(losses_a[warm:], losses_b):
        assert torch.equal(a, b), (float(a), float(b))
    assert len({float(x) for x in losses_b}) == steps
    for (n, pa), (_, pb) in zip(g_a.named_parameters(), g_b.named_parameters()):
        assert torch.equal(pa, pb), n
    torch.manual_seed(0)
    fresh = Graph(adapt_gan_opt(H=HW, W=HW, sample_intvs=N, device=DEV), n_train_images=B).to(DEV)
    moved = 0.0
    for (n, p0), (_, pb) in zip(fresh.named_parameters(), g_b.named_parameters()):
        moved = max(moved, float((p0 - pb).abs().max()))
        if n.startswith("nerf.mlp_feat"):
            assert torch.equal(p0, pb), n                      # the frozen trunk stays put
    assert moved > 1e-3


@pytest.mark.parametrize("b200,match", [(dict(rng="philox"), "philox"), (dict(nan_guard=True), "nan_guard")])
def test_adaptation_host_decisions_refuse_to_be_captured(b200, match):
    opt, g, optim, static, fn = _adapt_setup(stratified=True, **b200)
    for k, v in _batch(0).items():
        static[k].copy_(v)
    with pytest.raises(RuntimeError, match=match):
        GraphedStep(fn, optim, static=static, warmup=1)
    torch.cuda.synchronize()
    fn()                                                       # eagerly the same step still runs


def test_check_range_refuses_to_be_captured():
    opt, g, optim, static, fn = _adapt_setup()
    for k, v in _batch(0).items():
        static[k].copy_(v)
    fn()                                                       # a split-mode launch: the status word exists
    probe = torch.zeros(1, device=DEV)
    with pytest.raises(RuntimeError, match="check_range"):
        with torch.cuda.graph(torch.cuda.CUDAGraph()):
            probe.add_(1.0)
            mlp_tc32.check_range(DEV)
    mlp_tc32.check_range(DEV)                                  # eagerly it reads the word


def test_captured_pretrain_fp32_tc_step_matches_the_real_reference(golden, monkeypatch):
    """The eager pattern of test_gpu_fp32_train.test_pretrain_graph_fp32_tc_step_matches_the_real_reference, captured: the view
    matrices come from the CPU (camera.HOST_MATRICES, the reference's LAPACK bits) eagerly and enter the graph as static inputs;
    the fixture's jitter is a device tensor the graph reads.  The warm-up steps move the weights; they are put back before the
    first replay, whose outputs, losses and gradients are compared."""
    from texpose_b200.model.nerf_pretrain import Graph as Pretrain
    g = golden("pretrain")
    Bp, R = g.ray_idx.shape
    opt = env_opt(H=int(g.H), W=int(g.W), sample_intvs=int(g.N), device=DEV)
    opt.nerf.rand_rays = Bp * R
    opt.loss_weight = AttrDict(render=0, mask=-1, depth=-1)
    opt.data.erode_mask_loss = False
    opt.b200 = AttrDict(TC, rng="torch")
    torch.manual_seed(0)
    gr = Pretrain(opt).to(DEV)
    initial = {k: v.detach().clone() for k, v in gr.state_dict().items()}
    optim = torch.optim.Adam(gr.nerf.parameters(), lr=1e-3, capturable=True)
    host = camera.HOST_MATRICES
    camera.HOST_MATRICES = True
    try:
        kinv, pinv = camera.view_matrices(g.pose.to(DEV), g.intr.to(DEV))
    finally:
        camera.HOST_MATRICES = host
    static = dict(ray_idx=g.ray_idx.to(DEV), image=g.image.to(DEV), obj_mask=g.obj_mask.to(DEV), depth_gt=g.depth_gt.to(DEV),
                  pose=g.pose.to(DEV), intr=g.intr.to(DEV), z_near=g.z_near.to(DEV), z_far=g.z_far.to(DEV), kinv=kinv, pinv=pinv)
    rand = g.rand.to(DEV)
    real_rand = torch.rand
    monkeypatch.setattr(torch, "rand", lambda *s, **kw: rand if tuple(s) == tuple(rand.shape) else real_rand(*s, **kw))
    idx = torch.arange(Bp, device=DEV)
    out = {}

    def fn():
        var = AttrDict(idx=idx, **{k: static[k] for k in ("ray_idx", "image", "obj_mask", "depth_gt", "pose", "intr", "z_near", "z_far")})
        var.update(gr.render(opt, var.pose, intr=var.intr, ray_idx=var.ray_idx, depth_range=(var.z_near[:, :, None], var.z_far[:, :, None]),
                             mode="train", view=(static["kinv"], static["pinv"])))
        loss = gr.compute_loss(opt, var, mode="train")
        sum(10 ** float(opt.loss_weight[k]) * loss[k] for k in loss).backward()
        out.update(var={k: var[k].detach() for k in ("rgb", "depth", "opacity")})      # no reference to this step's autograd graph
        return AttrDict({k: v.detach() for k, v in loss.items()})

    step = GraphedStep(fn, optim, static=static, warmup=2)
    monkeypatch.undo()
    with torch.no_grad():
        for k, v in gr.state_dict().items():
            v.copy_(initial[k])
    _C.launch_counts.clear()
    loss = step()
    torch.cuda.synchronize()
    assert not _C.launch_counts
    var = out["var"]
    errs = {k: (var[k].cpu() - g["o_" + k]).abs().max().item() for k in ("rgb", "depth", "opacity")}
    errs.update({"l_" + k: abs(loss[k].item() - float(g["l_" + k])) for k in ("render", "mask", "depth")})
    worst, mag, pairs = 0.0, 0.0, []
    for n, p in gr.nerf.named_parameters():
        got = p.grad if p.grad.numel() <= 2048 else p.grad[:, ::8][::8]
        worst = max(worst, (got.cpu() - g["g/" + n]).abs().max().item())
        mag = max(mag, g["g/" + n].abs().max().item())
        pairs.append((n, got, g["g/" + n]))
    _check_grads("captured pretrain Graph vs reference", pairs, REL_GRAPH, tol=TOL)
    errs["grad"] = worst
    print("captured pretrain step, fp32 on the tensor cores, first replay vs the real reference:",
          {k: f"{v:.2e}" for k, v in errs.items()}, f"gradient error relative to max |grad| {mag:.3e}: {worst / mag:.2e}")
    for k, e in errs.items():
        assert e <= TOL, (k, e)
