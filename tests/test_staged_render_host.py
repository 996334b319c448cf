"""Host logic of the one-launch render (no GPU): which launch render_rays takes (lock-step bf16 / staged in either arithmetic /
refused) from `opt` and the layer shapes, and FrameGather's check of the keys a graph can produce."""
import pytest
import torch

from texpose_b200 import parallel
from texpose_b200.config import AttrDict, adapt_gan_opt, env_opt
from texpose_b200.layers.nerf import NeRF as PlainNeRF
from texpose_b200.layers.nerf_static_transient_light import NeRF as StlNeRF
from texpose_b200.model.nerf_pretrain import Graph as PretrainGraph

SMALL_TRUNK = dict(layers_feat=[None] + [256] * 6, skip=[2], layers_rgb=[None, 256, 256, 3], layers_trans=[None, 256, 256, 5])


def _opt(make, mlp, **arch):
    opt = make(H=8, W=8, sample_intvs=64)
    for k, v in arch.items():
        opt.arch[k] = v
    opt.b200 = AttrDict(mlp=mlp)
    return opt


@torch.no_grad()
def test_plain_model_routes():
    opt = _opt(env_opt, "fp32")
    m = PlainNeRF(opt)
    assert m.render_precision(opt) == 0
    assert m.render_precision(_opt(env_opt, "bf16")) == 1
    assert m.render_precision(_opt(env_opt, "auto")) == 1            # the bf16 kernel implements the 8 x 256 trunk
    opt5 = _opt(env_opt, "auto", layers_feat=[None] + [256] * 6, skip=[2])
    assert PlainNeRF(opt5).render_precision(opt5) == 0               # ... but not this one: auto means fp32 there
    for change in (dict(setbg_opaque=True), dict(sample_intvs=48)):
        o = _opt(env_opt, "fp32")
        for k, v in change.items():
            o.nerf[k] = v
        with pytest.raises(NotImplementedError):
            m.render_precision(o)
    o = _opt(env_opt, "fp32")
    o.camera.ndc = True
    with pytest.raises(NotImplementedError, match="ndc"):
        m.render_precision(o)
    o = _opt(env_opt, "fp32")
    o.nerf.depth.param = "inverse"
    with pytest.raises(NotImplementedError, match="metric"):
        m.render_precision(o)
    o = _opt(env_opt, "fp32")
    o.b200.fp32_engine = "simt"
    with pytest.raises(NotImplementedError, match="simt"):
        m.render_precision(o)
    o = _opt(env_opt, "fp32", layers_rgb=[None, 512, 3])
    with pytest.raises(NotImplementedError, match="256"):
        PlainNeRF(o).render_precision(o)


def test_plain_model_refuses_a_gradient_recording_render():
    opt = _opt(env_opt, "fp32")
    with torch.enable_grad(), pytest.raises(NotImplementedError, match="no_grad"):
        PlainNeRF(opt).render_precision(opt)


@torch.no_grad()
def test_static_transient_light_routes():
    opt = _opt(adapt_gan_opt, "bf16")
    m = StlNeRF(opt)
    assert m._lockstep_render_applies(opt, m._config(opt, "val"))          # the yaml's architecture in bf16: lock-step launch
    o = _opt(adapt_gan_opt, "auto")
    assert m._lockstep_render_applies(o, m._config(o, "val"))
    o = _opt(adapt_gan_opt, "fp32")
    assert not m._lockstep_render_applies(o, m._config(o, "val")) and m.render_precision(o) == 0
    o = _opt(adapt_gan_opt, "bf16", **SMALL_TRUNK)
    ms = StlNeRF(o)
    assert not ms._lockstep_render_applies(o, ms._config(o, "val")) and ms.render_precision(o) == 1
    o = _opt(adapt_gan_opt, "fp32", **SMALL_TRUNK)
    assert ms.render_precision(o) == 0
    o = _opt(adapt_gan_opt, "fp32")
    o.b200.static_only = True
    with pytest.raises(NotImplementedError, match="static-only"):
        m.render_precision(o, m._config(o, "eval"))
    o = _opt(adapt_gan_opt, "fp32")
    o.nerf.sample_intvs = 96
    with pytest.raises(NotImplementedError, match="samples per ray"):
        m.render_precision(o)
    o = _opt(adapt_gan_opt, "fp32", layers_rgb=[None, 128, 3])
    with pytest.raises(NotImplementedError, match="256-wide"):
        StlNeRF(o).render_precision(o)


def test_frame_gather_checks_the_keys_of_the_graph():
    """A FrameGather of the adaptation engine's keys cannot gather a pre-training frame (it has no transient outputs): ValueError
    before anything is launched."""
    assert parallel.PRETRAIN_KEYS == ("rgb", "depth", "opacity")
    assert set(parallel.PRETRAIN_KEYS) <= set(PretrainGraph.RENDER_KEYS)
    g = PretrainGraph(_opt(env_opt, "fp32"))
    fg = parallel.FrameGather.__new__(parallel.FrameGather)      # (the window needs a GPU; render checks the keys first)
    pose = torch.zeros(1, 3, 4)
    fg.keys = parallel.PER_RAY_KEYS
    with pytest.raises(ValueError, match="rgb_static"):
        fg.render(g, None, pose, None, None)
    fg.keys = parallel.PRETRAIN_KEYS
    with pytest.raises(ValueError, match="alpha_static"):
        fg.render(g, None, pose, None, None, local_keys=("alpha_static",))
