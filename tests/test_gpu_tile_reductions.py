"""Direct tests of the small-gradient reductions of the tensor-core backward on tile images built on the host, against float64
sums: tp_tc_image_ray_sums (per-ray sums: layer 0's view columns), tp_tc_images_colsum (bias gradients), tp_tc_thin_dw (thin
dW: output layers, xyz columns), tp_thin_colsum (output biases), tp_tc_dw_gemm + tp_reduce_partials (256 x 256 dW) and
tp_group_colsum (per-image latent rows), single-pass and split (bf16 hi / lo image pairs 2k, 2k + 1 of logical slot k).

Tile-image layout (csrc/mlp_tc_bwd.cu, image_ray_sums_kernel): element (s, c) of slot k of an image set with n_slots slots is the
bf16 at byte ((s >> 7) * n_slots + k) * 65536 + (c >> 3) * 2048 + (s & 127) * 16 + (c & 7) * 2; rows s >= S of the last tile are
zero, as the producers leave them.  Inputs are bf16-exact multiples of 1/64 (lo parts of 2^-9 / 64), so the float64 reference is
exact and the bound covers only the kernels' fp32 accumulation: 2e-6 * sum of |terms| per output.  Every launch is repeated and
must return the same bits.

The last test runs the staged forward with save and both dX chains at S % 128 != 0 and decodes what they wrote: every dz row
>= S of the last tile is exactly zero (images_colsum and the dW GEMM sum all 128 rows of it), and the saved trunk feature is the
float64 oracle's."""
import pytest
import torch

from oracle import texpose_oracle as O
from texpose_b200 import _C, mlp_tc_bwd, ops, synth
from texpose_b200.config import AttrDict, adapt_gan_opt
from texpose_b200.layers.nerf_static_transient_light import NeRF

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SIZES = [1, 127, 128, 129, 1776, 7200]
EPS = 2e-6          # fp32 accumulation, relative to the sum of |terms| of each output


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _big_S():
    """More tiles than tp_tc_thin_dw's 4 x SM-count blocks, so each block walks more than one tile; not a multiple of 128."""
    return (8 * _sms() + 3) * 128 + 77


def _values(shape, g, scale=1.0):
    """bf16-exact values k / 64 * scale, |k| <= 64."""
    return (torch.randint(-64, 65, shape, generator=g).double() / 64 * scale)


def pack(x):
    """x [n_slots, S, 256] (bf16-exact) -> tile images (uint8 bytes) of n_slots slots; padded rows zero."""
    n_slots, S, _ = x.shape
    n_tiles = (S + 127) // 128
    xp = torch.zeros(n_slots, n_tiles * 128, 256, dtype=torch.bfloat16)
    xp[:, :S] = x.to(torch.bfloat16)
    assert torch.equal(xp[:, :S].double(), x)
    img = xp.view(n_slots, n_tiles, 128, 32, 8).permute(1, 0, 3, 2, 4).contiguous()
    return img.view(torch.uint8).reshape(-1).to(DEV)


def unpack(images, n_slots, S):
    """Inverse of pack on the first ceil(S / 128) tiles of an image buffer -> [n_slots, n_tiles * 128, 256] float64 (padded rows
    included)."""
    n_tiles = (S + 127) // 128
    raw = images[:n_tiles * n_slots * 65536].cpu().view(torch.bfloat16).view(n_tiles, n_slots, 32, 128, 8)
    return raw.permute(1, 0, 3, 2, 4).reshape(n_slots, n_tiles * 128, 256).double()


def _slots(S, n_logical, split, g):
    """Logical slot values [n_logical, S, 256] and the packed images: split -> hi at 2k, lo (2^-9 of the scale) at 2k + 1."""
    hi = _values((n_logical, S, 256), g)
    if not split:
        return hi, pack(hi), [hi]
    lo = _values((n_logical, S, 256), g, scale=2.0 ** -9)
    both = torch.stack([hi, lo], dim=1).reshape(2 * n_logical, S, 256)
    return hi + lo, pack(both), [hi, lo]


def _close(got, ref, bound, what):
    got = got.detach().cpu().double()
    err = (got - ref).abs()
    assert got.shape == ref.shape, (what, tuple(got.shape), tuple(ref.shape))
    bad = err > bound
    assert not bool(bad.any()), (what, float(err.max()), float(bound.max()), int(bad.sum()))


def _twice(fn):
    a, b = fn(), fn()
    assert torch.equal(a, b), "a second call gave different bits"
    return a


@pytest.mark.parametrize("split", [False, True], ids=["single", "split"])
@pytest.mark.parametrize("N", [1, 8, 24, 37, 128, 200])
@pytest.mark.parametrize("S", SIZES)
def test_image_ray_sums(S, N, split):
    g = torch.Generator().manual_seed(S * 1000 + N)
    x, images, _ = _slots(S, 3, split, g)
    rays = (S + N - 1) // N
    got = _twice(lambda: mlp_tc_bwd.image_ray_sums(images, 1, 3, S, N, split=split))
    xp = torch.zeros(rays * N, 256, dtype=torch.float64)
    xp[:S] = x[1]
    ref = xp.view(rays, N, 256).sum(1)
    _close(got, ref, EPS * xp.abs().view(rays, N, 256).sum(1), "image_ray_sums")


@pytest.mark.parametrize("split", [False, True], ids=["single", "split"])
@pytest.mark.parametrize("S", SIZES + ["big"])
def test_images_colsum(S, split):
    S = _big_S() if S == "big" else S
    g = torch.Generator().manual_seed(S + 7)
    x, images, _ = _slots(S, 4, split, g)
    sel = [2, 0, 3]
    got = _twice(lambda: mlp_tc_bwd.images_colsum(images, 4, S, sel, split=split))
    _close(got, x[sel].sum(1), EPS * x[sel].abs().sum(1), "images_colsum")


@pytest.mark.parametrize("split", [False, True], ids=["single", "split"])
@pytest.mark.parametrize("M", [1, 3, 5])
@pytest.mark.parametrize("S", SIZES + ["big"])
def test_thin_dw(S, M, split):
    S = _big_S() if S == "big" else S
    g = torch.Generator().manual_seed(S * 10 + M)
    x, images, _ = _slots(S, 3, split, g)
    thin = _values((S, M), g)
    got = _twice(lambda: mlp_tc_bwd.thin_dw(thin.float().to(DEV), images, 2, 3, S, split=split))
    _close(got, thin.t() @ x[2], EPS * (thin.abs().t() @ x[2].abs()), "thin_dw")


@pytest.mark.parametrize("C", range(1, 9))
@pytest.mark.parametrize("S", SIZES + ["big"])
def test_thin_colsum(S, C):
    S = _big_S() if S == "big" else S
    g = torch.Generator().manual_seed(S + C)
    x = _values((S, C), g)
    got = _twice(lambda: mlp_tc_bwd.thin_colsum(x.float().to(DEV), S))
    _close(got, x.sum(0), EPS * x.abs().sum(0), "thin_colsum")


@pytest.mark.parametrize("split", [False, True], ids=["single", "split"])
@pytest.mark.parametrize("S", SIZES)
def test_dw_gemm(S, split):
    """Several jobs on distinct a / b slots in one launch, split over tile ranges, reduced with tp_reduce_partials; split: the
    three terms hi.hi + hi.lo + lo.hi (lo.lo, ~2^-18 of the product, is dropped by design)."""
    g = torch.Generator().manual_seed(S + 99)
    a, a_img, a_parts = _slots(S, 3, split, g)
    b, b_img, b_parts = _slots(S, 4, split, g)
    pairs = [(0, 1), (2, 0), (1, 3), (2, 2)]
    got = _twice(lambda: mlp_tc_bwd.dw_gemm(a_img, 3, b_img, 4, pairs, S, split=split))
    for j, (i, k) in enumerate(pairs):
        if split:
            (ah, al), (bh, bl) = [p[i] for p in a_parts], [p[k] for p in b_parts]
            terms = [(ah, bh), (ah, bl), (al, bh)]
        else:
            terms = [(a[i], b[k])]
        ref = sum(p.t() @ q for p, q in terms)
        _close(got[j], ref, EPS * sum(p.abs().t() @ q.abs() for p, q in terms), f"dw_gemm job {j}")


@pytest.mark.parametrize("rows,group,cols", [(150, 50, 256), (256, 4, 256), (2400, 1200, 256), (3000, 600, 48),
                                             (1001, 300, 256), (7, 1, 16)])
def test_group_colsum(rows, group, cols):
    """Per-image sums of per-ray rows (the latent gradients' g_img); groups longer than 512 rows are split into slices."""
    g = torch.Generator().manual_seed(rows + group)
    y = _values((rows, cols + 5), g)
    dY = y.float().to(DEV)[:, :cols]                       # row stride != cols
    got = _twice(lambda: ops.group_colsum(dY, rows, group))
    G_ = (rows + group - 1) // group
    yp = torch.zeros(G_ * group, cols, dtype=torch.float64)
    yp[:rows] = y[:, :cols]
    _close(got, yp.view(G_, group, cols).sum(1), EPS * yp.abs().view(G_, group, cols).sum(1), "group_colsum")


def test_packer_matches_the_documented_byte_layout():
    g = torch.Generator().manual_seed(1)
    S, n_slots = 300, 3
    x = _values((n_slots, S, 256), g)
    raw = pack(x).cpu()
    for k, s, c in [(0, 0, 0), (1, 5, 9), (2, 299, 255), (1, 128, 7), (2, 200, 130)]:
        off = ((s >> 7) * n_slots + k) * 65536 + (c >> 3) * 2048 + (s & 127) * 16 + (c & 7) * 2
        assert float(raw[off:off + 2].view(torch.bfloat16)[0]) == float(x[k, s, c])
    assert torch.equal(unpack(pack(x), n_slots, S)[:, :S], x)


# ---------------------------------------------------------------------------------------------- what the producers leave there

@pytest.mark.parametrize("engine", ["staged_bf16", "split"])
def test_chain_leaves_padded_dz_rows_zero_and_saves_the_oracle_feature(engine, monkeypatch):
    """Staged forward with save, then the heads' dX chains (tp_tc_chain_backward / _split) at S = 720 (80 rows in the last tile).
    The dz images and the saved activations are captured where the dW GEMM reads them."""
    B, R, N = 30, 2, 12
    S = B * R * N
    assert S % 128 != 0
    opt = adapt_gan_opt(device=DEV)
    opt.b200 = AttrDict(mlp="bf16") if engine == "staged_bf16" else AttrDict(mlp="fp32", fp32_engine="tc")
    torch.manual_seed(0)
    m = NeRF(opt).to(DEV)
    gen = torch.Generator().manual_seed(12)
    with torch.no_grad():
        for lin in list(m.mlp_feat) + list(m.mlp_rgb) + list(m.mlp_trans):
            lin.bias.copy_(torch.randn(lin.bias.shape, generator=gen).mul_(0.2).to(DEV))
    g = torch.Generator().manual_seed(4)
    center = torch.randn(B, R, 3, generator=g) * 0.02 + torch.tensor([0.3, 0.2, -0.8])
    ray = torch.randn(B, R, 3, generator=g) * 0.1 + torch.tensor([0.0, 0.0, 1.0])
    depth = (torch.rand(B, R, N, 1, generator=g) + torch.arange(N)[None, None, :, None]) / N * 1.2 + 0.2
    lt, ll = [t.to(DEV).requires_grad_(True) for t in synth.latents(B)]
    seen = []
    real = mlp_tc_bwd.dw_gemm

    def spy(a_images, a_nslots, b_images, b_nslots, pairs, S_, split=False):
        if not seen:
            seen.append((a_images, a_nslots, b_images, b_nslots, S_, split))
        return real(a_images, a_nslots, b_images, b_nslots, pairs, S_, split=split)

    monkeypatch.setattr(mlp_tc_bwd, "dw_gemm", spy)
    _C.launch_counts.clear()
    out = m.forward_samples(opt, center.to(DEV), ray.to(DEV), depth.to(DEV), lt, ll, mode="train")
    (out[0].square().mean() + out[1][..., 1].mean() + out[2].mean()).backward()
    torch.cuda.synchronize()
    counts = dict(_C.launch_counts)
    if engine == "staged_bf16":
        assert counts.get("tp_tc32_forward") == 1 and counts.get("tp_tc_chain_backward") == 2, counts
    else:
        assert counts.get("tp_tc32_forward_split_save") == 1 and counts.get("tp_tc_chain_backward_split") == 2, counts
    assert len(seen) == 1
    dz, n_dz, images, n_save, S_seen, split = seen[0]
    assert S_seen == S and split == (engine == "split")
    parts = 2 if split else 1
    # every dz image (hi and lo) of the last tile: rows >= S exactly zero, and the chain wrote non-zero rows below S
    dzi = unpack(dz, parts * n_dz, S)
    assert bool((dzi[:, S:] == 0).all()), [(k, int((dzi[k, S:] != 0).any(dim=1).sum())) for k in range(dzi.shape[0])]
    assert bool((dzi[::parts, :S] != 0).any(dim=2).any(dim=1).all())
    # the saved feature (slot 0) against the oracle's trunk in float64 (encoding as the reference rounds it)
    pts = O.points_from_depth(center, ray, depth)                  # fp32, as the kernels form the points
    feat_l = [(l.weight.detach().cpu().double(), l.bias.detach().cpu().double()) for l in m.mlp_feat]
    enc = torch.cat([pts, O.positional_encoding(pts, 10)], dim=-1).double()      # the reference's fp32 encoding
    feat, _ = O._trunk(enc, feat_l, (4,))
    feat = feat.reshape(S, 256)
    img = unpack(images, parts * n_save, S)
    saved = img[0, :S] + (img[1, :S] if split else 0)
    err = float((saved - feat).abs().max())
    print(f"{engine}: saved trunk feature vs float64 oracle: max-abs {err:.3e} (max |feature| {float(feat.abs().max()):.3e})")
    if split:
        assert err <= 1e-4, err                                    # the <= 1e-4 mode's contract
    else:                                                          # bf16 trunk and bf16 image: two bf16 ulps at max|feature|
        ulp = 2.0 ** (torch.floor(torch.log2(feat.abs().max())).item() - 7)
        assert err <= 2 * ulp, (err, ulp)
