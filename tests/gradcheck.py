"""Test helper (not a test): gradient comparisons sized to the gradient they check.

An absolute bound such as 1e-2 says nothing about a tensor whose largest entry is 3e-3: a kernel that returned zeros for it would
pass.  `assert_grad_close` holds a gradient to two bounds relative to the reference, the largest entry error over the largest
reference entry and the error norm over the reference norm.  `assert_latent_rows` holds a per-image latent table row by row:
every row the reference touches within `rel` of its own norm, every other row exactly zero.  Both print one line per tensor in
the style of the parity tests and return the measured errors."""
import torch


def rel_errors(got, want):
    """-> (max|got - want| / max|want|, ||got - want||_2 / ||want||_2), in float64 on the CPU (inf where the reference is zero
    and the gradient is not)."""
    a, b = got.detach().cpu().double(), want.detach().cpu().double()
    d = a - b
    mag, nrm = float(b.abs().max()) if b.numel() else 0.0, float(b.norm())
    err, dn = float(d.abs().max()) if d.numel() else 0.0, float(d.norm())
    e_max = err / mag if mag > 0 else (0.0 if err == 0 else float("inf"))
    e_norm = dn / nrm if nrm > 0 else (0.0 if dn == 0 else float("inf"))
    return e_max, e_norm


def assert_grad_close(name, got, want, *, rel_max, rel_norm, tag=""):
    """max|got - want| <= rel_max * max|want| and ||got - want|| <= rel_norm * ||want||; finite, same shape."""
    assert tuple(got.shape) == tuple(want.shape), (name, tuple(got.shape), tuple(want.shape))
    assert bool(torch.isfinite(got).all()), (name, "non-finite gradient")
    e_max, e_norm = rel_errors(got, want)
    mag = float(want.detach().abs().max()) if want.numel() else 0.0
    print(f"  {tag + ' ' if tag else ''}{name:26s} |grad|max {mag:9.3e}  rel max-abs {e_max:9.3e}  rel norm {e_norm:9.3e}")
    assert e_max <= rel_max, (name, "max-abs error relative to max|want|", e_max, rel_max)
    assert e_norm <= rel_norm, (name, "error norm relative to ||want||", e_norm, rel_norm)
    return e_max, e_norm


def assert_latent_rows(got, want, rows_used, rel, name="latent", tag=""):
    """Per-image latent gradient table [n_rows, C]: every row in `rows_used` satisfies ||got_r - want_r|| <= rel * ||want_r||
    (and the reference row is non-zero); every other row of `got` is exactly zero.  Returns the worst row error."""
    a, b = got.detach().cpu().double(), want.detach().cpu().double()
    assert a.shape == b.shape and a.dim() == 2, (name, tuple(a.shape), tuple(b.shape))
    used = sorted({int(r) for r in rows_used})
    worst = 0.0
    for r in used:
        nrm = float(b[r].norm())
        assert nrm > 0, (name, r, "the reference row the batch touches is zero")
        e = float((a[r] - b[r]).norm()) / nrm
        worst = max(worst, e)
        assert e <= rel, (name, r, "row error relative to its norm", e, rel)
    others = [r for r in range(a.shape[0]) if r not in set(used)]
    if others:
        assert bool((a[others] == 0).all()), (name, "rows no image touches are not zero",
                                              [r for r in others if bool((a[r] != 0).any())])
    print(f"  {tag + ' ' if tag else ''}{name:26s} {len(used)} rows used, worst row error rel norm {worst:9.3e}, "
          f"{len(others)} untouched rows exactly zero")
    return worst


def cotangent_mask(x, keep):
    """Identity in the forward; the backward multiplies the incoming cotangent by `keep` (broadcast to x).  Used to build the
    reference gradient of a loss whose seed is zeroed on some samples (the 'contribution dropped' mutants)."""
    return _CotangentMask.apply(x, keep)


class _CotangentMask(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, keep):
        ctx.save_for_backward(keep)
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        (keep,) = ctx.saved_tensors
        return g * keep.to(g.dtype), None


def swap_rows(t, i, j):
    out = t.clone()
    out[[i, j]] = t[[j, i]]
    return out
