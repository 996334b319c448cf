"""VERDICT r1 next-1 (ii) and (iv): the fused tcgen05 forward + backward at the REAL C3 configuration against the CPU oracle
(every head dW / db, both latent-embedding gradients), and data-parallel equivalence: two shards of the batch, exchanged over
the peer-window kernel, against the mean of the oracle's per-shard gradients (SURVEY 8e).  Tolerance: north-star 1e-2
max-abs for gradients of the reference's mean-normalised losses with the bf16 MLP path -- no relative carve-outs."""
import pytest
import torch

from tests import c3_problem as C3
from texpose_b200 import _C, parallel

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-2


def _report(tag, got, want):
    worst = 0.0
    for k in want:
        a, b = got[k].cpu(), want[k]
        err, mag = float((a - b).abs().max()), float(b.abs().max())
        worst = max(worst, err)
        print(f"  {tag} {k:26s} |grad|max {mag:9.3e}  max-abs err {err:9.3e}")
    return worst


@pytest.mark.timeout(900)
def test_c3_fused_backward_vs_oracle():
    inp = C3.inputs()
    opt, g = C3.graph(DEV)
    _C.launch_counts.clear()
    got, rand, loss, (zn, zf) = C3.cuda_step(opt, g, inp, slice(0, C3.B), DEV, seed=21)
    assert _C.launch_counts.get("tp_tc_heads_backward", 0) == 1          # the fused tcgen05 backward, not the staged kernels
    assert _C.launch_counts.get("tp_linear_backward_weight", 0) == 0     # ... and nothing on the fp32 SIMT path
    want, ref_loss, (ozn, ozf) = C3.oracle_step(g, inp, slice(0, C3.B), rand)
    assert torch.equal(zn, ozn) and torch.equal(zf, ozf)
    for k in ("render", "uncert", "trans_reg", "all"):
        assert abs(loss[k] - ref_loss[k]) <= 1e-2 * max(1.0, abs(ref_loss[k])), (k, loss[k], ref_loss[k])
    worst = _report("C3", got, want)
    print(f"C3 (16 x 256 x 128) bf16 gradients vs oracle: worst max-abs error {worst:.3e}")
    for k in want:
        assert got[k].shape == want[k].shape
        assert float((got[k].cpu() - want[k]).abs().max()) <= TOL, k
    # per-image latent gradients: every one of the 8 rows received the sum of its two images
    assert (want["latent_vars_light.weight"].abs().sum(dim=1) > 0).all()


@pytest.mark.timeout(900)
def test_data_parallel_two_shards_equal_mean_of_oracle_shard_gradients():
    """Rank r trains on images [8r, 8r+8); the gradients meet in the peer-window exchange (both ranks on this device, each on
    its own stream, the kernels waiting for each other as ranks on two GPUs do).  Every rank must hold the same bits, and they
    must equal the mean of the oracle's per-shard gradients (per-shard losses are means, SURVEY 8e)."""
    inp = C3.inputs()
    opt, g = C3.graph(DEV)
    world, half = 2, C3.B // 2
    names = [k for k, _ in C3.named_trainables(g)]
    ours, oracle = [], []
    for r in range(world):
        sl = slice(r * half, (r + 1) * half)
        got, rand, _, _ = C3.cuda_step(opt, g, inp, sl, DEV, seed=30 + r)
        ours.append(torch.cat([got[k].reshape(-1) for k in names]))
        want, _, _ = C3.oracle_step(g, inp, sl, rand)
        oracle.append(torch.cat([want[k].reshape(-1) for k in names]))
    n = ours[0].numel()
    wins = [parallel.PeerWindow(n, torch.device(DEV)) for _ in range(world)]
    try:
        outs = [torch.empty((n + 3) // 4 * 4, device=DEV) for _ in range(world)]
        streams = [torch.cuda.Stream(DEV) for _ in range(world)]
        for r in range(world):
            wins[r].buffers[1].copy_(ours[r])
        torch.cuda.synchronize()
        for r in (1, 0):
            parallel.peer_allreduce_mean([w.ptr for w in wins], r, n, 1, outs[r], grid_ctas=16, timeout_ms=5000, stream=streams[r])
        torch.cuda.synchronize()
        assert all(w.status() == 0 for w in wins)
        assert torch.equal(outs[0][:n], outs[1][:n])
        mean_ref = (oracle[0] + oracle[1]) / world
        off = 0
        for k, p in C3.named_trainables(g):
            m = p.numel()
            err = float((outs[0][off:off + m].cpu() - mean_ref[off:off + m]).abs().max())
            print(f"  DP {k:26s} max-abs err vs mean of oracle shard grads {err:9.3e}")
            assert err <= TOL, k
            off += m
    finally:
        for w in wins:
            w.close()
