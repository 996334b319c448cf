"""The C-ABI library loads on a CPU-only box and exports every symbol include/texpose_b200.h declares."""
import ctypes
import os

from texpose_b200 import _C


def test_header_symbols_exported():
    _C.build()
    protos = _C.declared_prototypes()
    names = [p[1] for p in protos]
    assert len(names) >= 25 and len(set(names)) == len(names)
    lib = ctypes.CDLL(_C.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"


def test_version_and_prototypes():
    lib = _C.load()
    assert lib.tp_version() == 100
    for ret, name, args in _C.declared_prototypes():
        fn = getattr(lib, name)
        assert len(fn.argtypes) == len(args)


def test_no_torch_types_in_abi():
    import re
    text = re.sub(r"/\*.*?\*/", " ", open(_C.HEADER).read(), flags=re.S)     # declarations only
    assert "torch" not in text and "at::" not in text and "Tensor" not in text


def test_sources_are_sm100a_only():
    assert "arch=compute_100a,code=sm_100a" in " ".join(_C.NVCC_FLAGS)
    assert os.path.exists(_C.LIB_PATH)


def test_host_side_helpers_without_gpu():
    """Pure host arithmetic of the C-ABI (no kernel launch): workspace sizes and the fused-backward applicability rule."""
    lib = _C.load()
    assert lib.tp_patch_loss_workspace() >= 8 and lib.tp_eval_epilogue_workspace(3) == 3 * 64
    assert lib.tp_tc_dz_bytes(129) == 2 * 6 * 65536
    assert lib.tp_tc_save_bytes(129) == 2 * (7 * 65536 + 4 * 4096)        # tile images + ReLU bitmasks, whole super-tiles
    # one tile per CTA (few tiles): a 128-sample range may touch at most 4 images -> images of >= 64 samples
    assert lib.tp_tc_heads_backward_supported(16 * 256 * 128, 256 * 128) == 1
    assert lib.tp_tc_heads_backward_supported(64 * 4 * 8, 32) == 0
    assert lib.tp_tc_heads_backward_supported(0, 128) == 0


def test_forward_rejects_unknown_flags_before_the_device():
    """tp_tc_nerf_stl_forward takes only flags bit 17 (static only); any other bit is a bad argument, reported before the
    device check.  S = 0, so no argument combination can launch anything."""
    lib = _C.load()
    p = 0x10000      # non-null, 16-byte aligned; never dereferenced

    def fwd(flags):
        return lib.tp_tc_nerf_stl_forward(p, p, p, 0, 32, 32, p, p, p, p, p, p, p, p, 1 << 30, None, flags, None)

    for flags in (0, 1 << 17):
        assert fwd(flags) in (0, -4)      # the dummy arguments pass every argument check (-4: no sm_100 device)
    for flags in (2, 0x20, 0x40):
        assert fwd(flags) == -1


def test_peer_window_layout_helpers_without_gpu():
    """Pure host arithmetic of the gradient-exchange window (csrc/peer.cu): [1 KB header | buffer 0 | buffer 1], buffers
    padded to 256 B; argument errors are reported before any CUDA call."""
    import ctypes
    lib = _C.load()
    for n in (0, 1, 63, 64, 65, 421385):
        cap = lib.tp_peer_capacity_bytes(n)
        assert cap % 256 == 0 and cap >= 4 * n and cap < 4 * n + 256
        assert lib.tp_peer_window_bytes(n) == 1024 + 2 * cap
        assert lib.tp_peer_data_offset(n, 0) == 1024 and lib.tp_peer_data_offset(n, 1) == 1024 + cap
        assert lib.tp_peer_data_offset(n, 2) == 1024
    out = ctypes.c_void_p()
    assert lib.tp_peer_window_create(16, ctypes.byref(out)) == -1            # smaller than the header
    assert lib.tp_peer_window_export(None, None) == -1 and lib.tp_peer_window_import(None, None) == -1
    assert lib.tp_peer_allreduce_mean(None, 2, 0, 8, 1, None, 0, 0, None) == -1
    assert lib.tp_peer_window_destroy(None) == 0 and lib.tp_peer_window_release(None) == 0


def test_flex_patch_sampler_matches_oracle_on_cpu():
    """FlexPatchSampler is host logic (three torch.rand draws): identical to the oracle restatement for the same RNG state,
    and the coordinates stay inside [-1, 1] (tools/patch_sampler.py:100-110)."""
    import torch
    from oracle import texpose_oracle as O
    from texpose_b200.tools.patch_sampler import FlexPatchSampler
    for seed, (B, P) in enumerate([(1, 2), (7, 16), (3, 5)]):
        torch.manual_seed(seed)
        want = O.flex_patch_coords(B, P)
        torch.manual_seed(seed)
        got = FlexPatchSampler()(nbatch=B, patch_size=P, device="cpu")
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
        assert got[0].shape == (B, P, P, 2) and got[0].abs().max() <= 1.0


def test_patch_sampler_anneals_like_the_reference():
    """ADVICE r1 (medium): Graph builds FlexPatchSampler(scale_anneal=0.0002) (model/nerf_adapt_st_gan.py:424) and the engine
    feeds it `iterations` (:185): min_scale = min(0.8, max(0.25, exp(-it * 2e-4))) (tools/patch_sampler.py:85-89)."""
    import math
    import torch
    from texpose_b200.config import adapt_gan_opt
    from texpose_b200.model.nerf_adapt_st_gan import Graph
    opt = adapt_gan_opt(H=32, W=32)
    g = Graph(opt, n_train_images=2)
    ps = g.patch_sampler
    assert ps.scale_anneal == 0.0002 and ps.min_scale == 0.25 and ps.max_scale == 1.0
    for it, want in ((0, 0.8), (1000, 0.8), (2000, math.exp(-0.4)), (5000, math.exp(-1.0)), (100000, 0.25)):
        ps.iterations = it
        torch.manual_seed(3)
        coords, scales = ps(nbatch=64, patch_size=4, device="cpu")
        assert abs(ps.scales_curr[0] - want) < 1e-12 and ps.scales_curr[1] == 1.0
        assert float(scales.min()) >= want - 1e-6 and float(scales.max()) <= 1.0
        assert coords.abs().max() <= 1.0 + 1e-6


def test_product_never_imports_the_oracle_and_refuses_cpu_tensors():
    """The oracle is test infrastructure: nothing under texpose_b200/ may import it or the reference copy (a product path routed
    through the CPU restatement would void every parity claim), and the tensor-level wrappers reject CPU tensors instead of falling
    back.  bench.py may touch it only in its CPU / eager-baseline legs (functions named below)."""
    import ast
    import os
    import pytest
    import torch
    from texpose_b200 import ops
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "texpose_b200")
    for base, _, files in os.walk(pkg):
        for f in files:
            if not f.endswith(".py"):
                continue
            tree = ast.parse(open(os.path.join(base, f)).read())
            for node in ast.walk(tree):
                names = []
                if isinstance(node, ast.Import):
                    names = [a.name for a in node.names]
                elif isinstance(node, ast.ImportFrom):
                    names = [node.module or ""]
                for n in names:
                    assert n.split(".")[0] not in ("oracle", "baseline"), (f, n)
            assert "/root/reference" not in open(os.path.join(base, f)).read(), f
    # bench.py: every oracle import sits inside one of the baseline helpers, none at module level or in the timed GPU path
    tree = ast.parse(open(os.path.join(root, "bench.py")).read())
    allowed = {"frame_inputs", "reference_graph", "cpu_reference_step", "eager_gpu_sample"}      # the reference arm / cpu_baseline / eager "before" legs
    for fn in [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef)]:
        inner = {m for sub in ast.walk(fn) if isinstance(sub, ast.FunctionDef) and sub is not fn for m in ast.walk(sub)}
        for node in ast.walk(fn):
            if node in inner:
                continue
            if isinstance(node, ast.ImportFrom) and (node.module or "").split(".")[0] == "oracle":
                assert fn.name in allowed, f"bench.py: {fn.name} imports the oracle"
    for node in tree.body:
        if isinstance(node, (ast.Import, ast.ImportFrom)):
            mod = node.module if isinstance(node, ast.ImportFrom) else node.names[0].name
            assert (mod or "").split(".")[0] != "oracle"
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.gather_rows(torch.zeros(1, 4, 3), torch.zeros(1, 2, dtype=torch.long))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.sample_depth(torch.zeros(1, 4), torch.ones(1, 4), 8, stratified=False)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No CPU path behind the drop-ins: without the built .so every entry point raises (and says how to build it), nothing falls
    back to torch or to the oracle."""
    import pytest
    monkeypatch.setattr(_C, "_lib", None)
    monkeypatch.setattr(_C, "LIB_PATH", str(tmp_path / "libtexpose_b200.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _C.load()
    with pytest.raises(RuntimeError, match="g.build"):
        _C.call("tp_version")
    monkeypatch.undo()
    assert _C.load().tp_version() == 100
