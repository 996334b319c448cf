"""Host side of the fp32-parity training step on the tensor cores (opt.b200.fp32_engine = 'tc'), without a GPU: the split chunk and
stage tables of the plain model's chain, the save-buffer layout, and the argument checks of the new entry points.  The pointers are
dummies that are never dereferenced: every call either fails an argument check (which comes before the device check) or passes
S = 0 samples, so on a machine with a B200 as well nothing is launched."""
import torch

from texpose_b200 import _C, mlp_tc_plain
from texpose_b200.config import AttrDict, env_opt
from texpose_b200.layers._mlp import MLPConfig

P = 0x10000      # non-null, 16-byte aligned; never dereferenced
ERR_BAD_ARG, ERR_BAD_SHAPE, ERR_ALIGN, ERR_ARCH = -1, -2, -3, -4


def _plain(nf=8, skip=(4,)):
    cfg = MLPConfig(L_3D=10, L_view=4, skip=skip, view_dep=True, n_feat=nf, n_rgb=2, n_trans=0)
    feat = []
    for li in range(nf):
        k = 63 if li == 0 else 256 + (63 if li in skip else 0)
        feat.append((torch.zeros(257 if li == nf - 1 else 256, k), torch.zeros(257 if li == nf - 1 else 256)))
    rgb = [(torch.zeros(128, 256 + 27 + 3), torch.zeros(128)), (torch.zeros(3, 128), torch.zeros(3))]
    return cfg, feat, mlp_tc_plain._padded_head(rgb)


def test_split_chunk_table_has_sixteen_k16_slots_per_layer():
    for nf, skip in ((8, (4,)), (4, (2,)), (2, ())):
        cfg, feat, rgb = _plain(nf, skip)
        rows0, stages0 = mlp_tc_plain._bwd_chunks(cfg, feat, rgb)
        rows, stages = mlp_tc_plain._bwd_chunks(cfg, feat, rgb, split=True)
        assert len(stages) == len(stages0) == nf + 1 and len(rows) == 2 + 16 * nf
        for s, s0 in zip(stages, stages0):      # same stage list except the chunk numbering and count
            assert s[0] == s0[0] and s[4:] == s0[4:]
            assert s[3] == (0 if s0[3] == 0 else 16)
        chunks = []
        for s in stages:
            if s[0] >= 0:
                chunks.append(s[1])
            chunks += list(range(s[2], s[2] + s[3]))
        assert chunks == list(range(len(rows)))          # every chunk streamed once, in stage order
        for s in stages:
            if s[3]:
                ks = [rows[c][4] - rows[s[2]][4] for c in range(s[2], s[2] + 16)]
                assert ks == list(range(0, 256, 16))     # K = 16 steps over the layer's 256 input rows
                assert all(rows[c][5] == 16 and rows[c][6] == 256 and rows[c][9] == 1 for c in range(s[2], s[2] + 16))
        thin = [rows[s[1]] for s in stages if s[0] >= 0]
        assert [r[5] for r in thin] == [3, 1]            # dz_rgb x W_out (3 rows), dz_sigma x W_last row 0


def test_split_save_layout_sizes():
    lib = _C.load()
    assert lib.tp_tc32_split_save_bytes(129, 3) == 2 * 3 * (2 * 65536 + 4096)      # hi / lo images + one bitmask per slot
    assert lib.tp_tc32_split_save_bytes(0, 3) == 0
    assert lib.tp_tc32_split_save_bytes(128, 1) == 2 * 65536 + 4096


def test_split_entry_points_reject_bad_arguments_before_the_device():
    lib = _C.load()
    st = torch.tensor([[0, 0, 0, 0, 0, 0], [-1, 0, 1, 16, 1, 1]], dtype=torch.int32)

    def chain(rows, n_chunks=17, thin1=None, n_saved=2, n_out=2, packed=P, cols0=3):
        t = torch.tensor(rows, dtype=torch.int32)
        return lib.tp_tc_chain_backward_split(P, cols0, thin1, 1, 0, packed, n_chunks, t.data_ptr(), len(rows), P, n_saved, P,
                                              n_out, None)

    ok = [[0, 0, 0, 0, 0, 0], [-1, 0, 1, 16, 1, 1]]
    assert chain(ok) in (0, ERR_ARCH)                                    # passes every argument check (S = 0: no launch)
    assert chain([[0, 0, 0, 0, 0, 0], [-1, 0, 1, 8, 1, 1]]) == ERR_BAD_SHAPE     # K = 32 chunk count of the bf16 chain
    assert chain([[-1, 0, 1, 16, 0, 0]]) == ERR_BAD_ARG                  # the first stage reads A tiles nobody wrote
    assert chain([[1, 0, 0, 0, 0, 0]]) == ERR_BAD_ARG                    # thin operand 1 is absent
    assert chain(ok, n_chunks=16) == ERR_BAD_ARG                         # chunks beyond the image
    assert chain([[0, 0, 0, 0, 2, 0]]) == ERR_BAD_ARG                    # mask slot beyond the saved slots
    assert chain([[0, 0, 0, 0, 0, 2]]) == ERR_BAD_ARG                    # dz slot beyond the output
    assert chain(ok, cols0=9) == ERR_BAD_SHAPE                           # thin operand wider than a K = 16 step
    assert chain(ok, packed=P + 4) == ERR_ALIGN
    assert lib.tp_tc_chain_backward_split(None, 3, None, 0, 0, P, 17, st.data_ptr(), 2, P, 2, P, 2, None) == ERR_BAD_ARG
    assert lib.tp_tc_pack_weights_split(None, 1, P, None) == ERR_BAD_ARG
    assert lib.tp_tc_pack_weights_split(P, 0, P, None) == ERR_BAD_SHAPE
    assert lib.tp_tc_pack_weights_split(P, 1, P + 8, None) == ERR_ALIGN

    def fwd(save=P, n_save=2, enc_slot=1):
        rows = torch.tensor([[0, 4, 0, 0, 0, 8, 0], [16, 0, 1, 0, 0, 1, -1]], dtype=torch.int32)
        return lib.tp_tc32_forward_split_save(P, P, P, 0, 32, 32, P, 5, rows.data_ptr(), 2, P, None, None, P, P, P, P, 1 << 30,
                                              save, n_save, enc_slot, None)

    assert fwd(save=None) == ERR_BAD_ARG                                 # a training launch must have a save buffer
    assert fwd(n_save=0) == ERR_BAD_SHAPE
    assert fwd(save=P + 4) == ERR_ALIGN
    # tp_tc32_forward keeps rejecting a save with precision 0: the split save has its own entry point
    rows = torch.tensor([[0, 4, 0, 0, 0, 8, 0], [16, 0, 1, 0, 0, 1, -1]], dtype=torch.int32)
    assert lib.tp_tc32_forward(P, P, P, 0, 32, 32, P, 5, rows.data_ptr(), 2, P, None, None, P, P, P, P, 1 << 30, 0, P, 2, 1,
                               None) == ERR_BAD_ARG


def test_engine_option_routes_only_fp32_tc_training():
    from texpose_b200.layers.nerf import NeRF
    m = NeRF(env_opt())
    for mlp, engine, want in (("fp32", None, False), ("fp32", "simt", False), ("fp32", "auto", False), ("fp32", "tc", True),
                              ("bf16", None, True), ("bf16", "simt", True)):
        opt = env_opt()
        opt.b200 = AttrDict(mlp=mlp, fp32_engine=engine)
        with torch.enable_grad():
            assert m.trains_on_tensor_cores(opt) is want, (mlp, engine)
        with torch.no_grad():
            assert m.trains_on_tensor_cores(opt) is False
