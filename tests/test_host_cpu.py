"""CPU-side checks: the C-ABI library builds, loads and exports every symbol include/tgpose_b200.h
declares; the host-side mirrors keep the reference's parameter names / shapes; no CPU fallback."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "tgpose_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tgp_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from tgpose_b200 import _lib
    lib = _lib.load()
    syms = _header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/tgpose_b200.h but not exported"
        assert s in _lib.SIGNATURES, f"{s} has no ctypes signature"
    assert sorted(_lib.SIGNATURES) == syms
    assert lib.tgp_version() >= 100
    assert isinstance(lib.tgp_launch_count(), int)


def test_gemm_args_struct_layout_matches_header():
    from tgpose_b200 import _lib
    # natural alignment of the C structs (LP64): tgp_out_seg 32 B, tgp_gemm_args 152 + 4*32 + 16 + (int mixed, a_kp,
    # a_group_cols, padded to 16) + the two gathered-residual index pointers
    assert ctypes.sizeof(_lib.OutSeg) == 32
    assert ctypes.sizeof(_lib.GemmArgs) == 152 + 4 * 32 + 16 + 16 + 16
    assert _lib.GemmArgs.res1_idx.offset == 152 + 4 * 32 + 16 + 16
    assert _lib.GemmArgs.res2_idx.offset == _lib.GemmArgs.res1_idx.offset + 8
    assert _lib.GemmArgs.seg.offset == 152
    assert _lib.GemmArgs.mixed.offset == 152 + 4 * 32 + 16
    assert _lib.GemmArgs.a_kp.offset == _lib.GemmArgs.mixed.offset + 4
    assert _lib.GemmArgs.a_group_cols.offset == _lib.GemmArgs.mixed.offset + 8
    assert ctypes.sizeof(_lib.ConcatSrc) == 40


def test_no_cpu_fallback():
    from tgpose_b200 import _lib, gcn3d
    n0 = _lib.launch_count()
    x = torch.rand(1, 16, 3)
    with pytest.raises(RuntimeError):
        gcn3d.get_neighbor_index(x, 4)
    layer = gcn3d.HS_layer(8, 8, 7)
    with pytest.raises(RuntimeError):
        layer(x, torch.rand(1, 16, 8), 4)
    # the heads have no eager torch branch either: train and eval mode both refuse CPU tensors
    from tgpose_b200 import posenet
    dec = posenet.FaceRecon_decoder(16) if hasattr(posenet, "FaceRecon_decoder") else None
    net = posenet.PoseNet9D()
    for mode in (True, False):
        net.train(mode)
        with pytest.raises(RuntimeError):
            net(torch.rand(2, 32, 3), torch.zeros(2, 1))
    for name in ("rot_green", "rot_red"):
        head = getattr(net, name)
        with pytest.raises(RuntimeError):
            head.train()(torch.rand(2, posenet.FEAT_C, 32))
    del dec
    # every refusal happens before a launch: a kernel handed host addresses faults the CUDA context after the call returned
    assert _lib.launch_count() == n0


def test_state_dict_names_and_shapes():
    """SURVEY 8b: parameter names/shapes are API (checkpoints, trainer/RL_TDA.py:64-97)."""
    from tgpose_b200.face_enc import Face_Enc
    torch.manual_seed(0)
    sd = Face_Enc().state_dict()
    assert tuple(sd["conv_0.directions"].shape) == (3, 896)
    assert tuple(sd["conv_0.STE_layer.weight"].shape) == (128, 3, 1)
    assert tuple(sd["conv_0.conv2.weight"].shape) == (128, 256, 1)
    for name, (cin, cout) in {"conv_1": (128, 128), "conv_2": (128, 256), "conv_3": (256, 256), "conv_4": (256, 512)}.items():
        assert tuple(sd[f"{name}.weights"].shape) == (cin, 8 * cout)
        assert tuple(sd[f"{name}.bias"].shape) == (8 * cout,)
        assert tuple(sd[f"{name}.directions"].shape) == (3, 7 * cout)
        assert tuple(sd[f"{name}.STE_layer.weight"].shape) == (cout, cin, 1)
        assert tuple(sd[f"{name}.conv2.weight"].shape) == (cout, 2 * cout, 1)
    assert "bn1.running_mean" in sd and "proj_layer.0.weight" in sd


def test_pack_layer_column_order():
    """the slab column permutation (cgroup, s, c4) used by the projection GEMM."""
    from tgpose_b200.autograd import _pack_layer
    S, C, cin = 7, 8, 5
    w = torch.arange(cin * (S + 1) * C, dtype=torch.float32).reshape(cin, (S + 1) * C)
    b = torch.arange((S + 1) * C, dtype=torch.float32)
    ste = torch.arange(C * cin, dtype=torch.float32).reshape(C, cin, 1) + 1000
    wcat, bcat, _ = _pack_layer(w, b, ste, S, C)
    assert wcat.shape == (cin, (S + 2) * C) and bcat.shape == ((S + 2) * C,)
    SC = S * C                                                     # packed order: [slab | centre | STE]
    assert torch.equal(wcat[:, SC:SC + C], w[:, :C]) and torch.equal(bcat[SC:SC + C], b[:C])
    for cg in range(C // 4):
        for s in range(S):
            for c4 in range(4):
                col = cg * S * 4 + s * 4 + c4
                assert torch.equal(wcat[:, col], w[:, C + s * C + cg * 4 + c4])
                assert bcat[col] == b[C + s * C + cg * 4 + c4]
    assert torch.equal(wcat[:, (S + 1) * C:], ste[:, :, 0].t())
    assert (bcat[(S + 1) * C:] == 0).all()


def test_pool_consumes_cpu_rng_like_reference():
    """Pool_layer draws torch.randperm(N) from the global CPU generator (gcn3d.py:242)."""
    torch.manual_seed(7)
    a = torch.randperm(128)[:32]
    torch.manual_seed(7)
    b = torch.randperm(128)
    c = torch.randperm(32)
    torch.manual_seed(7)
    assert torch.equal(torch.randperm(128)[:32], a)
    assert torch.equal(torch.randperm(32), c)
    g = np.load(os.path.join(ROOT, "tests", "golden", "convs.npz"))
    assert np.array_equal(b.numpy().astype(np.int16), g["p_perm"])


# ----------------------------------------------------------------------------------------- optimiser host logic
def test_ranger_struct_layouts_match_header():
    from tgpose_b200 import _lib, ranger
    # tgp_ranger_hyper: 7 floats, 2 ints, 2 floats; tgp_ranger_row: long long + 4 ints
    assert ctypes.sizeof(_lib.RangerHyper) == 48 and _lib.RangerHyper.gc_on_update.offset == 44
    assert _lib.RangerHyper.neg_step.offset == 24 and _lib.RangerHyper.rectified.offset == 28
    assert _lib.RangerHyper.max_norm.offset == 40
    rec = ranger._pack_rows(np.asarray([[64, 5, 1, 2]], np.int64))
    assert rec.dtype.itemsize == 24 and rec.tobytes()[:8] == (64).to_bytes(8, "little")
    assert int.from_bytes(rec.tobytes()[8:12], "little") == 5 and int.from_bytes(rec.tobytes()[16:20], "little") == 2


def test_ranger_row_table():
    """centralised tensors: one row per dim-0 slice (ranger2020.py:31-41); the rest: <= 4096-element pieces; every
    tensor starts on a 128-byte boundary; rows are disjoint and cover every element exactly once."""
    from tgpose_b200.ranger import ALIGN, ROW_PIECE, build_row_table
    shapes = [(128, 3, 1), (3, 896), (10001,), (), (5,), (2, 3, 5, 1), (0,)]
    offsets, total, rows = build_row_table(shapes)
    assert all(o % ALIGN == 0 for o in offsets) and total % ALIGN == 0
    cover = np.zeros(total, np.int32)
    for off, ln, gc, t in rows:
        cover[off:off + ln] += 1
        numel = int(np.prod(shapes[t])) if shapes[t] else 1
        assert offsets[t] <= off and off + ln <= offsets[t] + numel
        assert gc == (1 if len(shapes[t]) > 1 else 0)
        assert ln == (numel // shapes[t][0] if gc else min(ROW_PIECE, offsets[t] + numel - off))
    for t, s in enumerate(shapes):
        numel = int(np.prod(s)) if s else 1
        assert (cover[offsets[t]:offsets[t] + numel] == 1).all()
    assert cover.sum() == sum(int(np.prod(s)) if s else 1 for s in shapes)
    assert (rows[:, 3] == np.sort(rows[:, 3])).all()            # parameter order -> contiguous row range per group
    # gc_conv_only: only tensors with more than 3 dims are centralised; use_gc=False: none
    _, _, r2 = build_row_table(shapes, gc_conv_only=True)
    assert set(r2[r2[:, 2] == 1, 3]) == {5}
    _, _, r3 = build_row_table(shapes, use_gc=False)
    assert not r3[:, 2].any()


def test_radam_scalars_match_oracle_and_cross_threshold():
    from oracle import oracle as orc
    from tgpose_b200.ranger import radam_scalars
    seen = set()
    for step in range(1, 40):
        a, b = radam_scalars(step, 0.95, 0.999, 5), orc.radam_scalars(step, 0.95, 0.999, 5)
        assert a[0] == b[0] and abs(a[1] - b[1]) <= 1e-12 * abs(b[1])
        seen.add(a[0])
    assert seen == {False, True}
    assert radam_scalars(5, 0.95, 0.999, 5)[0] is False and radam_scalars(6, 0.95, 0.999, 5)[0] is True


def test_ranger_has_no_cpu_path():
    from tgpose_b200.ranger import Ranger
    with pytest.raises(RuntimeError):
        Ranger([torch.nn.Parameter(torch.zeros(4, 4))])


def test_training_glue_matches_reference():
    """the RL_TDA loss glue and lr schedule restated in train_step.py against the reference's own functions
    (losses/consistency_loss.py, tools/torch_utils/solver/lr_scheduler.py; tests/golden/train_glue.npz)."""
    from tgpose_b200 import train_step as ts
    from util import golden
    g = golden("train_glue")
    x1 = torch.from_numpy(g["x1"]).requires_grad_(True)
    pc_re = torch.from_numpy(g["pc_re"]).requires_grad_(True)
    l1 = ts.feat_consistency_loss(x1, torch.from_numpy(g["x2"]), float(g["feat_consist_w"]))
    l2 = ts.prop_sym_matching_loss(torch.from_numpy(g["pc"]), pc_re, torch.from_numpy(g["gt_R"]), torch.from_numpy(g["gt_t"]),
                                   torch.from_numpy(g["sym"]))
    (l1 + l2).backward()
    assert abs(float(l1) - float(g["feat_loss"])) <= 1e-5 * abs(float(g["feat_loss"]))
    assert abs(float(l2) - float(g["sym_loss"])) <= 1e-5 * abs(float(g["sym_loss"]))
    assert np.allclose(x1.grad.numpy(), g["g_x1"], rtol=1e-4, atol=1e-8)
    assert np.allclose(pc_re.grad.numpy(), g["g_pc_re"], rtol=1e-4, atol=1e-9)
    wi, wf, ap = g["lr_args"]
    for it, f in zip(g["lr_iters"], g["lr_factor"]):
        mine = ts.flat_and_anneal_factor(int(it), int(g["lr_total"]), warmup_iters=int(wi), warmup_factor=float(wf), anneal_point=float(ap))
        assert abs(mine - f) <= 1e-12 + 1e-9 * abs(f), (it, mine, f)
    # the scheduler object applies the factor of iteration `it` after `it` step() calls, like LambdaLR
    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=2.0)
    sch = ts.FlatAndAnneal(opt, int(g["lr_total"]), warmup_iters=int(wi), warmup_factor=float(wf), anneal_point=float(ap))
    assert abs(opt.param_groups[0]["lr"] - 2.0 * g["lr_factor"][0]) < 1e-12
    for _ in range(10):
        sch.step()
    assert abs(opt.param_groups[0]["lr"] - 2.0 * g["lr_factor"][list(g["lr_iters"]).index(10)]) < 1e-12
