"""GPU: tgp_chamfer_fwd / tgp_chamfer_bwd against the arithmetic of the reference's own kernel (losses/chamfer3D/
chamfer3D.cu).  Distances and indices must be BIT-EQUAL on tie-free inputs: the arithmetic form (difference, then
fma(dz,dz, fma(dx,dx, dy*dy))) and the strict '<' of chamfer3D.cu:32-40 are part of the contract.

Two comparisons: the CPU oracle (oracle.c orc_chamfer_nn / orc_chamfer_bwd, the same arithmetic and tie rule, always
run) and -- when build() found the unmodified reference sources and compiled them into oracle/_ref/chamfer3D -- the
reference's kernel itself on the same inputs (SURVEY 8c: "GPU oracle and kernel to beat")."""
import numpy as np
import pytest
import torch

from oracle import build_ref
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    """the reference's pybind module `chamfer_3D`, or None when oracle/_ref/chamfer3D was not built (the repository
    does not ship the reference's sources)."""
    return build_ref.load_chamfer()


def _alloc(B, n, m, dev):
    return (torch.zeros(B, n, device=dev), torch.zeros(B, m, device=dev),
            torch.zeros(B, n, dtype=torch.int32, device=dev), torch.zeros(B, m, dtype=torch.int32, device=dev))


def _assert_equal_to_oracle(a, b, o):
    o1, o2, oi1, oi2 = orc.chamfer_forward(a.cpu().numpy(), b.cpu().numpy())
    for name, x, y in zip(("dist1", "dist2", "idx1", "idx2"), (o1, o2, oi1, oi2), o):
        y = y.cpu().numpy()
        assert np.array_equal(x, y), f"{name}: {int((x != y).sum())} of {x.size} differ from the oracle"


# (4,100,200): the reference's own unit-test shape (losses/metrics/CD/unit_test.py:14-35), all in the ragged tail path of
# chamfer3D.cu:88-131; 1028 x 1024: BASELINE configs[2]; 2500 x 3000: more than one 512-candidate batch + a ragged tail,
# more than one of our 2048-candidate tiles; (3,1,1), (2,5,70): degenerate sizes
@pytest.mark.parametrize("B,n,m", [(4, 100, 200), (8, 1028, 1024), (2, 2500, 3000), (3, 1, 1), (2, 5, 70), (1, 513, 2049)])
def test_forward_bit_equal_to_reference_kernel(ref, B, n, m):
    from tgpose_b200 import ops
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(B * 1000 + n + m)
    a = (torch.rand(B, n, 3, generator=g) - 0.5).to(dev)
    b = (torch.rand(B, m, 3, generator=g) - 0.5).to(dev)
    o = _alloc(B, n, m, dev)
    ops.chamfer_forward(a, b, *o)
    torch.cuda.synchronize()
    if ref is not None:
        r = _alloc(B, n, m, dev)
        assert ref.forward(a, b, *r) == 1
        torch.cuda.synchronize()
        for name, x, y in zip(("dist1", "dist2", "idx1", "idx2"), r, o):
            assert torch.equal(x, y), f"{name}: {int((x != y).sum())} of {x.numel()} differ from the reference kernel"
    _assert_equal_to_oracle(a, b, o)


def test_forward_ties_take_the_lowest_index_like_the_reference(ref):
    """duplicated candidates: exact distance ties; strict '<' keeps the first (chamfer3D.cu:36)."""
    from tgpose_b200 import ops
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(11)
    a = torch.rand(2, 300, 3, generator=g)
    b = torch.rand(2, 150, 3, generator=g)
    b = torch.cat([b, b, b[:, :40]], dim=1)           # every candidate appears 2-3 times
    a, b = a.to(dev), b.to(dev)
    o = _alloc(2, 300, 340, dev)
    ops.chamfer_forward(a, b, *o)
    if ref is not None:
        r = _alloc(2, 300, 340, dev)
        ref.forward(a, b, *r)
        for x, y in zip(r, o):
            assert torch.equal(x, y)
    _assert_equal_to_oracle(a, b, o)
    assert int(o[2].max()) < 150                      # always the first copy


def test_backward_matches_reference_kernel(ref):
    from tgpose_b200 import ops
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(5)
    B, n, m = 4, 257, 300
    a, b = torch.rand(B, n, 3, generator=g).to(dev), torch.rand(B, m, 3, generator=g).to(dev)
    gd1, gd2 = torch.randn(B, n, generator=g).to(dev), torch.randn(B, m, generator=g).to(dev)
    o = _alloc(B, n, m, dev)
    ops.chamfer_forward(a, b, *o)
    og1, og2 = torch.zeros(B, n, 3, device=dev), torch.zeros(B, m, 3, device=dev)
    ops.chamfer_backward(a, b, gd1, gd2, o[2], o[3], og1, og2)
    torch.cuda.synchronize()
    expected = [orc.chamfer_backward(a.cpu().numpy(), b.cpu().numpy(), gd1.cpu().numpy(), gd2.cpu().numpy(),
                                     o[2].cpu().numpy(), o[3].cpu().numpy())]
    if ref is not None:
        rg1, rg2 = torch.zeros(B, n, 3, device=dev), torch.zeros(B, m, 3, device=dev)
        assert ref.backward(a, b, rg1, rg2, gd1, gd2, o[2], o[3]) == 1
        torch.cuda.synchronize()
        expected.append((rg1.cpu().numpy(), rg2.cpu().numpy()))
    # the scattered terms are accumulated with fp32 atomics (order not fixed): rel 1e-5 of the gradient scale
    for e1, e2 in expected:
        for x, y in ((e1, og1), (e2, og2)):
            scale = float(np.abs(x).max())
            assert float(np.abs(x - y.cpu().numpy()).max()) <= 1e-5 * scale
