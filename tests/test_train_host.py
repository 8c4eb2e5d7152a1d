"""Host-side logic of the training engine that needs no GPU: the zeroed-accumulator pool, the operand-split preconditions, the
arithmetic claim behind the 3xTF32 mode (aero_b200/train_engine.py, include/aero_b200.h aero_split_tf32) and FusedAdam's
param-group options (aero_b200/optim.py)."""
import numpy as np
import pytest
import torch

from aero_b200 import Aero, aero_kwargs, cabi
from aero_b200.engine import tf32_round
from aero_b200.optim import FusedAdam
from aero_b200.train_engine import TrainEngine


def _engine():
    torch.manual_seed(0)
    return TrainEngine(Aero(**aero_kwargs("aero_4-16_512_256")).train())


def test_zero_pool_hands_out_disjoint_aligned_zeroed_views():
    e = _engine()
    e._reset()
    a = e._new(5, zero=True, dtype=torch.float64)
    b = e._new(3, 7, zero=True)
    c = e._new(130, zero=True)
    d = e._new(9, zero=True, dtype=torch.float64)
    for t in (a, b, c, d):
        assert float(t.abs().sum()) == 0.0 and t.is_contiguous() and t.data_ptr() % 16 == 0
    a.fill_(1.0); b.fill_(2.0); c.fill_(3.0); d.fill_(4.0)                 # no carve-out overlaps another
    assert float(a.sum()) == 5 and float(b.sum()) == 42 and float(c.sum()) == 390 and float(d.sum()) == 36
    assert a.untyped_storage().data_ptr() == d.untyped_storage().data_ptr()            # same pool per dtype
    assert b.untyped_storage().data_ptr() == c.untyped_storage().data_ptr() != a.untyped_storage().data_ptr()
    big = e._new(1 << 19, zero=True)                                       # beyond the per-request cap: a plain allocation
    assert big.untyped_storage().data_ptr() != b.untyped_storage().data_ptr() and float(big.abs().sum()) == 0.0
    e._reset()                                                             # a new pass starts from a fresh pool
    assert float(e._new(5, zero=True, dtype=torch.float64).sum()) == 0.0


def test_operand_split_preconditions():
    p = cabi.TapGemmParams()
    p.B, p.F_in, p.T_in = 2, 3, 10
    C_ = 8
    sb, sf, st = 3 * 10 * C_, 10 * C_, C_
    t = torch.zeros(2 * 3 * 10 * C_)
    assert TrainEngine._splittable(t, C_, sb, sf, st, p)
    assert TrainEngine._splittable(None, 0, 0, 0, 0, p)
    assert not TrainEngine._splittable(t[:-4], C_, sb, sf, st, p)                       # strides reach past the buffer
    assert not TrainEngine._splittable(t.double(), C_, sb, sf, st, p)
    wide = torch.zeros(2 * 3 * 10 * 16)
    assert TrainEngine._splittable(wide, C_, 3 * 10 * 16, 10 * 16, 16, p)               # a channel slice of a wider tensor
    assert not TrainEngine._splittable(wide[1:], C_, 3 * 10 * 16, 10 * 16, 16, p)       # misaligned base (and too short)


def test_three_tf32_products_reproduce_the_fp32_product():
    """x = hi + lo, hi = TF32(x), lo = TF32(x - hi): hi*hi' + hi*lo' + lo*hi' with exact products (11-bit x 11-bit significands) and fp32
    accumulation differs from the fp64 dot product by ~1e-7 relative; one plain TF32 product by ~3e-4 (the two training modes' op-level
    accuracy: tests/test_gpu_train_tc.py measures 1e-6 .. 1e-5 and 1e-3 on the device, where the accumulation is the tensor core's)."""
    g = torch.Generator().manual_seed(3)
    a, b = torch.randn(64, 2048, generator=g), torch.randn(2048, 48, generator=g)
    a_hi, b_hi = tf32_round(a), tf32_round(b)
    a_lo, b_lo = tf32_round(a - a_hi), tf32_round(b - b_hi)
    assert float((a_hi + a_lo - a).abs().max()) <= 2.0 ** -21 * float(a.abs().max())   # the split loses at most 2^-22 |x| per operand
    ref = a.double() @ b.double()
    one = (a_hi.double() @ b_hi.double())
    three = (a_lo.double() @ b_hi.double() + a_hi.double() @ b_lo.double() + a_hi.double() @ b_hi.double())
    e1 = float((one - ref).norm() / ref.norm())
    e3 = float((three - ref).norm() / ref.norm())
    assert 5e-5 < e1 < 1e-3, e1
    assert e3 < 5e-7, e3
    # device-side rounding (cvt.rna.tf32: ties away) == the host helper used for the goldens
    x = torch.tensor([1.0 + 2.0 ** -11, 1.0 + 2.0 ** -11 + 2.0 ** -20, -(1.0 + 2.0 ** -11)])
    assert np.allclose(tf32_round(x).numpy(), [1.0 + 2.0 ** -10, 1.0 + 2.0 ** -10, -(1.0 + 2.0 ** -10)])


def test_fused_adam_state_dict_steps_torch_adam():
    """A checkpoint of the fast trainer's optimizer resumes under torch.optim.Adam: its param groups carry every option
    torch.optim.Adam.step reads (no KeyError on the first step).  The options FusedAdam does not implement are refused."""
    p = torch.ones(3, requires_grad=True)
    sd = FusedAdam([p], lr=1e-2).state_dict()
    assert {"weight_decay": 0, "amsgrad": False, "maximize": False}.items() <= sd["param_groups"][0].items()
    q = torch.ones(3, requires_grad=True)
    ref = torch.optim.Adam([q])
    ref.load_state_dict(sd)
    q.grad = torch.tensor([1.0, -2.0, 0.0])
    ref.step()
    assert torch.allclose(q.detach(), torch.tensor([0.99, 1.01, 1.0]))
    for bad in (dict(weight_decay=1e-4), dict(amsgrad=True), dict(maximize=True)):
        with pytest.raises(ValueError):
            FusedAdam([p], **bad)
