"""-m gpu: the torch.library custom ops (aero_b200/ops.py, SURVEY.md section 8b) on CUDA tensors, eagerly and inside
``torch.compile(fullgraph=True)`` graphs, and the multi-GPU product API (``aero_b200.parallel.ShardedAero``) over NCCL
when the machine has two GPUs."""
import os
import subprocess
import sys

import pytest
import torch

from util import SEED, rel_l2, trained_like_, white_noise

from aero_b200 import Aero, aero_kwargs

pytestmark = pytest.mark.gpu


def build(exp):
    torch.manual_seed(SEED)
    m = Aero(**aero_kwargs(exp)).eval()
    m.load_state_dict(trained_like_(m.state_dict()))
    return m


def test_custom_ops_on_cuda_and_under_torch_compile():
    from aero_b200 import ops, spec
    x = white_noise((2, 1, 8000)).cuda()
    z = torch.ops.aero_b200.stft(x, 512, 64, 512)
    want = torch.view_as_real(torch.stft(x.reshape(-1, 8000), 512, 64, 512, window=torch.hann_window(512).cuda(), normalized=True,
                                         return_complex=True)).reshape(2, 1, 257, 126, 2)
    assert z.shape == want.shape and rel_l2(z.cpu(), want.cpu()) < 1e-5
    y = torch.ops.aero_b200.istft(z, 64, 512, 8000)
    assert y.shape == (2, 1, 8000) and rel_l2(y.cpu(), x.cpu()) < 1e-5           # STFT -> iSTFT round trip (north_star: 1e-5)

    m = build("aero_4-16_512_256").cuda()
    h = ops.register_model(m)
    a = white_noise((2, 1, 8000), seed=3).cuda()
    direct = m(a).clone()
    via_op = torch.ops.aero_b200.generator_forward(a, h)
    assert rel_l2(via_op.cpu(), direct.cpu()) < 2e-4

    @torch.compile(fullgraph=True)
    def pipeline(sig, hr):
        pr = torch.ops.aero_b200.generator_forward(sig * 1.0, h)
        zs = torch.ops.aero_b200.stft(pr, 512, 64, 512)
        zh = torch.ops.aero_b200.stft(hr, 512, 64, 512)
        return pr, (zs - zh).abs().mean()
    hr = white_noise((2, 1, 32000), seed=4).cuda()
    pr, dist_ = pipeline(a, hr)
    assert rel_l2(pr.cpu(), direct.cpu()) < 2e-4 and torch.isfinite(dist_)
    zs = torch.view_as_real(spec.spectro(direct, 512, 64, win_length=512))
    zh = torch.view_as_real(spec.spectro(hr, 512, 64, win_length=512))
    assert abs(float(dist_) - float((zs - zh).abs().mean())) < 1e-3 * float(dist_)
    with pytest.raises(Exception):
        torch.ops.aero_b200.stft(x.cpu(), 512, 64, 512)                           # no CPU kernel is registered


def test_model_on_a_non_current_device_and_variable_lengths_stay_bounded():
    """ADVICE round 1: launches must target the model's device, not the caller's current device; a loop over many
    distinct clip lengths (reference test.py / evaluate.py) must not grow the workspace cache without bound."""
    m = build("aero_4-16_512_256").cuda()
    eng = m._engine()
    ref = m(white_noise((1, 1, 6000)).cuda()).clone()
    if torch.cuda.device_count() >= 2:
        m1 = build("aero_4-16_512_256").to("cuda:1")
        with torch.cuda.device(0):
            out1 = m1(white_noise((1, 1, 6000)).to("cuda:1"))
        assert out1.device.index == 1 and rel_l2(out1.cpu(), ref.cpu()) < 2e-4
    torch.cuda.synchronize()
    for i, n in enumerate(range(4000, 4000 + 40 * 64, 64)):
        m(white_noise((1, 1, n), seed=i).cuda())
    torch.cuda.synchronize()
    per_set = [sum(t.numel() * t.element_size() for t in s.values()) for s in eng._bufsets.values()]
    assert len(eng._bufsets) <= eng.max_shape_sets and sum(per_set) <= eng.max_shape_sets * max(per_set)
    assert len(eng._graphs) <= eng.max_shape_sets
    assert rel_l2(m(white_noise((1, 1, 6000)).cuda()).cpu(), ref.cpu()) < 2e-4


_NCCL_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["AERO_ROOT"]); sys.path.insert(0, os.path.join(os.environ["AERO_ROOT"], "tests"))
import torch, torch.distributed as dist
from util import SEED, rel_l2, trained_like_, white_noise
from aero_b200 import Aero, aero_kwargs
from aero_b200.parallel import ShardedAero
rank = int(os.environ["RANK"]); torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
torch.manual_seed(SEED)
m = Aero(**aero_kwargs("aero_4-16_512_256")).eval(); m.load_state_dict(trained_like_(m.state_dict())); m = m.cuda()
mix = white_noise((5, 1, 6000))
full = ShardedAero(m).forward(mix, gather=True)
single = m(mix.cuda())
err = rel_l2(full.cpu(), single.cpu())
assert full.shape == single.shape and err < 2e-4, err
if rank == 0: print("SHARDED_OK", err)
dist.destroy_process_group()
'''


def test_sharded_aero_over_nccl_two_gpus(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    script = tmp_path / "worker.py"
    script.write_text(_NCCL_WORKER)
    env = dict(os.environ, AERO_ROOT=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29533", str(script)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "SHARDED_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_custom_op_autograd_stft_istft():
    """torch.ops.aero_b200.stft / .istft are differentiable: their backward formulas (adjoint kernels) against autograd through
    torch.stft / torch.istft in fp64."""
    from aero_b200 import ops  # noqa: F401
    x = white_noise((2, 3000), seed=1)
    xd = x.double().requires_grad_(True)
    w = torch.hann_window(400).double()
    zt = torch.view_as_real(torch.stft(xd, 512, 100, 400, w, normalized=True, return_complex=True))
    R = white_noise(tuple(zt.shape), seed=2).double()
    (zt * R).sum().backward()
    xg = x.cuda().requires_grad_(True)
    z = torch.ops.aero_b200.stft(xg, 512, 100, 400)
    (z * R.float().cuda()).sum().backward()
    torch.cuda.synchronize()
    assert rel_l2(z.detach().cpu(), zt.detach()) < 1e-5 and rel_l2(xg.grad.cpu(), xd.grad) < 1e-5

    zin = white_noise((2, 257, 31, 2), seed=3)
    zin[:, 0, :, 1] = 0
    zin[:, 256, :, 1] = 0
    zd = zin.double().requires_grad_(True)
    yt = torch.istft(torch.view_as_complex(zd), 512, 100, 400, w, normalized=True, length=2900)
    Ry = white_noise(tuple(yt.shape), seed=4).double()
    (yt * Ry).sum().backward()
    zg = zin.cuda().requires_grad_(True)
    y = torch.ops.aero_b200.istft(zg, 100, 400, 2900)
    (y * Ry.float().cuda()).sum().backward()
    torch.cuda.synchronize()
    gref = zd.grad.clone()
    assert rel_l2(y.detach().cpu(), yt.detach()) < 1e-5
    # (imaginary parts of DC / Nyquist do not influence the C2R transform: both sides give zero there up to round-off)
    assert rel_l2(zg.grad.cpu(), gref) < 1e-5
