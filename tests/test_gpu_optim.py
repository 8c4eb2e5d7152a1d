"""-m gpu: aero_b200.optim.FusedAdam (csrc/train.cu adam_kernel, one launch per group) over many steps against
torch.optim.Adam(foreach=False) on fp64 CPU copies of the same parameters fed the same gradients; the optimizer state carried
from step to step (moments, per-parameter step counts, the cached device chunk tables, state_dict in both directions); and
what an optimizer step must make visible to the inference engine's caches (packed weights, CUDA graphs) and to the trainers.

Parameters are compared by their accumulated displacement p_k - p_0, not by p_k: next to p_0 an Adam update is ~1e-3 relative,
so a bar on p_k could not see a wrong update."""
import copy

import numpy as np
import pytest
import torch

from util import SEED, rel_l2, trained_like_, white_noise

from aero_b200 import Aero, aero_kwargs, cabi
from aero_b200.optim import _CHUNK, FusedAdam

pytestmark = pytest.mark.gpu
DEV = "cuda"
# Adam's fp32 arithmetic is a few roundings per element and step, ~1e-7 relative against fp64.  The displacement also carries
# the rounding of p itself to fp32 after every step, up to ulp(p)/2 per element: at |p| ~ 0.01 (a typical weight) that is
# ~1e-9, which next to the update of a small lr with an eps-dominated or scaled-down gradient (lr * 0.01 ~ 1e-6) would be ~1e-3
# relative and would hide the kernel.  So the parameters start at 1e-3 (1e-5 for the eps-dominated ones), where that term is
# < 2e-6 relative per tensor in every case below.
TOL = 1e-5


def v_tol(beta2):
    """Bar for exp_avg_sq.  aero_adam_step takes the betas as fp32, so the kernel's (1 - beta2) is off by
    |fl32(beta2) - beta2| / (1 - beta2) relative -- 1.3e-5 at 0.999, 1.7e-4 at 0.9999 -- and exp_avg_sq carries that factor.
    Its bias correction is computed from the same fp32 beta2, so the update does not: within one optimizer the displacement is
    held to TOL.  Where moments cross between FusedAdam and torch.optim.Adam (load_state_dict), one side divides the other's
    exp_avg_sq by its own bias correction, and the update moves by up to half that factor: those displacements get this bar."""
    return TOL + abs(float(np.float32(beta2)) - beta2) / (1 - beta2)


def _grad(kind, shape, k, seed):
    """Gradient of step k (1-based) for one parameter, fp32 on the CPU."""
    g = torch.Generator().manual_seed(seed * 1000 + k)
    if kind == "unit":
        return torch.randn(shape, generator=g)
    if kind == "tiny":          # eps-dominated: |g| ~ 1e-9 against eps = 1e-8
        return 1e-9 * torch.randn(shape, generator=g)
    if kind == "big":
        return 1e3 * torch.randn(shape, generator=g)
    if kind == "zero":
        return torch.zeros(shape)
    if kind == "flip":          # same magnitudes, sign alternating every step
        return (-1.0) ** k * torch.randn(shape, generator=torch.Generator().manual_seed(seed)).abs()
    if kind == "stop":          # O(1) for three steps, then exact zeros (the moments decay, the parameter still moves)
        return torch.randn(shape, generator=g) if k <= 3 else torch.zeros(shape)
    raise ValueError(kind)


class Pair:
    """FusedAdam on fp32 CUDA parameters and the fp64 CPU reference on clones of them, stepped with the same gradients.

    groups: list of (dict(lr, betas, eps), [(numel, kind), ...]).  zeroing: "none" -- zero_grad() (set_to_none) and fresh .grad
    tensors every step, so the chunk table is rebuilt; "flat" -- every .grad is a view of one persistent buffer written in place,
    as aero_b200.trainer.GeneratorTrainer does."""

    def __init__(self, groups, zeroing="none", grad_scale=1.0, seed=0):
        self.zeroing, self.grad_scale = zeroing, grad_scale
        self.ps, self.qs, self.kinds, self.beta2 = [], [], [], []
        fused_groups, ref_groups = [], []
        i = 0
        for hyper, specs in groups:
            pg, qg = [], []
            for numel, kind in specs:
                scale = 1e-5 if kind == "tiny" else 1e-3
                p0 = scale * torch.randn(numel, generator=torch.Generator().manual_seed(seed + 7919 * i))
                p = p0.to(DEV, copy=True).requires_grad_(True)
                q = p0.double().requires_grad_(True)
                pg.append(p)
                qg.append(q)
                self.kinds.append((kind, numel, seed + i))
                self.beta2.append(hyper["betas"][1])
                i += 1
            self.ps += pg
            self.qs += qg
            fused_groups.append(dict(hyper, params=pg))
            ref_groups.append(dict(hyper, params=qg))
        self.p0 = [p.detach().cpu().double() for p in self.ps]
        self.q0 = [q.detach().clone() for q in self.qs]
        self.opt = FusedAdam(fused_groups)
        self.ref = torch.optim.Adam(ref_groups, foreach=False)
        if zeroing == "flat":
            self.flat = torch.zeros(sum(p.numel() for p in self.ps), device=DEV)
            off = 0
            for p in self.ps:
                p.grad = self.flat[off:off + p.numel()].view(p.shape)
                off += p.numel()
        self.k = 0

    def set_grads(self, skip=()):
        self.k += 1
        if self.zeroing == "none":
            self.opt.zero_grad()
        else:
            self.flat.zero_()
        for j, (p, q, (kind, numel, seed)) in enumerate(zip(self.ps, self.qs, self.kinds)):
            if j in skip:
                assert self.zeroing == "none"
                p.grad = q.grad = None
                continue
            g = _grad(kind, (numel,), self.k, seed)
            if self.zeroing == "none":
                p.grad = g.to(DEV)
            else:
                p.grad.copy_(g)
            q.grad = g.double() * self.grad_scale

    def step(self, skip=()):
        self.set_grads(skip)
        self.opt.step(grad_scale=self.grad_scale)
        self.ref.step()

    def check(self, opt=None, crossed=False):
        """Compare the state of `opt` (default: the FusedAdam) with the reference: per parameter rel_l2 of exp_avg, exp_avg_sq
        and the displacement, each against its bar (see v_tol; `crossed`: the moments came from the other kind of optimizer).
        Returns the worst of each."""
        opt = opt or self.opt
        worst = [0.0, 0.0, 0.0]
        torch.cuda.synchronize()
        for p, q, p0, q0, b2 in zip(self.ps, self.qs, self.p0, self.q0, self.beta2):
            st, rs = opt.state.get(p), self.ref.state.get(q)
            assert bool(st) == bool(rs)
            if not st:
                assert torch.equal(p.detach().cpu().double(), p0)
                continue
            assert int(st["step"]) == int(rs["step"])
            es = (rel_l2(st["exp_avg"].cpu(), rs["exp_avg"]), rel_l2(st["exp_avg_sq"].cpu(), rs["exp_avg_sq"]),
                  rel_l2(p.detach().cpu().double() - p0, q.detach() - q0))
            bars = (TOL, v_tol(b2), v_tol(b2) if crossed else TOL)
            assert all(e < t for e, t in zip(es, bars)), (int(rs["step"]), p.numel(), es, bars)
            worst = [max(a, b) for a, b in zip(worst, es)]
        return worst


def _run(pair, steps, skip_at=None, each=None):
    worst = [0.0, 0.0, 0.0]
    for k in range(1, steps + 1):
        if each is not None:
            each(pair, k)
        pair.step(skip=(skip_at or {}).get(k, ()))
        worst = [max(a, b) for a, b in zip(worst, pair.check())]
    return worst


EDGE_SIZES = [1, 3, 255, _CHUNK - 1, _CHUNK, _CHUNK + 1, 3 * _CHUNK + 17, 0]
KINDS = ["unit", "tiny", "big", "zero", "flip", "stop"]


@pytest.mark.parametrize("zeroing", ["none", "flat"])
@pytest.mark.parametrize("grad_scale", [1.0, 0.5, 0.125])
def test_adam_matches_fp64_adam_over_ten_steps(zeroing, grad_scale):
    """Sizes around the 65536-element chunk of the device table, an empty parameter (also alone in a group: no launch, step
    counted as torch does), three groups with different lr / betas / eps and a scheduler-like lr change, gradients in every
    regime, both ways of zeroing gradients.  An fp32 emulation of the kernel's arithmetic gives, worst per tensor over all ten
    steps and all cases, 1e-6 (exp_avg), 1.7e-4 (exp_avg_sq, the fp32 beta2 = 0.9999 of one group; see v_tol) and 3.5e-6
    (displacement); bar 1e-5."""
    groups = [
        (dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8), [(n, KINDS[i % len(KINDS)]) for i, n in enumerate(EDGE_SIZES)]),
        (dict(lr=3e-4, betas=(0.8, 0.99), eps=1e-6), [(4096, "big"), (513, "flip"), (129, "stop"), (50, "zero")]),
        (dict(lr=2e-3, betas=(0.95, 0.9999), eps=1e-8), [(257, "tiny"), (1000, "unit"), (3, "flip")]),
        (dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8), [(0, "unit")]),
    ]
    pair = Pair(groups, zeroing=zeroing, grad_scale=grad_scale, seed=11)

    def schedule(pair, k):
        if k in (4, 8):
            for g in pair.opt.param_groups + pair.ref.param_groups:
                g["lr"] *= 0.5

    worst = _run(pair, 10, each=schedule)
    print(f"zeroing={zeroing} grad_scale={grad_scale}: worst rel_l2 exp_avg {worst[0]:.2e} exp_avg_sq {worst[1]:.2e} "
          f"displacement {worst[2]:.2e}")


def test_parameter_that_skipped_a_step_gets_its_own_bias_correction():
    """torch.optim.Adam counts steps per parameter: one whose .grad was None on step 1 takes step 1's bias correction on its
    first update, not step 2's (which makes that update ~0.74 of the right one)."""
    pair = Pair([(dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8), [(1000, "unit"), (70000, "unit"), (300, "unit")])], seed=21)
    _run(pair, 5, skip_at={1: (1,)})
    assert [int(pair.opt.state[p]["step"]) for p in pair.ps] == [5, 4, 5]


def test_resume_on_the_same_optimizer_uses_the_loaded_moments():
    """Restore-best / resume: load_state_dict on an optimizer that has already stepped (gradients in a persistent buffer, so
    nothing else forces the device table to be rebuilt).  The pre-load moments are kept alive by the test, so an optimizer that
    still wrote into them would write only into memory the test owns; they must stay untouched."""
    groups = [(dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8), [(70000, "unit"), (255, "flip")]),
              (dict(lr=5e-4, betas=(0.8, 0.99), eps=1e-8), [(1000, "big")])]
    pair = Pair(groups, zeroing="flat", seed=31)
    pair.step()
    saved, saved_ref = copy.deepcopy(pair.opt.state_dict()), copy.deepcopy(pair.ref.state_dict())
    pair.step()
    pair.step()
    old = [(pair.opt.state[p]["exp_avg"], pair.opt.state[p]["exp_avg_sq"]) for p in pair.ps]
    old_copy = [(m.clone(), v.clone()) for m, v in old]
    pair.opt.load_state_dict(saved)
    pair.ref.load_state_dict(saved_ref)
    for _ in range(2):
        pair.step()
        pair.check()
    assert [int(pair.opt.state[p]["step"]) for p in pair.ps] == [3, 3, 3]
    for (m, v), (m0, v0) in zip(old, old_copy):
        assert torch.equal(m, m0) and torch.equal(v, v0), "FusedAdam wrote into the moments it held before load_state_dict"


def test_stepped_fused_adam_loads_a_torch_adam_checkpoint():
    """A FusedAdam that has already stepped (other gradients) takes parameters and state of a CUDA fp32 torch.optim.Adam run,
    then continues that run."""
    groups = [(dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8), [(70000, "unit"), (300, "stop")])]
    pair = Pair(groups, zeroing="flat", seed=41)
    tadam_p = [p.detach().clone().requires_grad_(True) for p in pair.ps]
    tadam = torch.optim.Adam(tadam_p, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, foreach=False)
    for _ in range(2):
        pair.set_grads()
        for tp, p in zip(tadam_p, pair.ps):
            tp.grad = p.grad.clone()
        tadam.step()
        pair.ref.step()
    for _ in range(3):                   # the FusedAdam side runs ahead on unrelated gradients
        for p in pair.ps:
            p.grad.copy_(torch.randn_like(p))
        pair.opt.step()
    old = [(pair.opt.state[p]["exp_avg"], pair.opt.state[p]["exp_avg_sq"]) for p in pair.ps]
    old_copy = [(m.clone(), v.clone()) for m, v in old]
    with torch.no_grad():
        for p, tp in zip(pair.ps, tadam_p):
            p.copy_(tp)
    pair.opt.load_state_dict(tadam.state_dict())
    pair.check(crossed=True)
    for _ in range(3):
        pair.step()
        pair.check(crossed=True)
    for (m, v), (m0, v0) in zip(old, old_copy):
        assert torch.equal(m, m0) and torch.equal(v, v0)


@pytest.mark.parametrize("direction", ["fused_to_torch", "torch_to_fused"])
def test_state_dict_round_trip_continues_the_trajectory(direction):
    """Two steps on one optimizer, its state_dict loaded into the other kind, two more steps: the same trajectory as four
    steps of one fp64 Adam."""
    hyper = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    pair = Pair([(hyper, [(70000, "unit"), (255, "flip")]), (dict(hyper, lr=3e-4), [(1000, "big")])], seed=51)
    first = pair.opt if direction == "fused_to_torch" else torch.optim.Adam(
        [dict(g, params=g["params"]) for g in pair.opt.param_groups], foreach=False)
    for _ in range(2):
        pair.set_grads()
        first.step()
        pair.ref.step()
    if direction == "fused_to_torch":
        second = torch.optim.Adam([dict(g, params=g["params"]) for g in pair.opt.param_groups], foreach=False)
    else:
        second = pair.opt
    second.load_state_dict(first.state_dict())
    for _ in range(2):
        pair.set_grads()
        second.step()
        pair.ref.step()
        pair.check(second, crossed=True)


def test_one_launch_per_group_per_step():
    """The bench's training step counts on one Adam launch per optimizer: with every parameter at the same step count a group
    is one launch, whatever its size.  Parameters at different step counts cost one launch per distinct count; a group with
    nothing to update (no gradients, or only empty parameters) costs none."""
    lib = cabi.load()
    hyper = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    pair = Pair([(hyper, [(3 * _CHUNK + 5, "unit"), (7, "unit")]), (hyper, [(100, "unit")]), (hyper, [(0, "unit")])],
                zeroing="flat", seed=61)

    def launches(fn):
        torch.cuda.synchronize()
        n0 = lib.aero_launch_count()
        fn()
        torch.cuda.synchronize()
        return lib.aero_launch_count() - n0

    for _ in range(3):
        pair.set_grads()
        assert launches(pair.opt.step) == 2
    pair.ps[2].grad = None                                   # group 1: nothing to update
    assert launches(pair.opt.step) == 1
    pair.ps[2].grad = torch.ones(100, device=DEV)
    pair.ps[1].grad = None
    assert launches(pair.opt.step) == 2                      # group 0: one count; group 1: one count
    pair.ps[1].grad = torch.ones(7, device=DEV)
    assert launches(pair.opt.step) == 3                      # group 0 now holds two step counts


@pytest.mark.parametrize("bad", ["non_contiguous", "fp64", "non_contiguous_grad"])
def test_unsupported_parameter_raises(bad):
    if bad == "non_contiguous":
        p = torch.empty_strided((4, 6), (1, 4), device=DEV).fill_(1.0).requires_grad_(True)
        p.grad = torch.ones(4, 6, device=DEV)
    elif bad == "fp64":
        p = torch.ones(5, dtype=torch.float64, device=DEV, requires_grad=True)
        p.grad = torch.ones_like(p)
    else:
        p = torch.ones(4, 6, device=DEV, requires_grad=True)
        p.grad = torch.ones(6, 4, device=DEV).t()
    before = p.detach().clone()
    with pytest.raises(TypeError):
        FusedAdam([p]).step()
    torch.cuda.synchronize()
    assert torch.equal(p.detach(), before)


# ------------------------------------------------------------------------------------------------ evaluation after a step
def _no_ftb_model():
    torch.manual_seed(SEED)
    m = Aero(**dict(aero_kwargs("aero_4-16_512_256"), enc_freq_attn=4))
    m.load_state_dict(trained_like_(m.state_dict()))
    assert not list(m.buffers())        # nothing but the optimizer changes a tensor version
    assert sum(p.numel() for p in m.parameters()) == 18427906
    return m


def _shipped_model():
    torch.manual_seed(SEED)
    m = Aero(**aero_kwargs("aero_4-16_512_256"))
    m.load_state_dict(trained_like_(m.state_dict()))
    assert list(m.buffers())            # FTB BatchNorm running statistics
    return m


def _fresh_eval(m, x):
    args, kwargs = m._init_args_kwargs            # how the reference's checkpoint writer re-creates the model
    f = Aero(*args, **kwargs)
    f.load_state_dict(m.state_dict())
    f = f.cuda().eval()
    f.use_cuda_graph(False)
    out = f(x)
    torch.cuda.synchronize()
    return out.cpu()


@pytest.mark.parametrize("graph", [True, False], ids=["graph", "eager"])
@pytest.mark.parametrize("route", ["autograd", "trainer"])
@pytest.mark.parametrize("model", ["no_ftb", "aero_4-16_512_256"])
def test_eval_after_a_training_step_sees_the_new_weights(model, route, graph):
    """Per-epoch validation: eval forwards (the third one replays a captured CUDA graph under "auto"), one training step with
    FusedAdam (through loss.backward() + optimizer.step(), or GeneratorTrainer.step with gradients in its flat buffer), eval
    again.  The output must be that of a fresh model built from the stepped state_dict (same kernels, so expected identical;
    bar 1e-6) and must differ from the pre-step output.  Without FTB no BatchNorm statistics change in train mode, so the
    only thing that tells the engine's caches the weights changed is the optimizer step itself."""
    from aero_b200.trainer import GeneratorTrainer
    m = (_no_ftb_model() if model == "no_ftb" else _shipped_model()).cuda()
    m.use_cuda_graph("auto" if graph else False)
    x = white_noise((2, 1, 4000), seed=SEED + 9).cuda()
    m.eval()
    before = [m(x).cpu() for _ in range(3)]
    assert all(torch.equal(before[0], b) for b in before[1:])
    target = white_noise((2, 1, 16000), seed=SEED + 10).cuda() * 0.1
    if route == "autograd":
        opt = FusedAdam(m.parameters(), lr=3e-4)
        m.train()
        loss = (m(x) - target).abs().mean()
        loss.backward()
        opt.step()
    else:
        tr = GeneratorTrainer(m, lr=3e-4)
        tr.step(x, lambda pr: (pr - target).abs().mean())
    m.eval()
    after = [m(x).cpu() for _ in range(3)]       # eager, eager, then (graph) a capture of the new weights
    want = _fresh_eval(m, x)
    errs = [rel_l2(a, want) for a in after]
    moved = rel_l2(before[0], want)
    print(f"{model} {route} graph={graph}: eval after step vs fresh model {max(errs):.2e}, pre-step output vs fresh {moved:.2e}")
    assert max(errs) <= 1e-6, errs
    assert moved > 1e-4, moved


# ------------------------------------------------------------------------------------------------ GAN steps vs the plain route
def _plain_gan_step(m, d, opt_g, opt_d, lr_b, hr_b, stft, n_layers=4, lmbda=100.0):
    """The reference solver's route (src/solver.py:292-320,475-520,602-612): plain autograd through model(lr) and the
    discriminator, torch.optim.Adam for each network, zero_grad before each backward."""
    relu, l1 = torch.nn.functional.relu, torch.nn.functional.l1_loss
    m.train()
    pr = m(lr_b)
    sc, mag = stft(pr.squeeze(1), hr_b.squeeze(1))
    fake_detached, real, fake = d(pr.detach()), d(hr_b), d(pr)
    d_loss = sum(relu(1 + s[-1]).mean() for s in fake_detached) + sum(relu(1 - s[-1]).mean() for s in real)
    w = (4.0 / (n_layers + 1)) / d.num_D
    feat = 0.0
    for i in range(d.num_D):
        for j in range(len(fake[i]) - 1):
            feat = feat + w * l1(fake[i][j], real[i][j].detach())
    adv = sum(relu(1 - s[-1]).mean() for s in fake)
    opt_g.zero_grad()
    (sc + mag + adv + lmbda * feat).backward()
    opt_g.step()
    opt_d.zero_grad()
    d_loss.backward()
    opt_d.step()


def _displacement_error(ps, qs, p0):
    """rel_l2 of (p - p0) against (q - p0) over all parameters of a network together, and the worst single parameter."""
    num = den = 0.0
    worst = 0.0
    for p, q, z in zip(ps, qs, p0):
        a, b = p.detach().double() - z, q.detach().double() - z
        num += float((a - b).pow(2).sum())
        den += float(b.pow(2).sum())
        worst = max(worst, float((a - b).norm() / b.norm().clamp_min(1e-30)))
    return (num / den) ** 0.5, worst


GAN_TOL = 1e-2


def test_gan_trainer_steps_match_plain_autograd_with_torch_adam():
    """Three GanTrainer.step calls (flat gradient buffers, FusedAdam, discriminator zeroed in between) against the reference's
    route from the same weights and BatchNorm buffers, with one eval forward between steps 2 and 3.  Both networks' parameter
    displacements are compared after every step, over all parameters of a network together.

    The two routes' generator gradients differ by up to 1e-4 (test_gan_training_step_runs_and_updates_both_networks), and Adam's
    sign-like early updates turn that into O(1) differences on elements whose gradient is rounding noise (e.g. a bias in front
    of a BatchNorm, whose true gradient is zero).  The bar, 1e-2 over a whole network, caps that amplification; the errors of
    every step are printed so that it can be tightened to about three times a measured run."""
    from aero_b200.discriminator import Discriminator
    from aero_b200.losses import MultiResolutionSTFTLoss
    from aero_b200.trainer import GanTrainer
    torch.manual_seed(SEED)
    kw = aero_kwargs("aero_4-16_512_256")
    sd_g = trained_like_(Aero(**kw).state_dict())
    torch.manual_seed(SEED + 1)
    sd_d = Discriminator(3, 16, 4, 4).state_dict()
    nets = []
    for _ in range(2):
        m = Aero(**kw)
        m.load_state_dict(sd_g)
        d = Discriminator(3, 16, 4, 4)
        d.load_state_dict(sd_d)
        nets.append((m.cuda(), d.cuda()))
    (ma, da), (mb, db) = nets
    g0 = [p.detach().double().clone() for p in ma.parameters()]
    d0 = [p.detach().double().clone() for p in da.parameters()]
    tr = GanTrainer(ma, da, lr=3e-4)
    opt_g = torch.optim.Adam(mb.parameters(), lr=3e-4, betas=(0.9, 0.999), eps=1e-8)
    opt_d = torch.optim.Adam(db.parameters(), lr=3e-4, betas=(0.9, 0.999), eps=1e-8)
    stft = MultiResolutionSTFTLoss()
    rows = []
    for k in range(3):
        lr_b = white_noise((2, 1, 4000), seed=SEED + 20 + k).cuda()
        hr_b = white_noise((2, 1, 16000), seed=SEED + 30 + k).cuda() * 0.1
        if k == 2:
            ea, eb = ma.eval()(lr_b), mb.eval()(lr_b)
            rows.append(("eval", rel_l2(ea.cpu(), eb.cpu())))
        tr.step(lr_b, hr_b, stft)
        _plain_gan_step(mb, db, opt_g, opt_d, lr_b, hr_b, stft)
        torch.cuda.synchronize()
        eg, eg_worst = _displacement_error(ma.parameters(), mb.parameters(), g0)
        ed, ed_worst = _displacement_error(da.parameters(), db.parameters(), d0)
        rows.append((k + 1, eg, eg_worst, ed, ed_worst))
        for (n, a), (_, b) in zip(ma.named_buffers(), mb.named_buffers()):
            assert rel_l2(a.cpu(), b.cpu()) < 1e-4, (k, n)
    print("GAN steps, trainer vs plain route (step, G all, G worst param, D all, D worst param):", rows)
    for r in rows:
        if r[0] == "eval":
            assert r[1] < 1e-3, r
        else:
            assert r[1] < GAN_TOL and r[3] < GAN_TOL, r
