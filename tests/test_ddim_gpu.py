"""DDIM sampler on the GPU: the update kernel against the fp64 oracle, whole DDIM trajectories of both model families against the
oracle, coexistence with the DDPM loop on one handle, Philox keying, the ensemble driver and the foreign-model loop.

The trajectory gate is rel-L2 of x0 <= 1e-2.  Each Family R trajectory case also runs the oracle with the time-embedding bug a
stride > 1 invites (the next step embedded at tau_k - 1, what the DDPM side branch computes) and checks that this wrong answer is
at least 3x the gate away, so the gate can tell the two apart."""
import os
import subprocess
import sys

import pytest
import torch

from diffusionmodelscustom_b200 import DiffusionUtils, generation, synth
from diffusionmodelscustom_b200 import _native as N
from diffusionmodelscustom_b200.modules import NativeModel
from oracle import ddpm_oracle as O
from tests import ddim_oracle as DO
from tests import gpu_util as G
from tests.cases import D_CASES, R_CASES
from tests.model_util import build_ours_d, build_ours_r, inputs_d, inputs_r

pytestmark = pytest.mark.gpu
GATE = 1e-2
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ----------------------------------------------------------------------------------------------- op level
def _op(x, eps, z, ahat_d, T, t, tp, eta, seed=0, offset=0, scale=1.0):
    """b2d_op_ddim_update on a copy of x inside a NaN-poisoned buffer: the elements past x must stay untouched."""
    n = x.numel()
    buf = torch.full((n + 64,), float("nan"), device="cuda")
    buf[:n] = x.reshape(-1).cuda()
    zd = None if z is None else z.contiguous().cuda()
    ed = eps.contiguous().cuda()
    N.check(N.lib().b2d_op_ddim_update(buf.data_ptr(), ed.data_ptr(), N.ptr(zd), ahat_d.data_ptr(), T, t, tp, float(eta), x.shape[0],
                                       x[0].numel(), seed, offset, float(scale), G.stream()))
    torch.cuda.synchronize()
    assert torch.isnan(buf[n:]).all(), "the update wrote past its output"
    return buf[:n].reshape(x.shape).cpu()


@pytest.mark.parametrize("t,tp", [(999, 899), (500, 499), (120, 37), (999, -1), (3, -1)])
@pytest.mark.parametrize("eta", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("scale", [1.0, 0.005])
def test_ddim_update_with_injected_noise_matches_oracle(t, tp, eta, scale):
    _, _, ahat = O.schedule_tables(1000, 1e-4, 0.02)
    g = torch.Generator().manual_seed(t * 7 + max(tp, 0))
    x = torch.randn(3, 1, 32, 32, generator=g) * 4
    eps = torch.randn(3, 1, 32, 32, generator=g)
    z = torch.randn(3, 1, 32, 32, generator=g)
    out = _op(x, eps, z, ahat.cuda(), 1000, t, tp, eta, scale=scale)
    ref = DO.ddim_step(x, eps, z * scale, t, tp, eta, ahat.double())
    assert G.rel_l2(out, ref) <= 1e-6, (t, tp, eta, G.rel_l2(out, ref))


@pytest.mark.parametrize("t,tp", [(999, 899), (500, 480)])
def test_ddim_update_philox_noise_is_deterministic_and_standard_normal(t, tp):
    _, _, ahat = O.schedule_tables(1000, 1e-4, 0.02)
    ahd = ahat.cuda()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(8, 1, 64, 64, generator=g) * 4
    eps = torch.randn(8, 1, 64, 64, generator=g)
    zs = []
    for eta in (0.5, 1.0):
        a = _op(x, eps, None, ahd, 1000, t, tp, eta, seed=1234)
        b = _op(x, eps, None, ahd, 1000, t, tp, eta, seed=1234)
        assert torch.equal(a, b)
        mean = DO.ddim_step(x, eps, None, t, tp, eta, ahat.double())
        _, _, sigma = DO.ddim_coefficients(t, tp, eta, ahat.double())
        z = (a.double() - mean) / sigma
        assert abs(float(z.mean())) < 0.02 and abs(float(z.std()) - 1.0) < 0.02, eta
        assert abs(float((z ** 4).mean()) - 3.0) < 0.15
        zs.append(z)
    # both eta values read the same draw (keyed by (seed; sample, element, t)), up to the fp32 rounding of the update
    assert G.rel_l2(zs[0], zs[1]) < 1e-3
    # keyed by the global sample index: a shard at offset 4 draws samples 4..7, and another seed or t draws other numbers
    shard = _op(x[4:], eps[4:], None, ahd, 1000, t, tp, 1.0, seed=1234, offset=4)
    assert torch.equal(shard, _op(x, eps, None, ahd, 1000, t, tp, 1.0, seed=1234)[4:])
    assert not torch.equal(_op(x, eps, None, ahd, 1000, t, tp, 1.0, seed=1235), _op(x, eps, None, ahd, 1000, t, tp, 1.0, seed=1234))
    # the last step never draws
    assert torch.equal(_op(x, eps, None, ahd, 1000, t, -1, 1.0, seed=1), _op(x, eps, None, ahd, 1000, t, -1, 1.0, seed=2))


def test_ddim_update_rejects_bad_arguments():
    _, _, ahat = O.schedule_tables(100, 1e-4, 0.02)
    x = torch.zeros(1, 1, 8, 8, device="cuda")
    ahd = ahat.cuda()
    for t, tp, eta in ((0, -1, 0.0), (100, 50, 0.0), (50, 50, 0.0), (50, 0, 0.0), (50, 10, 1.5), (50, 10, -0.1)):
        rc = N.lib().b2d_op_ddim_update(x.data_ptr(), x.data_ptr(), None, ahd.data_ptr(), 100, t, tp, eta, 1, 64, 0, 0, 1.0,
                                        G.stream())
        assert rc != 0, (t, tp, eta)


# ----------------------------------------------------------------------------------------------- trajectories
def _r_oracle(sd, inp):
    return lambda x, tt: O.family_r_forward(sd, x.float(), tt, inp["y"], inp["cond"], inp["lsm"], inp["topo"]).double()


# The synthetic weights barely depend on t: with them, embedding the wrong timestep moves x0 by only 0.7 %, below the gate.  The
# trajectory cases scale every time projection by this factor, so that eps depends on t strongly enough (5-7 % for the wrong
# embedding at these shapes) for the gate to see the difference.
TEMB_GAIN = 16.0


def _t_sensitive_r(case):
    net, sd = build_ours_r(case)
    sd = {k: (v * TEMB_GAIN if "time_projection" in k else v) for k, v in sd.items()}
    net.load_state_dict(sd, strict=True)
    return net, sd


def _buggy(fn, ts):
    """The model as a DDPM-style side branch would drive it over a strided sequence: step k >= 1 embeds tau_{k-1} - 1."""
    wrong = {ts[k]: ts[k - 1] - 1 for k in range(1, len(ts))}
    return lambda x, tt: fn(x, torch.full_like(tt, wrong.get(int(tt[0]), int(tt[0]))))


@pytest.mark.parametrize("name,S,eta", [("full_64_randbn", 10, 0.0), ("full_64_randbn", 25, 0.0), ("full_64_randbn", 10, 1.0),
                                        ("full_64_randbn", 25, 1.0), ("cfg3_full_128", 10, 0.0)])
def test_family_r_ddim_trajectory_vs_oracle(name, S, eta):
    case = R_CASES[name]
    B = 2 if name == "full_64_randbn" else case["batch"]
    net, sd = _t_sensitive_r(case)
    inp, dev = inputs_r(case, B)
    du = DiffusionUtils(1000, 1e-4, 0.02, "cuda")
    ts = du.ddim_timesteps(S)
    z = torch.randn((S, B, 1, case["hw"], case["hw"]), generator=torch.Generator().manual_seed(S))
    NativeModel.saturation_count(reset=True)
    x0 = du.sample_ddim(dev["x"], net, dev["y"], dev["cond"], dev["lsm"], dev["topo"], steps=S, eta=eta, noise=z.cuda(), seed=4)
    assert torch.isfinite(x0).all()
    assert NativeModel.saturation_count() == 0
    fn = _r_oracle(sd, inp)
    ahat = du.alpha_hat.cpu().double()
    ref = DO.ddim_sample(fn, inp["x"], ts, eta, ahat, noise=z)
    err = G.rel_l2(x0, ref)
    assert err <= GATE, (name, S, eta, err)
    wrong = DO.ddim_sample(_buggy(fn, ts), inp["x"], ts, eta, ahat, noise=z)
    assert G.rel_l2(wrong, ref) >= 3 * GATE, ("the gate cannot see the side-branch bug at this case", G.rel_l2(wrong, ref))
    assert G.rel_l2(x0, wrong) > err


def test_family_d_ddim_trajectory_vs_oracle():
    case = D_CASES["downscale_32"]
    net, sd = build_ours_d(case)
    inp, dev = inputs_d(case)
    du = DiffusionUtils(1000, 1e-4, 0.02, "cuda")
    S = 10
    NativeModel.saturation_count(reset=True)
    x0 = du.sample_ddim(dev["x"], net, cond_img=dev["y_lowres"], steps=S, eta=0.0)
    assert NativeModel.saturation_count() == 0
    fn = lambda x, tt: O.family_d_forward(sd, x.float(), tt, inp["y_lowres"]).double()
    ref = DO.ddim_sample(fn, inp["x"], du.ddim_timesteps(S), 0.0, du.alpha_hat.cpu().double())
    assert G.rel_l2(x0, ref) <= GATE, G.rel_l2(x0, ref)


# ----------------------------------------------------------------------------------------------- coexistence with DDPM
def test_ddpm_path_is_unchanged_around_ddim_calls():
    case = R_CASES["full_64_randbn"]
    B, T = 2, 1000
    net, _ = build_ours_r(case)
    inp, dev = inputs_r(case, B)
    du = DiffusionUtils(T, 1e-4, 0.02, "cuda")
    z = synth.step_noise(B, 1, case["hw"], T, seed=12).cuda()
    args = (dev["y"], dev["cond"], dev["lsm"], dev["topo"])
    first = du.sample(dev["x"], net, *args, noise=z, seed=3)
    n_ddpm = net.launch_count()
    a = du.sample_ddim(dev["x"], net, *args, steps=10, noise=z[:10], seed=3)
    n10 = net.launch_count()
    b = du.sample_ddim(dev["x"], net, *args, steps=25, noise=z[:25], seed=3)
    n25 = net.launch_count()
    a2 = du.sample_ddim(dev["x"], net, *args, steps=10, noise=z[:10], seed=3)
    second = du.sample(dev["x"], net, *args, noise=z, seed=3)
    assert torch.equal(first, second)
    assert torch.equal(a, a2)
    assert net.launch_count() == n_ddpm
    fresh_net, _ = build_ours_r(case)
    assert torch.equal(du.sample(dev["x"], fresh_net, *args, noise=z, seed=3), first)
    per_step = (n_ddpm - 2) / (T - 1)
    for S, n in ((10, n10), (25, n25)):
        assert abs(n - S * per_step) <= 0.05 * S * per_step + 8, (S, n, per_step)
    assert G.rel_l2(a, b) > 0     # the two step counts are different samplers


def test_host_entry_runs_ddim_and_resets_to_ddpm():
    case = R_CASES["full_64_randbn"]
    B, S = 2, 10
    net, _ = build_ours_r(case)
    inp, dev = inputs_r(case, B)
    du = DiffusionUtils(1000, 1e-4, 0.02, "cuda")
    z = torch.randn((S, B, 1, 64, 64), generator=torch.Generator().manual_seed(1))
    ref = du.sample_ddim(dev["x"], net, dev["y"], dev["cond"], dev["lsm"], dev["topo"], steps=S, eta=1.0, noise=z.cuda())
    h = net._ensure(B, 64, dev["x"].device)
    net._set_sampler(h, (du.ddim_timesteps(S), 1.0))
    out = inp["x"].clone()
    with torch.cuda.device(dev["x"].device):
        net._cond_key = None
        N.check(N.lib().b2d_sample_host(h, out.data_ptr(), inp["lsm"].data_ptr(), inp["topo"].data_ptr(), inp["cond"].data_ptr(), 0, 0,
                                        inp["y"].data_ptr(), z.data_ptr(), 0, 0, 1.0, B))
    assert G.rel_l2(out, ref) < 1e-5
    # sample_host sets the DDPM loop again
    zz = synth.step_noise(B, 1, 64, 1000, seed=2)
    h1 = du.sample_host(inp["x"], net, inp["y"], inp["cond"], inp["lsm"], inp["topo"], noise=zz)
    h2 = du.sample(dev["x"], net, dev["y"], dev["cond"], dev["lsm"], dev["topo"], noise=zz.cuda())
    assert G.rel_l2(h1, h2) < 1e-5


def test_ddim_philox_is_shard_invariant_and_deterministic():
    case = R_CASES["cfg2_lsmtopo_64"]
    net, _ = build_ours_r(case)
    inp, dev = inputs_r(case, 4)
    du = DiffusionUtils(1000, 1e-4, 0.02, "cuda")
    kw = dict(steps=10, eta=1.0)
    full = du.sample_ddim(dev["x"], net, None, None, dev["lsm"], dev["topo"], seed=99, **kw)
    again = du.sample_ddim(dev["x"], net, None, None, dev["lsm"], dev["topo"], seed=99, **kw)
    assert torch.equal(full, again)
    lo = du.sample_ddim(dev["x"][:2], net, None, None, dev["lsm"][:2], dev["topo"][:2], seed=99, sample_offset=0, **kw)
    hi = du.sample_ddim(dev["x"][2:], net, None, None, dev["lsm"][2:], dev["topo"][2:], seed=99, sample_offset=2, **kw)
    assert G.rel_l2(torch.cat([lo, hi]), full) < 2e-3
    other = du.sample_ddim(dev["x"], net, None, None, dev["lsm"], dev["topo"], seed=100, **kw)
    assert G.rel_l2(other, full) > 1e-2


_ENV_SCRIPT = r"""
import json, sys, torch
sys.path.insert(0, sys.argv[1])
from diffusionmodelscustom_b200 import DiffusionUtils
from tests.cases import R_CASES
from tests.model_util import build_ours_r, inputs_r
case = R_CASES["full_64_randbn"]
net, _ = build_ours_r(case)
inp, dev = inputs_r(case, 2)
z = torch.randn((10, 2, 1, 64, 64), generator=torch.Generator().manual_seed(3)).cuda()
x0 = DiffusionUtils(1000, 1e-4, 0.02, "cuda").sample_ddim(dev["x"], net, dev["y"], dev["cond"], dev["lsm"], dev["topo"], steps=10,
                                                          eta=1.0, noise=z)
torch.save(x0.cpu(), sys.argv[2])
"""


@pytest.mark.parametrize("env", ["B2D_NO_GRAPH", "B2D_NO_TEMB_PIPE"])
def test_ddim_without_graphs_or_embedding_pipeline(env, tmp_path):
    """Both switches are read once per process: the run without them is compared against a subprocess with one of them set."""
    case = R_CASES["full_64_randbn"]
    net, _ = build_ours_r(case)
    inp, dev = inputs_r(case, 2)
    z = torch.randn((10, 2, 1, 64, 64), generator=torch.Generator().manual_seed(3)).cuda()
    ref = DiffusionUtils(1000, 1e-4, 0.02, "cuda").sample_ddim(dev["x"], net, dev["y"], dev["cond"], dev["lsm"], dev["topo"], steps=10,
                                                               eta=1.0, noise=z)
    out = str(tmp_path / "x0.pt")
    r = subprocess.run([sys.executable, "-c", _ENV_SCRIPT, ROOT, out], env=dict(os.environ, **{env: "1"}), capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert G.rel_l2(torch.load(out), ref) < 1e-5


# ----------------------------------------------------------------------------------------------- ensemble driver
def test_ensemble_ddim_is_independent_of_sub_batch_and_slices(monkeypatch):
    case = R_CASES["full_64_randbn"]
    net, _ = build_ours_r(case)
    D, M = 3, 5
    inp = synth.synth_inputs(D, 64, seed=77, has_lsm=True, has_topo=True, has_cond=True, num_classes=4)
    du = DiffusionUtils(1000, 1e-4, 0.02, "cuda")
    kw = dict(season=inp["y"], cond_img=inp["cond"], lsm=inp["lsm"], topo=inp["topo"], seed=11, eta=1.0)
    a, st10 = generation.generate_ensemble(net, du, D, M, sub_batch=4, steps=10, return_stats=True, **kw)
    b, st10b = generation.generate_ensemble(net, du, D, M, sub_batch=15, steps=10, return_stats=True, **kw)
    assert a.shape == (D, M, 1, 64, 64) and torch.isfinite(a).all()
    assert G.rel_l2(a, b) <= 2e-3
    assert float((a[0, 0] - a[0, 1]).abs().max()) > 1e-3
    _, st20 = generation.generate_ensemble(net, du, D, M, sub_batch=15, steps=20, return_stats=True, **kw)
    assert 1.9 <= st20["launches"] / st10b["launches"] <= 2.1, (st10b["launches"], st20["launches"])
    # the second date alone: the slice [M, 2M) of the member list, keyed by the same global member indices; against a full run
    # whose second sub-batch is exactly that slice (same program, same batch)
    by_date = generation.generate_ensemble(net, du, D, M, sub_batch=M, steps=10, **kw)
    monkeypatch.setattr(generation, "shard_range", lambda n, w, r: (M, 2 * M))
    one = generation.generate_ensemble(net, du, D, M, sub_batch=15, steps=10, **kw)
    assert one.shape == (M, 1, 64, 64)
    assert G.rel_l2(one, by_date[1]) <= 1e-6
    # steps=None keeps the DDPM loop of the same handle
    monkeypatch.undo()
    ddpm = generation.generate_ensemble(net, DiffusionUtils(9, 1e-4, 0.02, "cuda"), D, M, sub_batch=15, season=inp["y"],
                                        cond_img=inp["cond"], lsm=inp["lsm"], topo=inp["topo"], seed=11)
    assert torch.isfinite(ddpm).all() and G.rel_l2(ddpm, b) > 1e-2


# ----------------------------------------------------------------------------------------------- foreign eps-model
class _TinyEps(torch.nn.Module):
    def __init__(self):
        super().__init__()
        g = torch.Generator().manual_seed(0)
        self.conv = torch.nn.Conv2d(1, 1, 3, padding=1)
        with torch.no_grad():
            self.conv.weight.copy_(torch.randn(1, 1, 3, 3, generator=g) * 0.2)
            self.conv.bias.fill_(0.1)

    def forward(self, x, t, *unused):
        return torch.tanh(self.conv(x)) + torch.sin(t.to(x.dtype) / 37.0)[:, None, None, None]


@pytest.mark.parametrize("eta", [0.0, 1.0])
def test_foreign_model_loop_matches_oracle(eta):
    T, S, B = 100, 10, 3
    model = _TinyEps()
    du = DiffusionUtils(T, 1e-4, 0.02, "cuda")
    g = torch.Generator().manual_seed(8)
    x = torch.randn(B, 1, 16, 16, generator=g)
    z = torch.randn(S, B, 1, 16, 16, generator=g)
    out = du.sample_ddim(x.cuda(), model.cuda(), steps=S, eta=eta, noise=z.cuda())
    cpu_model = _TinyEps().double()
    ref = DO.ddim_sample(lambda xx, tt: cpu_model(xx, tt), x, du.ddim_timesteps(S), eta, du.alpha_hat.cpu().double(), noise=z)
    assert G.rel_l2(out, ref) <= 1e-5, G.rel_l2(out, ref)
    with pytest.raises(N.NativeError):
        du.sample_ddim(x, model.cpu(), steps=S)
