"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):  python oracle/gen_golden.py
The reference (Feuermagier/Beyond_Deep_Ensembles @ b805d6f) is imported from /root/reference,
driven through its public optimizer API on seeded inputs, with noise injected at the
reference's own draw points (src.algos.util.normal_like, ivorn.normal_like and
torch.distributions.lowrank_multivariate_normal._standard_normal).  Outputs are small .npz
files; the tests never need the reference again.
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import torch

REF = "/root/reference"
ROOT = Path(__file__).resolve().parent.parent
OUT = ROOT / "tests" / "golden"
sys.path.insert(0, REF)
sys.path.insert(0, str(ROOT / "tests"))

import src.algos.util as ref_util  # noqa: E402
import src.algos.ivorn as ref_ivorn  # noqa: E402
from src.algos.svgd import SVGDOptimizer, rbf  # noqa: E402
from src.algos.swag import SwagOptimizer  # noqa: E402
from src.algos.ivorn import iVONOptimizer  # noqa: E402
from src.algos.bbb import BBBOptimizer, GaussianPrior, MixturePrior  # noqa: E402
from src.algos.util import GaussianParameter  # noqa: E402
from src.algos.algo import LastLayerBayesianOptimizer  # noqa: E402
from src.algos.ensemble import DeepEnsemble  # noqa: E402

import golden_models as gm  # noqa: E402

torch.set_num_threads(1)  # deterministic reduction order inside ATen


class NoiseTape:
    """Replays pre-drawn noise in call order and records what was handed out."""

    def __init__(self, seed: int):
        self.gen = torch.Generator().manual_seed(seed)
        self.log: list[np.ndarray] = []

    def like(self, tensor):
        z = torch.randn(tensor.shape, generator=self.gen, dtype=torch.float32).to(tensor.dtype)
        self.log.append(z.reshape(-1).numpy().copy())
        return z

    def standard_normal(self, shape, dtype, device):
        z = torch.randn(shape, generator=self.gen, dtype=torch.float32).to(dtype)
        self.log.append(z.reshape(-1).numpy().copy())
        return z


def batches(seed: int, steps: int, in_dim: int = 8, bs: int = 32):
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(in_dim, generator=g)
    xs, ys = [], []
    for _ in range(steps):
        x = torch.randn(bs, in_dim, generator=g)
        xs.append(x)
        ys.append(x @ w + 0.1 * torch.randn(bs, generator=g))
    return torch.stack(xs), torch.stack(ys)


# ---------------------------------------------------------------------------------------
def gen_rbf():
    """rbf() itself (svgd.py:14-32) in fp32 and fp64 plus the fused identity inputs."""
    cases = [(5, 37, 0), (10, 501, 1), (20, 1000, 2), (3, 64, 3), (2, 9, 4), (10, 4099, 5), (16, 257, 6), (1, 33, 7)]
    out = {}
    for n, D, seed in cases:
        g = torch.Generator().manual_seed(100 + seed)
        scale = 0.05 * (1 + 0.1 * torch.arange(n, dtype=torch.float32)).unsqueeze(1)
        X = scale * torch.randn(n, D, generator=g)
        key = f"n{n}_D{D}"
        out[f"{key}_X"] = X.numpy()
        k32, _ = rbf(X.clone())
        k64, gk64 = rbf(X.double())
        d64 = torch.cdist(X.double(), X.double(), p=2) ** 2
        out[f"{key}_K32"] = k32.numpy()
        out[f"{key}_K64"], out[f"{key}_gK64"] = k64.numpy(), gk64.numpy()
        out[f"{key}_d64"] = d64.numpy()
        q = torch.quantile(d64, 0.5)
        out[f"{key}_median64"] = np.array(q.item())
        # h_override branch (svgd.py:19-20); its gradient only where a test reads it (keeps the file under 1 MB)
        ko, gko = rbf(X.double(), h_override=0.7)
        out[f"{key}_K64_h07"] = ko.numpy()
        if key == "n10_D501":
            out[f"{key}_gK64_h07"] = gko.numpy()
    np.savez_compressed(OUT / "rbf.npz", **out)


class RecordingAdam(torch.optim.Adam):
    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.recorded = []

    def step(self, closure=None):
        self.recorded.append(torch.cat([p.grad.reshape(-1) for g in self.param_groups for p in g["params"]]).numpy().copy())
        return super().step(closure)


def gen_svgd():
    """Three full reference SVGDOptimizer steps on the UCI MLP (D=501, n=10, Adam)."""
    n, steps = 10, 3
    torch.manual_seed(7)
    model = gm.make_mlp()
    g = torch.Generator().manual_seed(11)
    D = sum(p.numel() for p in model.parameters())
    init = (0.3 * torch.randn(n, D, generator=g)).numpy()
    gm.load_flat(model.parameters(), init[0])
    calls = {"k": 0}

    def reset():
        calls["k"] += 1
        gm.load_flat(model.parameters(), init[calls["k"]])

    base = RecordingAdam(model.parameters(), lr=1e-2)
    opt = SVGDOptimizer(model.parameters(), reset, base, particle_count=n, dataset_size=768, l2_reg=0.01,
                        kernel_grad_scale=1.0)
    xs, ys = batches(21, steps)
    losses, parts = [], []
    for s in range(steps):
        fwd, bwd = gm.mse_closures(model, xs[s], ys[s])
        losses.append(opt.step(fwd, bwd).item())
        parts.append(np.stack([gm.flat_params(opt._params_for_particle(i)) for i in range(n)]))
    # sample_parameters cursor semantics (svgd.py:107-112)
    seen = []
    for _ in range(n + 2):
        opt.sample_parameters()
        seen.append(gm.flat_params(model.parameters()))
    np.savez_compressed(OUT / "svgd_steps.npz", init=init, xs=xs.numpy(), ys=ys.numpy(), losses=np.array(losses),
                        new_grads=np.stack(base.recorded).reshape(steps, n, D), particles=np.stack(parts),
                        sampled=np.stack(seen))


def gen_svgd_sgd():
    """Reference SVGDOptimizer with the CIFAR base optimizer (experiments/cifar/cifar.yaml:219-223:
    SGD lr 0.05, momentum 0.9, Nesterov, weight decay 3e-4) plus a StepLR schedule and a base-optimizer
    checkpoint round trip after step 2 — pins the shared-state / stepped-once-per-particle semantics of
    svgd.py:92-103 that the fused apply kernel reproduces.  n = 5 (the shipped particle count)."""
    n, steps = 5, 4
    torch.manual_seed(9)
    model = gm.make_mlp()
    g = torch.Generator().manual_seed(13)
    D = sum(p.numel() for p in model.parameters())
    init = (0.3 * torch.randn(n, D, generator=g)).numpy()
    gm.load_flat(model.parameters(), init[0])
    calls = {"k": 0}

    def reset():
        calls["k"] += 1
        gm.load_flat(model.parameters(), init[calls["k"]])

    base = torch.optim.SGD(model.parameters(), lr=0.05, momentum=0.9, nesterov=True, weight_decay=3e-4)
    opt = SVGDOptimizer(model.parameters(), reset, base, particle_count=n, dataset_size=768, l2_reg=3e-4,
                        kernel_grad_scale=1.0)
    sched = torch.optim.lr_scheduler.StepLR(base, step_size=2, gamma=0.5)
    xs, ys = batches(23, steps)
    losses, parts, bufs, lrs = [], [], [], []
    for s in range(steps):
        fwd, bwd = gm.mse_closures(model, xs[s], ys[s])
        lrs.append(base.param_groups[0]["lr"])
        losses.append(opt.step(fwd, bwd).item())
        sched.step()
        parts.append(np.stack([gm.flat_params(opt._params_for_particle(i)) for i in range(n)]))
        bufs.append(np.concatenate([base.state[p]["momentum_buffer"].reshape(-1).numpy() for p in model.parameters()]))
    np.savez_compressed(OUT / "svgd_sgd_steps.npz", init=init, xs=xs.numpy(), ys=ys.numpy(), losses=np.array(losses),
                        particles=np.stack(parts), momentum_buffers=np.stack(bufs), lrs=np.array(lrs))


def gen_swag():
    """Reference SwagOptimizer: 6 SGD steps with K=4 (so the ring wraps), then two samples."""
    K, steps = 4, 6
    torch.manual_seed(3)
    model = gm.make_mlp()
    g = torch.Generator().manual_seed(5)
    D = sum(p.numel() for p in model.parameters())
    init = (0.3 * torch.randn(D, generator=g)).numpy()
    gm.load_flat(model.parameters(), init)
    base = torch.optim.SGD(model.parameters(), lr=0.05, momentum=0.9)
    opt = SwagOptimizer(model.parameters(), base, update_interval=2, start_epoch=1, deviation_samples=K)
    xs, ys = batches(22, 2 * steps)
    losses, thetas = [], []
    # epoch 0: before start_epoch -> no moments collected; epoch 1: every 2nd step collects
    for s in range(2 * steps):
        if s == 2:
            opt.complete_epoch()
        fwd, bwd = gm.mse_closures(model, xs[s], ys[s])
        losses.append(opt.step(fwd, bwd).item())
        thetas.append(gm.flat_params(model.parameters()))
    tape = NoiseTape(41)
    import torch.distributions.lowrank_multivariate_normal as lrmn
    orig = lrmn._standard_normal
    lrmn._standard_normal = tape.standard_normal
    try:
        samples = []
        for _ in range(2):
            opt.sample_parameters()
            samples.append(gm.flat_params(model.parameters()))
    finally:
        lrmn._standard_normal = orig
    # a further step must restore the original parameters first (swag.py:38,76-82)
    fwd, bwd = gm.mse_closures(model, xs[0], ys[0])
    loss_after = opt.step(fwd, bwd).item()
    np.savez_compressed(
        OUT / "swag_steps.npz", init=init, xs=xs.numpy(), ys=ys.numpy(), losses=np.array(losses),
        thetas=np.stack(thetas), mean=opt.state["__mean"].numpy(), sq=opt.state["__sq_weights"].numpy(),
        deviations=opt.state["__deviations"].numpy(), updates=np.array(opt.state["__updates"]),
        eps=np.concatenate(tape.log), eps_sizes=np.array([a.size for a in tape.log]), samples=np.stack(samples),
        loss_after=np.array(loss_after), theta_after=gm.flat_params(model.parameters()))


def gen_ivon():
    """Reference iVONOptimizer: 3 steps, mc_samples=2, injected noise."""
    steps, S = 3, 2
    torch.manual_seed(9)
    model = gm.make_mlp()
    g = torch.Generator().manual_seed(13)
    D = sum(p.numel() for p in model.parameters())
    init = (0.3 * torch.randn(D, generator=g)).numpy()
    gm.load_flat(model.parameters(), init)
    tape = NoiseTape(43)
    orig_u, orig_i = ref_util.normal_like, ref_ivorn.normal_like
    ref_util.normal_like = tape.like
    ref_ivorn.normal_like = tape.like
    try:
        opt = iVONOptimizer(model.parameters(), lr=1e-2, prior_prec=10.0, dataset_size=768, damping=1e-3,
                            mc_samples=S, augmentation=1.0, tempering=1.0)
        xs, ys = batches(23, steps)
        losses, means, moms, precs = [], [], [], []
        for s in range(steps):
            fwd, bwd = gm.mse_closures(model, xs[s], ys[s])
            losses.append(opt.step(fwd, bwd).item())
            st = [opt.state[p] for p in model.parameters()]
            means.append(torch.cat([t["mean"].reshape(-1) for t in st]).numpy().copy())
            moms.append(torch.cat([t["momentum"].reshape(-1) for t in st]).numpy().copy())
            precs.append(torch.cat([t["precision"].reshape(-1) for t in st]).numpy().copy())
        n_step_noise = len(tape.log)
        opt.sample_parameters()
        sampled = gm.flat_params(model.parameters())
    finally:
        ref_util.normal_like, ref_ivorn.normal_like = orig_u, orig_i
    np.savez_compressed(OUT / "ivon_steps.npz", init=init, xs=xs.numpy(), ys=ys.numpy(), losses=np.array(losses),
                        means=np.stack(means), momenta=np.stack(moms), precisions=np.stack(precs),
                        eps=np.concatenate(tape.log), eps_sizes=np.array([a.size for a in tape.log]),
                        n_step_noise=np.array(n_step_noise), sampled=sampled)


def gen_bbb():
    """Reference BBBOptimizer on a Rank-1 MLP: Gaussian prior KL + L2 on deterministic weights."""
    steps = 3
    torch.manual_seed(15)
    model = gm.Rank1MLP(GaussianParameter)
    g = torch.Generator().manual_seed(17)
    init = {}
    for name, p in model.named_parameters():
        if name.endswith("rho"):
            init[name] = np.full(p.shape, -3.0, dtype=np.float32) + 0.1 * torch.randn(p.shape, generator=g).numpy()
        elif name.endswith("mean"):
            init[name] = (1.0 + 0.1 * torch.randn(p.shape, generator=g)).numpy()
        else:
            init[name] = (0.3 * torch.randn(p.shape, generator=g)).numpy()
    gm.init_rank1(model, init)
    tape = NoiseTape(47)
    orig_u = ref_util.normal_like
    ref_util.normal_like = tape.like
    try:
        prior = GaussianPrior(0.5, 0.8)
        base = torch.optim.Adam(model.parameters(), lr=1e-2)
        opt = BBBOptimizer(model.parameters(), base, prior, dataset_size=100, mc_samples=2, kl_rescaling=0.5,
                           components=1, l2_scale=0.01)
        xs, ys = batches(24, steps)
        losses, states = [], []
        for s in range(steps):
            fwd, bwd = gm.mse_closures(model, xs[s], ys[s])
            losses.append(opt.step(fwd, bwd).item())
            states.append({k: v.detach().numpy().copy() for k, v in model.named_parameters()})
    finally:
        ref_util.normal_like = orig_u
    out = {f"init/{k}": v for k, v in init.items()}
    for s, st in enumerate(states):
        out.update({f"step{s}/{k}": v for k, v in st.items()})
    np.savez_compressed(OUT / "bbb_steps.npz", xs=xs.numpy(), ys=ys.numpy(), losses=np.array(losses),
                        eps=np.concatenate(tape.log), eps_sizes=np.array([a.size for a in tape.log]), **out)


def gen_vectors():
    """Vector-level fixtures from the reference's own primitives (KL, priors, GaussianParameter)."""
    g = torch.Generator().manual_seed(51)
    P = 1237
    out = {}
    gp = GaussianParameter(P)
    with torch.no_grad():
        gp.mean.copy_(0.3 * torch.randn(P, generator=g))
        gp.rho.copy_(-3 + 2.0 * torch.randn(P, generator=g))
        gp.rho[:4] = torch.tensor([25.0, 19.9, 20.1, -30.0])  # softplus threshold / underflow edges
    eps = torch.randn(P, generator=g)
    orig = ref_util.normal_like
    ref_util.normal_like = lambda t: eps.clone()
    try:
        w = gp.sample()
    finally:
        ref_util.normal_like = orig
    gw = torch.randn(P, generator=g)
    w.backward(gw)
    out.update(mu=gp.mean.detach().numpy().copy(), rho=gp.rho.detach().numpy().copy(), eps=eps.numpy().copy(),
               w=w.detach().numpy().copy(), grad_w=gw.numpy().copy(), grad_mu=gp.mean.grad.numpy().copy(),
               grad_rho=gp.rho.grad.numpy().copy())
    gp.mean.grad = None
    gp.rho.grad = None
    prior = GaussianPrior(0.5, 0.8)
    kl = gp.kl_divergence(prior)
    kl.backward()
    out.update(kl_gauss=np.array(kl.item()), kl_gauss_gmu=gp.mean.grad.numpy().copy(),
               kl_gauss_grho=gp.rho.grad.numpy().copy())
    gp.mean.grad = None
    gp.rho.grad = None
    with torch.no_grad():
        gp.mean[:6] = torch.tensor([0.0, 1e-3, 3.0, -7.5, 0.02, 12.0])  # clamp edges of the mixture
    mix = MixturePrior(0.3, 1.0, 0.0025)
    klm = gp.kl_divergence(mix)
    klm.backward()
    out.update(mix_mu=gp.mean.detach().numpy().copy(), kl_mix=np.array(klm.item()), kl_mix_gmu=gp.mean.grad.numpy().copy())
    np.savez_compressed(OUT / "vectors.npz", **out)


def gen_ensemble():
    """DeepEnsemble.predict round-robin (ensemble.py:28-44) over two SVGD members."""
    members, n = 2, 3
    pairs, inits = [], []
    for m in range(members):
        torch.manual_seed(60 + m)
        model = gm.make_mlp()
        g = torch.Generator().manual_seed(70 + m)
        D = sum(p.numel() for p in model.parameters())
        init = (0.3 * torch.randn(n, D, generator=g)).numpy()
        gm.load_flat(model.parameters(), init[0])
        k = {"k": 0}

        def reset(model=model, init=init, k=k):
            k["k"] += 1
            gm.load_flat(model.parameters(), init[k["k"]])

        opt = SVGDOptimizer(model.parameters(), reset, torch.optim.SGD(model.parameters(), lr=0.1), particle_count=n,
                            dataset_size=100)
        pairs.append((model, opt))
        inits.append(init)
    ens = DeepEnsemble(pairs)
    xs, _ = batches(25, 1)
    with torch.no_grad():
        preds = ens.predict(lambda mdl: mdl(xs[0]).squeeze(-1), samples=7)
    np.savez_compressed(OUT / "ensemble_predict.npz", inits=np.stack(inits), x=xs[0].numpy(), preds=preds.numpy())


def gen_ensemble_swag():
    """DeepEnsemble.predict over two SWAG members (ensemble.py:28-44 -> swag.py:53-58): 7 predictions, 4 + 3 draws,
    low-rank / diagonal noise injected at LowRankMultivariateNormal's draw point.  Pins the batched sampler
    (SwagOptimizer.presample, announced by predict) to the reference's one-by-one draws."""
    K, members = 4, 2
    pairs, inits = [], []
    xs, ys = batches(27, 8)
    for m in range(members):
        torch.manual_seed(80 + m)
        model = gm.make_mlp()
        g = torch.Generator().manual_seed(90 + m)
        D = sum(p.numel() for p in model.parameters())
        init = (0.3 * torch.randn(D, generator=g)).numpy()
        gm.load_flat(model.parameters(), init)
        base = torch.optim.SGD(model.parameters(), lr=0.05, momentum=0.9)
        opt = SwagOptimizer(model.parameters(), base, update_interval=1, start_epoch=0, deviation_samples=K)
        for s in range(6):   # 6 updates: the K=4 deviation matrix has rolled
            fwd, bwd = gm.mse_closures(model, xs[s], ys[s])
            opt.step(fwd, bwd)
        pairs.append((model, opt))
        inits.append(init)
    ens = DeepEnsemble(pairs)
    tape = NoiseTape(43)
    import torch.distributions.lowrank_multivariate_normal as lrmn
    orig = lrmn._standard_normal
    lrmn._standard_normal = tape.standard_normal
    try:
        with torch.no_grad():
            preds = ens.predict(lambda mdl: mdl(xs[7]).squeeze(-1), samples=7)
    finally:
        lrmn._standard_normal = orig
    np.savez_compressed(OUT / "ensemble_swag_predict.npz", inits=np.stack(inits), xs=xs.numpy(), ys=ys.numpy(),
                        preds=preds.numpy(), eps=np.concatenate(tape.log), eps_sizes=np.array([a.size for a in tape.log]))


if __name__ == "__main__":
    OUT.mkdir(parents=True, exist_ok=True)
    if len(sys.argv) > 1:  # regenerate selected fixtures only:  python oracle/gen_golden.py gen_svgd_sgd
        for name in sys.argv[1:]:
            globals()[name]()
        sys.exit(0)
    gen_rbf()
    gen_svgd()
    gen_svgd_sgd()
    gen_swag()
    gen_ivon()
    gen_bbb()
    gen_vectors()
    gen_ensemble()
    gen_ensemble_swag()
    for f in sorted(OUT.glob("*.npz")):
        print(f.name, f.stat().st_size)
