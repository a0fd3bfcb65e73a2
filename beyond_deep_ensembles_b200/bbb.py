"""Bayes By Backprop / Rank-1 VI optimizer and priors — drop-in for src/algos/bbb.py.

The data term comes from the user's closures (the Bayesian layers sample in their forward);
this optimizer adds the prior term: KL of every Gaussian parameter (K9, value + analytic
gradient in one fused kernel each way, no autograd graph of ~8 eager ops per tensor) and the
L2 penalty of the deterministic parameters (K10), then lets the base optimizer step.
"""
from __future__ import annotations

import torch

from . import dist as bdist
from . import noise, util
from .algo import BayesianOptimizer


class GaussianPrior:
    """N(mu, sigma^2) prior (reference: bbb.py:9-21)."""
    _bde_kind = "gauss"

    def __init__(self, mu, sigma):
        self.mu, self.sigma = mu, sigma
        self.dist = torch.distributions.Normal(mu, sigma)

    def log_prob(self, x):
        return self.dist.log_prob(x)

    def kl_divergence(self, mu2, sigma2):
        """KL(N(mu2, sigma2^2) || prior) summed over all entries, from (mean, std) TENSORS.
        API compatibility for the activation-space layers of bbb_layers.py (outside the optimizer
        path); BBBOptimizer itself goes through GaussianParameter.kl_divergence -> K9."""
        ratio = sigma2 / self.sigma
        shift = (self.mu - mu2) / self.sigma
        per_entry = 0.5 * (2 * torch.log(self.sigma / sigma2) - 1 + ratio.pow(2) + shift.pow(2))
        return per_entry.sum()


class MixturePrior:
    """Scale mixture of two zero-mean Gaussians (reference: bbb.py:23-37); each component's
    log-density is clamped to [-23, 0] before the mixture is formed, as there."""
    _bde_kind = "mixture"

    def __init__(self, pi, sigma1, sigma2, validate_args=None):
        self.pi = torch.tensor(pi)
        self.sigma1, self.sigma2 = sigma1, sigma2
        self.dist1 = torch.distributions.Normal(0, sigma1, validate_args)
        self.dist2 = torch.distributions.Normal(0, sigma2, validate_args)

    def log_prob(self, value):
        weights = (torch.log(self.pi), torch.log(1 - self.pi))
        parts = [w + torch.clamp(d.log_prob(value), -23, 0) for w, d in zip(weights, (self.dist1, self.dist2))]
        return torch.logaddexp(parts[0], parts[1])

    def kl_divergence(self, mu2, sigma2):
        # a point estimate: minus the log-density of the means; sigma2 is ignored (bbb.py:36-37)
        return -self.log_prob(mu2).sum()


def collect_kl(model) -> torch.Tensor:
    """Sum of the `kl` attributes over the module tree below `model` (bbb.py:39-40)."""
    total = 0
    for layer in model.children():
        total = total + getattr(layer, "kl", 0) + collect_kl(layer)
    return total


class BBBOptimizer(BayesianOptimizer):
    """Bayes By Backprop (reference: bbb.py:43-99); use Bayesian layers built on
    util.GaussianParameter for the layers that should be treated as Bayesian."""

    def __init__(self, params, base_optimizer, prior, dataset_size, mc_samples=1, kl_rescaling=1, components=1,
                 l2_scale=0, process_group=None):
        """`process_group` (extension, default None = like the reference): the torch.distributed group whose ranks
        each hold a COLUMN SLICE of every parameter (SURVEY.md §8e).  Sampling, the KL / L2 gradients and the base
        optimizer stay local; the group (i) places every Gaussian tensor's slice in the job-wide Philox stream, so
        the ranks draw disjoint noise, and (ii) sums the prior term's VALUE (one scalar all-reduce; only the logged
        loss needs it — each rank differentiates its own slice)."""
        defaults = {"prior": prior, "l2_scale": l2_scale}
        super().__init__(params, defaults)
        self.state["__base_optimizer"] = base_optimizer
        self.mc_samples = mc_samples
        self.kl_rescaling = kl_rescaling
        self.components = components
        self.dataset_size = dataset_size
        self._group = bdist.SINGLE if process_group is None else process_group
        if bdist.world(self._group) > 1:
            self._place_gaussian_slices()

    def _place_gaussian_slices(self):
        """Collective (one all_gather_object): per Gaussian tensor, the exclusive prefix over the ranks of the
        slice lengths (rounded up to whole Philox quads) becomes the owner's `column_offset`."""
        import torch.distributed as dist
        owners = []
        for param in self._params():
            owner = getattr(getattr(param, "get_parameter_kl", None), "__self__", None)
            if owner is not None and hasattr(owner, "column_offset") and getattr(owner, "mean", None) is param:
                owners.append(owner)
        world, rank = bdist.world(self._group), dist.get_rank(self._group)
        rows = [None] * world
        mine = ([(o.mean.numel() + 3) // 4 * 4 for o in owners], noise.seed(), noise.stream_position())
        dist.all_gather_object(rows, mine, group=self._group)
        if any(len(r[0]) != len(owners) for r in rows):
            raise ValueError("the ranks of a D-sharded BBB optimizer hold different numbers of Gaussian tensors")
        noise.restore_stream_position(max(r[2] for r in rows))
        for k, owner in enumerate(owners):
            owner.column_offset = sum(r[0][k] for r in rows[:rank])
            owner.noise_seed = int(rows[0][1])

    def step(self, forward_closure, backward_closure, grad_scaler=None):
        if grad_scaler is not None:
            # grad_scaler.step(base) runs the scaler's own unscale_, which a ShardedGradScaler agrees over the group
            self._refuse_scaler_if_sharded(grad_scaler, bdist.world(self._group), self._group)
        base = self.state["__base_optimizer"]
        base.zero_grad()

        total_data_loss = None
        for _ in range(self.mc_samples):
            if total_data_loss is None:
                total_data_loss = forward_closure()
            else:
                total_data_loss += forward_closure()

        # KL and L2 are collected once per step (bbb.py:69-76).  Every tensor the fused kernels understand
        # goes into ONE multi-tensor launch per prior (value) + one in backward (all gradients); anything
        # else — a foreign prior object, a parameter whose KL is a user-supplied callable, non-contiguous
        # storage — is evaluated per tensor through its own get_parameter_kl.
        total_kl_loss = torch.zeros((), device=self._params_device())   # no host-to-device copy
        batches = {}   # id(prior) -> (prior, [(mean, rho)])
        deterministic = []
        for group in self.param_groups:
            l2_scale = group["l2_scale"]
            prior = group["prior"]
            for param in group["params"]:
                if hasattr(param, "get_parameter_kl"):
                    pair = self._gaussian_pair(param, prior) if self.batch_prior_terms else None
                    if pair is None:
                        total_kl_loss += param.get_parameter_kl(prior)
                    else:
                        batches.setdefault(id(prior), (prior, []))[1].append(pair)
                elif not getattr(param, "_is_gaussian_mean", False) and not getattr(param, "_is_gaussian_rho", False):
                    # the reference adds 0 * ||theta||^2 when l2_scale == 0; skipping the pass over
                    # D parameters is identical for finite weights
                    if l2_scale != 0:
                        if self.batch_prior_terms and param.is_contiguous() and param.dtype == torch.float32:
                            deterministic.append((param, l2_scale))
                        else:
                            total_kl_loss += util.l2_penalty(param, l2_scale)
        for prior, pairs in batches.values():
            total_kl_loss += util.prior_terms(pairs, prior, deterministic)
            deterministic = []
        if deterministic:
            total_kl_loss += util.prior_terms([], None, deterministic)

        # D-sharded: the other ranks' share of the prior term, as a value (no gradient crosses ranks)
        total_kl_loss = bdist.allreduce_scalar_value(total_kl_loss, self._group)

        pi = self.kl_rescaling / self.dataset_size
        # the KL is not divided by the MC sample count: it was collected once (bbb.py:79-80)
        loss = pi * total_kl_loss + total_data_loss / (self.mc_samples * self.components)
        if not loss.isnan().any():
            backward_closure(loss)

            if grad_scaler is not None:
                grad_scaler.step(base)
            else:
                base.step()

        return loss

    # one launch for the whole prior term (class attribute; False: one K9 / K10 launch per tensor)
    batch_prior_terms = True

    @staticmethod
    def _gaussian_pair(mean_param, prior):
        """(mean, rho) when `mean_param` belongs to a GaussianParameter whose KL against `prior` is the
        stock one (util.gaussian_kl), else None."""
        owner = getattr(mean_param.get_parameter_kl, "__self__", None)
        rho = getattr(owner, "rho", None)
        if rho is None or getattr(owner, "mean", None) is not mean_param or util.prior_kind(prior) is None:
            return None
        func = getattr(mean_param.get_parameter_kl, "__func__", None)
        if func is not getattr(type(owner), "kl_divergence", None) or not getattr(type(owner), "_bde_fused_kl", False):
            return None
        if not (mean_param.is_contiguous() and rho.is_contiguous() and rho.shape == mean_param.shape
                and mean_param.dtype == torch.float32 and rho.dtype == torch.float32):
            return None
        return mean_param, rho

    def sample_parameters(self):
        """The Bayesian layers sample in their forward pass (bbb.py:92-96)."""
        pass

    def get_base_optimizer(self):
        return self.state["__base_optimizer"]
