"""Placeholders of the stand-in reference.  Every class install() rebinds fails when constructed, so a factory that
still reaches one of them after install() fails loudly.  GaussianParameter keeps the reference's interface (mean /
rho with std = softplus(rho), the markers BBBOptimizer reads) because install() patches its methods in place
instead of replacing the class: the layers hold the class object itself."""
from __future__ import annotations

import torch
import torch.nn as nn


class Unpatched:
    def __init__(self, *args, **kwargs):
        raise AssertionError(f"stand-in {type(self).__name__} constructed: install() did not rebind it")


class GaussianParameter(nn.Module):
    def __init__(self, size):
        super().__init__()
        self.overwrite_mean(torch.empty(size))
        self.rho = nn.Parameter(torch.empty(size))
        self.rho._is_gaussian_rho = True

    def blundell_init(self, mean_std=0.1):
        nn.init.normal_(self.mean, 0, mean_std)
        nn.init.constant_(self.rho, -3)

    def sample(self):
        raise AssertionError("stand-in GaussianParameter.sample called: install() did not patch it")

    def kl_divergence(self, prior):
        raise AssertionError("stand-in GaussianParameter.kl_divergence called: install() did not patch it")

    def overwrite_mean(self, mean):
        self.mean = nn.Parameter(mean)
        self.mean.get_parameter_kl = self.kl_divergence
        self.mean._is_gaussian_mean = True
