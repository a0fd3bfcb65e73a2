"""Stand-in of the reference's UCI factory: it binds the optimizer classes by name when it is imported, as the
reference's experiment factories do, and builds a DeepEnsemble of small regression models (output [B, 1, 2]: mean
and std) for an algorithm name and a config."""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from golden_models import Rank1Linear
from src.algos.bbb import BBBOptimizer, GaussianPrior
from src.algos.ensemble import DeepEnsemble
from src.algos.ivorn import iVONOptimizer
from src.algos.svgd import SVGDOptimizer
from src.algos.swag import SwagOptimizer
from src.algos.util import GaussianParameter


class GaussOut(nn.Module):
    def forward(self, x):
        return torch.stack((x[:, 0], F.softplus(x[:, 1])), dim=-1).unsqueeze(1)


class BayesLinear(nn.Module):
    def __init__(self, in_features, out_features):
        super().__init__()
        self.weight = GaussianParameter((out_features, in_features))
        self.bias = GaussianParameter(out_features)

    def forward(self, x):
        return F.linear(x, self.weight.sample(), self.bias.sample())


def make_model(name, cfg):
    d = cfg["in_dim"]
    if name == "bbb":
        layers = [BayesLinear(d, 50), nn.ReLU(), BayesLinear(50, 2)]
    elif name == "rank1":
        layers = [Rank1Linear(GaussianParameter, d, 50), nn.ReLU(), Rank1Linear(GaussianParameter, 50, 2)]
    else:
        layers = [nn.Linear(d, 50), nn.ReLU(), nn.Linear(50, 2)]
    model = nn.Sequential(*layers, GaussOut())
    for m in model.modules():
        if isinstance(m, GaussianParameter):
            m.blundell_init()
    return model


def make_optimizer(name, model, cfg):
    opt = cfg["optimizer"]
    if name == "ivon":
        s = opt["ivon"]
        return iVONOptimizer(model.parameters(), s["lr"], s["prior_prec"], s["dataset_size"], damping=s["damping"],
                             mc_samples=s["mc_samples"])
    base = torch.optim.Adam(model.parameters(), **opt["base"])
    if name == "svgd":
        s = opt["svgd"]

        def reset():
            for m in model.modules():
                if isinstance(m, nn.Linear):
                    m.reset_parameters()
        return SVGDOptimizer(model.parameters(), reset, base, s["particle_count"], s["dataset_size"], l2_reg=s["l2_reg"],
                             kernel_grad_scale=s["kernel_grad_scale"])
    if name == "swag":
        s = opt["swag"]
        return SwagOptimizer(model.parameters(), base, s["update_interval"], start_epoch=s["start_epoch"],
                             deviation_samples=s["deviation_samples"])
    s = opt[name]   # bbb / rank1
    return BBBOptimizer(model.parameters(), base, GaussianPrior(0.0, cfg["prior_std"]), s["dataset_size"],
                        mc_samples=s["mc_samples"], kl_rescaling=s["kl_rescaling"], components=s.get("components", 1),
                        l2_scale=s.get("l2_scale", 0))


def get_model(name, config, device):
    pairs = []
    for _ in range(config["members"]):
        model = make_model(name, config).to(device)
        pairs.append((model, make_optimizer(name, model, config)))
    return DeepEnsemble(pairs)
