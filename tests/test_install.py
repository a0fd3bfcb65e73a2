"""install(): an experiment factory that binds the optimizer classes by name at import builds this package's
optimizers once install() has rebound those names inside the reference's modules, without any edit to them.  The
reference checkout is replaced by tests/reference_standin: the module layout install() patches, with placeholders that
fail when used, and a UCI factory.  Runs in a subprocess because it rebinds names inside those modules; the C-ABI is
the oracle-backed double (CPU)."""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
STANDIN = ROOT / "tests" / "reference_standin"

SCRIPT = r'''
import sys, torch
sys.path.insert(0, "ROOT"); sys.path.insert(0, "ROOT/tests")
import fake_abi
class P:
    def setattr(self, o, n, v): setattr(o, n, v)
fake_abi.install(P())
import beyond_deep_ensembles_b200 as bde
patched = bde.install("STANDIN")
assert "src.algos.svgd.SVGDOptimizer" in patched and "src.algos.ivorn.iVONOptimizer" in patched, patched
from experiments.uci.models import get_model          # the factory, imported AFTER install()
from src.algos.util import GaussianParameter
assert GaussianParameter._bde_fused_kl                 # patched in place: the layers hold the class itself
torch.manual_seed(0)
x, y = torch.randn(32, 8), torch.randn(32)
base = {"in_dim": 8, "std_init": 1.0, "learn_var": False, "members": 2, "prior_std": 1.0}
cfgs = {
    "svgd": {"optimizer": {"base": {"lr": 1e-3, "weight_decay": 0},
                           "svgd": {"particle_count": 5, "l2_reg": 0.01, "dataset_size": 768, "kernel_grad_scale": 1.0}}},
    "swag": {"optimizer": {"base": {"lr": 1e-3}, "swag": {"start_epoch": 0, "update_interval": 1, "deviation_samples": 5}}},
    "ivon": {"optimizer": {"ivon": {"lr": 1e-3, "prior_prec": 1.0, "dataset_size": 768, "damping": 1e-3, "mc_samples": 2}}},
    "rank1": {"optimizer": {"base": {"lr": 1e-3}, "rank1": {"mc_samples": 2, "kl_rescaling": 1.0, "dataset_size": 768,
                                                             "components": 1, "l2_scale": 0.1}}},
    "bbb": {"optimizer": {"base": {"lr": 1e-3}, "bbb": {"mc_samples": 2, "kl_rescaling": 1.0, "dataset_size": 768}}},
}
expect = {"svgd": bde.SVGDOptimizer, "swag": bde.SwagOptimizer, "ivon": bde.iVONOptimizer, "rank1": bde.BBBOptimizer,
          "bbb": bde.BBBOptimizer}
for name, extra in cfgs.items():
    ens = get_model(name, {**base, **extra}, "cpu")
    assert type(ens) is bde.DeepEnsemble and len(ens.models) == 2
    for model, opt in ens.models_and_optimizers:
        assert type(opt) is expect[name], (name, type(opt))
        def fwd():
            out = model(x)                      # [32, 1, 2]: mean and std from the reference's GaussLayer
            return ((out[..., 0].squeeze(-1) - y) ** 2).mean()
        l0 = opt.step(fwd, lambda l: l.backward())
        opt.complete_epoch()
        l1 = opt.step(fwd, lambda l: l.backward())
        assert torch.isfinite(l0) and torch.isfinite(l1), name
    with torch.no_grad():
        preds = ens.predict(lambda m: m(x)[..., 0], samples=4)
    assert preds.shape[0] == 4
    sd = ens.state_dict(); ens.load_state_dict(sd)
print("INSTALL_OK")
'''


def test_reference_factories_build_b200_optimizers():
    script = SCRIPT.replace("ROOT", str(ROOT)).replace("STANDIN", str(STANDIN))
    res = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "INSTALL_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
