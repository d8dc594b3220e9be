"""compat/: the top-level `models`, `utils`, `gpytorch`, `pymc3` names the reference's experiment drivers import resolve to
the B200-native mirrors (SURVEY.md 8(b), 8(f)4).  Import-only: no GPU is touched."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# what the reference's experiments/{spatial_exp,spatio_temporal_exp,deepgp_spatial_bench}.py import from these packages
# (spatial_exp.py:21-27, spatio_temporal_exp.py:18-24, deepgp_spatial_bench.py:10-20)
WANTED = {
    "gpytorch.kernels": ["ScaleKernel", "RBFKernel", "PeriodicKernel", "InducingPointKernel"],
    "gpytorch.constraints": ["GreaterThan"],
    "gpytorch.mlls": ["VariationalELBO", "AddedLossTerm", "DeepApproximateMLL", "ExactMarginalLogLikelihood"],
    "gpytorch.models": ["ExactGP"],
    "gpytorch.likelihoods": ["GaussianLikelihood"],
    "gpytorch.distributions": ["MultivariateNormal"],
    "models.gibbs_kernels": ["LogNormalPriorProcess", "PositivePriorProcess", "GibbsKernel", "GibbsSafeScaleKernel",
                             "InducingGibbsKernel", "InducingGibbsKernelST"],
    "models.nonstationary_models": ["DiagonalSparseGP", "DiagonalExactGP"],
    "models.spatio_temporal_models": ["SparseSpatioTemporal_Nonstationary"],
    "models.dgps": ["DeepGPHiddenLayer", "DeepGP"],
    "models.multivariate_gibbs_kernel": ["MultivariateGibbsKernel"],
    "models.sparse_multivariate_gibbs_kernel": ["SparseMultivariateGibbsKernel"],
    "models.latent_priors": ["MatrixVariateNormalPrior"],
    "utils.config": ["BASE_SEED", "EPSILON", "DATASET_DIR", "RESULTS_DIR"],
    "utils.metrics": ["rmse", "nlpd", "negative_log_predictive_density", "get_trainable_param_names"],
    "utils.metrics2": ["nlpd", "rmse"],
    "utils.dataprep": ["download_data", "prep_inputs", "prep_outputs", "whitening_transform", "train_test_split"],
    "utils.functional": ["op", "dot", "mv", "t"],
    "pymc3.gp.util": ["kmeans_inducing_points"],
}


def _run(code):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "compat"),
                                                       os.path.join(ROOT, "compat", "optional_stubs")]))
    return subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)


def test_top_level_names_resolve_to_the_mirrors():
    code = "import importlib, json, sys\nwanted = %r\nmissing = []\n" % WANTED + (
        "for mod, names in wanted.items():\n"
        "    m = importlib.import_module(mod)\n"
        "    missing += [mod + '.' + n for n in names if not hasattr(m, n)]\n"
        "import models.gibbs_kernels as g, nonstationary_precip_b200.models.gibbs_kernels as h\n"
        "assert g.GibbsKernel is h.GibbsKernel\n"
        "import gpytorch\nassert issubclass(g.GibbsKernel, gpytorch.kernels.Kernel)\n"
        "print(json.dumps(missing))\n")
    r = _run(code)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip().splitlines()[-1] == "[]", r.stdout


# module-top import forms beyond `from pkg.mod import names`: bare, aliased and star imports of the shims, and every
# submodule of the inert plotting / table stand-ins in compat/optional_stubs
IMPORT_FORMS = """
import gpytorch
import pymc3 as pm
import models.gibbs_kernels as gk
from models.nonstationary_models import *
from utils.metrics import *
import cartopy
import cartopy.crs as ccrs
import cartopy.feature as cfeature
import matplotlib
import matplotlib.pyplot as plt
import matplotlib.pylab as pylab
from matplotlib import cm, colors
from prettytable import PrettyTable
"""


def test_bare_aliased_star_and_stubbed_imports_execute():
    code = IMPORT_FORMS + (
        "import nonstationary_precip_b200.models.nonstationary_models as nm, nonstationary_precip_b200.utils as nu\n"
        "assert pm.gp.util.kmeans_inducing_points is nu.dataprep.kmeans_inducing_points\n"
        "assert DiagonalSparseGP is nm.DiagonalSparseGP and DiagonalExactGP is nm.DiagonalExactGP\n"
        "assert rmse is nu.metrics.rmse and nlpd is nu.metrics.nlpd\n"
        "assert issubclass(gk.GibbsKernel, gpytorch.kernels.Kernel)\n"
        "for use in (lambda: plt.figure(), lambda: ccrs.PlateCarree(), lambda: cfeature.BORDERS.with_scale('10m'),\n"
        "            lambda: pylab.show(), lambda: cm.get_cmap('viridis'), lambda: colors.Normalize()):\n"
        "    try:\n"
        "        use()\n"
        "    except RuntimeError as e:\n"
        "        assert 'stub' in str(e)\n"
        "    else:\n"
        "        raise AssertionError('a plotting stub did something')\n"
        "t = PrettyTable(['Modules', 'Parameters'])\n"
        "t.add_row(['m', 3])\n"
        "assert 'Modules' in str(t) and 'm | 3' in str(t)\n"
        "print('ok')\n")
    r = _run(code)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stderr[-3000:]
