"""B200-native rollout hot path of the Decision-Pretrained Transformer (sm_100a only).

Python mirror of the reference's env / controller / rollout interface over libdpt_b200.so
(hand-written CUDA behind the C ABI in include/dpt_b200.h).  There is no CPU fallback.
"""
import importlib
import sys

from . import _lib, rng, kernels          # noqa: F401
from .rng import seed                     # noqa: F401
from . import envs, collect_data          # noqa: F401
from .envs import base_env, bandit_env, gpu_bandit_env, darkroom_env   # noqa: F401
from . import ctrls, evals                # noqa: F401
from .ctrls import ctrl_bandit, ctrl_darkroom   # noqa: F401
from .evals import eval_bandit, eval_linear_bandit, eval_darkroom, eval_interactive_bandit   # noqa: F401
from . import models, dataset             # noqa: F401
from .models import net                   # noqa: F401
from . import train                       # noqa: F401

__all__ = ["seed", "kernels", "envs", "collect_data", "install_dropin"]

_DROPIN = ("envs", "ctrls", "evals", "models", "collect_data", "dataset", "utils")


def install_dropin():
    """Expose the reference's top-level module names (``envs.bandit_env``, ``collect_data``,
    ``ctrls.ctrl_bandit``, ``evals.eval_bandit``, ``models.net``) so reference call sites such as
    ``from envs.bandit_env import BanditEnvVec`` resolve to this package."""
    pkg = sys.modules[__name__]
    for name in _DROPIN:
        try:
            mod = importlib.import_module("." + name, __name__)
        except ImportError:
            continue
        sys.modules[name] = mod
        for sub, m in list(sys.modules.items()):
            if sub.startswith(__name__ + "." + name + "."):
                sys.modules[name + sub[len(__name__ + "." + name):]] = m
    return pkg
