"""attack_vc_b200 -- B200-native (sm_100a) adversarial perturbation loop of attack-vc.

Only the hot path lives here: ``csrc/`` (CUDA kernels + the C-ABI of include/avc_b200.h) and the
host-side mirror of the reference's attack interface (``engine.Engine``; the drop-in module is the
top-level ``attack_utils.py``).  Importing this package never falls back to PyTorch math: if
``libavc_b200.so`` is missing, using it raises."""
from .engine import AvcError, Engine, engine_for, invalidate_engine  # noqa: F401
from .defend import Defender  # noqa: F401,E402

__all__ = ["Engine", "AvcError", "engine_for", "invalidate_engine", "Defender"]
