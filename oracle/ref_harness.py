"""Import the UNMODIFIED reference (build container only; TEST INFRASTRUCTURE).

The reference is read from /root/reference in the build container and from
``baseline/_ref`` (a verbatim, git-ignored copy made by ``__graft_entry__.build()``)
on the GPU box.  Used by ``oracle/gen_golden.py``, which records the reference's
outputs under tests/golden, and by ``bench.py --impl reference``.  Two shims, both described in SURVEY.md section 8(c):

  * a stub ``gym`` module (``environment.py`` imports gym at module level; only
    ``gym.Wrapper``, ``gym.ObservationWrapper``, ``gym.spaces.Box`` and
    ``gym.make`` are touched at import/def time);
  * ``worker.calculate_mixed_td_errors`` is wrapped so its ``learning_steps``
    argument is int64: the reference accumulates a uint8 running offset
    (worker.py:272-274) which NumPy >= 2 no longer promotes, wrapping at 256.
    The wrapper restores the NumPy-1.x behaviour the code was written for and
    optionally records the raw TD vector (its first argument, worker.py:359).
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_COPY = os.path.join(os.path.dirname(_HERE), "baseline", "_ref")        # verbatim copy made by __graft_entry__.build(); travels to the GPU box
REF_ROOT = os.environ.get("R2D2_REF") or ("/root/reference" if os.path.isfile("/root/reference/worker.py") else _COPY)


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "worker.py"))


_cached = None


def load():
    """Returns a namespace with the reference modules and the TD capture list."""
    global _cached
    if _cached is not None:
        return _cached
    if not available():
        raise RuntimeError(f"reference not found under {REF_ROOT}")

    if "gym" not in sys.modules:
        gym = types.ModuleType("gym")

        class Wrapper:
            def __init__(self, env=None):
                self.env = env

        class ObservationWrapper(Wrapper):
            pass

        spaces = types.ModuleType("gym.spaces")
        spaces.Box = lambda **kw: types.SimpleNamespace(**kw)

        def make(*a, **k):
            raise RuntimeError("gym stub: no emulator in this environment")

        gym.Wrapper, gym.ObservationWrapper, gym.spaces, gym.make = Wrapper, ObservationWrapper, spaces, make
        sys.modules["gym"] = gym
        sys.modules["gym.spaces"] = spaces

    saved = {k: sys.modules.pop(k) for k in ("worker", "model", "priority_tree", "config", "environment")
             if k in sys.modules}
    sys.path.insert(0, REF_ROOT)
    try:
        import config as ref_config            # noqa: E402
        import priority_tree as ref_tree       # noqa: E402
        import model as ref_model              # noqa: E402
        import worker as ref_worker            # noqa: E402
    finally:
        sys.path.remove(REF_ROOT)
    # keep the reference modules reachable only through this namespace
    mods = {k: sys.modules.pop(k) for k in ("worker", "model", "priority_tree", "config", "environment")}
    sys.modules.update(saved)

    captured_td = []
    original = ref_worker.calculate_mixed_td_errors

    def shimmed(td_error, learning_steps):
        captured_td.append(np.array(td_error, copy=True))
        return original(td_error, np.asarray(learning_steps).astype(np.int64))

    ref_worker.calculate_mixed_td_errors = shimmed
    _cached = types.SimpleNamespace(config=ref_config, priority_tree=ref_tree, model=ref_model,
                                    worker=ref_worker, captured_td=captured_td, modules=mods)
    return _cached
