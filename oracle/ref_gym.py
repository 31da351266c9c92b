"""Import the REAL reference (openai/gym 0.26.2) for parity tests and CPU timing.  Test infrastructure only.

Looks for the installed copy ``oracle/_ref`` (built by ``oracle/make_ref.py`` where the reference's source is
available; the tests that need it skip without it).  The frozen reference predates
numpy 2: two aliases it still uses (``np.bool8``: gym/utils/passive_env_checker.py:225, ``np.float_``:
gym/envs/classic_control/acrobot.py:446) are added to the numpy module, outside the reference tree (SURVEY.md
Appendix D).
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
INSTALLED = os.path.join(HERE, "_ref")


def reference_path():
    return INSTALLED if os.path.isfile(os.path.join(INSTALLED, "gym", "version.py")) else None


def import_reference():
    """-> the reference's ``gym`` module (asserts 0.26.2); raises ImportError when no copy is available."""
    path = reference_path()
    if path is None:
        raise ImportError("the reference is not installed in oracle/_ref (python oracle/make_ref.py)")
    for name, value in (("bool8", np.bool_), ("float_", np.float64)):
        if not hasattr(np, name):
            setattr(np, name, value)
    if path not in sys.path:
        sys.path.insert(0, path)
    warnings.filterwarnings("ignore")
    import gym
    assert gym.__version__ == "0.26.2", gym.__version__
    assert os.path.abspath(gym.__file__).startswith(os.path.abspath(path)), gym.__file__
    return gym
