"""Import the UNMODIFIED reference (elfi-dev/elfi v0.8.7): from the checkout that the environment
variable ELFI_REFERENCE points to (the directory holding its `elfi/` package) if it is set, else
from the copy in oracle/_ref/ that `make -C oracle` (run by __graft_entry__.build()) makes when a
checkout is present.  It is not part of this repository; without it the reference-driven tests
skip and the committed goldens stand in.

TEST / BASELINE INFRASTRUCTURE ONLY.  Used by tests/golden/gen_golden*.py to produce the
committed golden fixtures, by the reference-driven plugin tests and by ``bench.py --impl
reference`` (the CPU arm); never imported by the product (`elfi_b200/`).

The reference needs packages that are absent here (matplotlib, GPy, arviz, numdifftools,
ipyparallel, dask, toolz) and uses NumPy-1 aliases; none of them touch the sampler hot
path, so they are stubbed (SURVEY.md §8c recipe).
"""
import sys
import types
from unittest.mock import MagicMock

import numpy as np

import os

REFERENCE_ROOT = os.path.abspath(os.environ['ELFI_REFERENCE']) if os.environ.get('ELFI_REFERENCE') \
    else os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')


def reference_available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, 'elfi'))


def import_reference():
    """Return the reference `elfi` module (import it on first call)."""
    if not reference_available():
        raise ImportError('the reference ELFI package was not found in {}: build with a checkout '
                          'of elfi-dev/elfi present, or set ELFI_REFERENCE'.format(REFERENCE_ROOT))
    if 'elfi' in sys.modules and getattr(sys.modules['elfi'], '__file__', '').startswith(
            REFERENCE_ROOT):
        return sys.modules['elfi']
    for name in ['matplotlib', 'matplotlib.pyplot', 'matplotlib.colors', 'matplotlib.axes',
                 'GPy', 'GPy.kern', 'GPy.models', 'GPy.priors', 'arviz', 'numdifftools',
                 'ipyparallel', 'dask', 'dask.distributed']:
        sys.modules.setdefault(name, MagicMock())
    if 'toolz' not in sys.modules:
        toolz = types.ModuleType('toolz')
        functoolz = types.ModuleType('toolz.functoolz')

        def compose(*funcs):
            def composed(*a, **k):
                out = funcs[-1](*a, **k)
                for f in reversed(funcs[:-1]):
                    out = f(out)
                return out
            return composed
        functoolz.compose = compose
        toolz.functoolz = functoolz
        toolz.compose = compose
        sys.modules['toolz'] = toolz
        sys.modules['toolz.functoolz'] = functoolz
    if not hasattr(np, 'Inf'):
        np.Inf = np.inf
    if not hasattr(np, 'float_'):
        np.float_ = np.float64
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import elfi
    return elfi
