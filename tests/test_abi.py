"""CPU-side checks of the drop-in boundary: the shared library loads and exports exactly
the entry points include/elfi_b200.h declares (no compute calls: no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    text = open(os.path.join(ROOT, 'include', 'elfi_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(elfi_b200_\w+)\s*\(', text)))


def test_header_declares_functions():
    names = header_functions()
    assert 'elfi_b200_ctx_create' in names
    assert 'elfi_b200_dist_euclid_thr_f64' in names
    assert len(names) >= 6


def test_library_exports_every_header_symbol():
    from elfi_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    missing = [n for n in header_functions() if not hasattr(lib, n)]
    assert not missing, 'declared in include/elfi_b200.h but not exported: {}'.format(missing)


def test_binding_covers_header():
    from elfi_b200 import _lib
    assert sorted(_lib.SIGNATURES) == header_functions()
    lib = _lib.load()
    assert lib.elfi_b200_version() == 100


def test_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    from elfi_b200 import _lib, ops
    import numpy as np
    with pytest.raises(_lib.ElfiB200Error):
        ops.dist_euclid(np.zeros((4, 2)), np.zeros(2))


def test_product_never_imports_oracle():
    """The product path must not route through the CPU oracle (or the reference)."""
    pkg = os.path.join(ROOT, 'elfi_b200')
    bad = []
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                if re.search(r'^\s*(import|from)\s+(elfi_oracle|oracle|ref_shim)\b', src, re.M):
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad


def test_library_reads_no_environment():
    """What the CUDA library computes depends on its arguments only, never on environment
    variables of the process that loads it."""
    bad = []
    for top in (os.path.join(ROOT, 'elfi_b200', 'csrc'), os.path.join(ROOT, 'include')):
        for dirpath, _, files in os.walk(top):
            for f in files:
                if 'getenv' in open(os.path.join(dirpath, f), errors='replace').read():
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad
