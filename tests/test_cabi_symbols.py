"""-m "not gpu": librenet_b200.so builds for sm_100a, loads, and exports every symbol include/renet_b200.h
declares (no compute calls here -- there is no GPU in the authoring container)."""
import ctypes
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def so_path():
    from renet_b200 import build
    return build.build()


def _declared():
    txt = open(os.path.join(ROOT, 'include', 'renet_b200.h')).read()
    txt = re.sub(r'/\*.*?\*/', '', txt, flags=re.S)
    return sorted(set(re.findall(r'\b(renet_[a-z0-9_]+)\s*\(', txt)))


def test_header_symbols_exported(so_path):
    names = _declared()
    assert len(names) >= 12
    lib = ctypes.CDLL(so_path)
    for n in names:
        assert hasattr(lib, n), 'missing export: ' + n


def test_python_binding_covers_header(so_path):
    from renet_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared()
    L = _lib.lib()
    assert L.renet_version() >= 100
    assert L.renet_last_error() == b''
    assert L.renet_csr_workspace_bytes(1000, 5000) > 0          # host-only size query
    assert L.renet_gru_workspace_bytes(100, 10, 5, 200) > 0


def test_argument_validation_needs_no_gpu(so_path):
    from renet_b200 import _lib
    L = _lib.lib()
    rc = L.renet_rgcn_block_fwd(None, None, None, None, None, None, None, None, None, 10, 5, 200, 200, 7, 4, 1, None)
    assert rc == -1 and b'num_bases' in L.renet_last_error()
    rc = L.renet_rgcn_block_fwd(None, None, None, None, None, None, None, None, None, 10, 5, 200, 200, 100, 4, 1, None)
    assert rc == -1 and b'null pointer' in L.renet_last_error()


def test_sass_is_sm100a(so_path):
    from renet_b200 import build
    cuobjdump = os.path.join(os.path.dirname(build.NVCC), 'cuobjdump')     # the toolkit that built the library
    out = subprocess.run([cuobjdump, '-lelf', so_path], capture_output=True, text=True).stdout
    assert 'sm_100a' in out, out


def test_hot_path_never_imports_oracle():
    pkg = os.path.join(ROOT, 'renet_b200')
    for f in os.listdir(pkg):
        if f.endswith('.py'):
            src = open(os.path.join(pkg, f)).read()
            assert not re.search(r'^\s*(from|import)\s+oracle', src, flags=re.M), f


def test_missing_library_fails_loudly(tmp_path, monkeypatch):
    from renet_b200 import _lib
    monkeypatch.setattr(_lib, '_lib', None)
    monkeypatch.setattr(_lib, 'LIB_PATH', str(tmp_path / 'nope.so'))
    with pytest.raises(RuntimeError, match='no CPU or PyTorch fallback'):
        _lib.lib()
