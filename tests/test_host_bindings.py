"""CPU: the ctypes binding in kwiiyatta_b200/_lib.py, without loading the library."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from kwiiyatta_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCALARS = {'int': ctypes.c_int, 'int64_t': ctypes.c_int64, 'size_t': ctypes.c_size_t,
           'double': ctypes.c_double}


def _ctype(decl, is_return):
    """ctypes type of a C declaration (a return type, or a parameter with its name)."""
    words = decl.replace('*', ' * ').split()
    words = [w for w in words if w != 'const']
    if '*' in words:
        return ctypes.c_char_p if is_return and words[0] == 'char' else ctypes.c_void_p
    base = words[0]
    assert base in SCALARS, f'no ctypes mapping for {decl!r}'
    return SCALARS[base]


def header_prototypes():
    """{name: (restype, [argtypes])} of every kw_* prototype in include/kwiiyatta_b200.h."""
    with open(os.path.join(ROOT, 'include', 'kwiiyatta_b200.h')) as f:
        text = f.read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    text = re.sub(r'^\s*#.*$', '', text, flags=re.M)
    protos = {}
    for stmt in text.split(';'):
        m = re.search(r'(\w[\w\s*]*?)\b(kw_\w+)\s*\(([^()]*)\)\s*$', stmt)
        if m is None:
            continue
        ret, name, params = m.groups()
        params = [p.strip() for p in params.split(',')]
        args = [] if params == ['void'] else [_ctype(p, False) for p in params]
        protos[name] = (_ctype(ret, True), args)
    return protos


def test_signatures_match_header_types():
    protos = header_prototypes()
    assert len(protos) >= 30, sorted(protos)
    assert set(protos) == set(_lib.SIGNATURES), set(protos) ^ set(_lib.SIGNATURES)
    for name, (res, args) in protos.items():
        got_res, got_args = _lib.SIGNATURES[name]
        assert got_res is res, f'{name}: return type {got_res} in SIGNATURES, {res} in the header'
        assert list(got_args) == args, f'{name}: arguments {got_args} in SIGNATURES, {args} in ' \
            'the header'


class _FakeLib:
    """Stands in for the loaded library: records the arguments of ``kw_probe``."""

    def __init__(self, rc):
        self.rc, self.args = rc, None

    def kw_probe(self, *args):
        self.args = args
        return self.rc

    def kw_last_error(self):
        return b'the probe says no'


@pytest.fixture
def fake_lib(monkeypatch):
    def install(rc):
        fake = _FakeLib(rc)
        monkeypatch.setattr(_lib, 'lib', lambda: fake)
        return fake
    return install


def test_call_passes_buffers_as_pointers_and_scalars_as_themselves(fake_lib):
    fake = fake_lib(0)
    t = torch.zeros(3, dtype=torch.float64)
    a = np.zeros(4, dtype=np.int32)
    assert _lib.call('kw_probe', t, a, None, 7, 2.5, True) is None
    assert fake.args == (t.data_ptr(), a.ctypes.data, None, 7, 2.5, True)
    assert all(type(x) is int for x in fake.args[:2])


@pytest.mark.parametrize('rc, exc', [(_lib.KW_ERR_INVALID, ValueError),
                                     (_lib.KW_ERR_UNSUPPORTED, NotImplementedError),
                                     (_lib.KW_ERR_WORKSPACE, _lib.KwError),
                                     (_lib.KW_ERR_CUDA, _lib.KwError)])
def test_call_raises_on_a_failed_status(fake_lib, rc, exc):
    fake_lib(rc)
    with pytest.raises(exc) as info:
        _lib.call('kw_probe', 1)
    assert type(info.value) is exc
    assert str(info.value) == f'kw_probe failed ({rc}): the probe says no'
