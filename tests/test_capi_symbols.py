"""CPU: libaogym.so loads and exports every symbol include/aogym.h declares; the ctypes structs
mirror the header (no compute calls -- there is no GPU here)."""
import collections
import ctypes
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'aogym.h')


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as g
    from adaptive_optics_gym_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        g.build()
    return _lib.load()


def declared_symbols():
    src = open(HEADER).read()
    return re.findall(r'AOG_API\s+[\w\s\*]+?\b(aog_\w+)\s*\(', src)


def test_header_declares_the_path():
    syms = declared_symbols()
    for s in ('aog_create', 'aog_destroy', 'aog_set_table', 'aog_reset', 'aog_step', 'aog_step_host',
              'aog_reset_host', 'aog_get_field', 'aog_set_screens', 'aog_generate_screens'):
        assert s in syms


def test_every_declared_symbol_is_exported(lib):
    for s in declared_symbols():
        assert hasattr(lib, s), f'{s} declared in include/aogym.h but not exported by libaogym.so'
    assert b'sm_100a' in lib.aog_version()


def test_each_kernel_is_compiled_once(lib):
    """A header that defines kernels and is included by both translation units builds (and ships) each of them twice:
    every kernel name must appear once in the library's SASS."""
    from adaptive_optics_gym_b200 import _lib
    cuobjdump = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(cuobjdump):
        pytest.skip('cuobjdump not found')
    sass = subprocess.run([cuobjdump, '-sass', _lib.LIB_PATH], check=True, capture_output=True, text=True).stdout
    names = re.findall(r'Function : (\S+)', sass)
    assert names, 'no kernels found in the SASS dump'
    twice = sorted(n for n, k in collections.Counter(names).items() if k > 1)
    assert not twice, f'{len(twice)} kernels compiled more than once: {twice}'


def test_ctypes_structs_mirror_header():
    from adaptive_optics_gym_b200 import _lib
    src = open(HEADER).read()

    def fields(name):
        body = re.search(r'typedef struct %s \{(.*?)\} %s;' % (name, name), src, re.S).group(1)
        body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
        return re.findall(r'(\w+);', body)

    assert [f[0] for f in _lib.AogConfig._fields_] == fields('aog_config')
    assert [f[0] for f in _lib.AogOutputs._fields_] == fields('aog_outputs')
    assert [f[0] for f in _lib.AogCounters._fields_] == fields('aog_counters')
    # table / field ids
    for name, tid in _lib.TABLE_IDS.items():
        m = re.search(r'AOG_TABLE_%s\s*=\s*(\d+)' % name.upper(), src)
        assert m and int(m.group(1)) == tid, name
    for name, fid in _lib.FIELD_IDS.items():
        m = re.search(r'AOG_FIELD_%s\s*=\s*(\d+)' % name.upper(), src)
        assert m and int(m.group(1)) == fid, name
    assert ctypes.sizeof(_lib.AogConfig) == 18 * 4 + 13 * 8 + 8


def test_product_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under the product package may reference it."""
    pkg = os.path.join(ROOT, 'adaptive_optics_gym_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle', txt, re.M), f
    for f in ('gym_AO/__init__.py', 'gym_AO/envs/__init__.py'):
        assert 'oracle' not in open(os.path.join(ROOT, f)).read()
