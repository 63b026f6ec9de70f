"""The C-ABI library loads and exports every symbol include/p3d.h declares (no compute: runs without a GPU)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


def header_source():
    """include/p3d.h without comments and preprocessor lines."""
    src = open(os.path.join(ROOT, 'include', 'p3d.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return re.sub(r'^[ \t]*#.*$', '', src, flags=re.M)


def declared_symbols():
    return sorted(set(re.findall(r'\b(p3d_[a-z0-9_]+)\s*\(', header_source())))


# the kind of a value at the ABI: what has to agree between a C declaration and its ctypes mirror
_C_KINDS = {'int': 'i32', 'int32_t': 'i32', 'int64_t': 'i64', 'uint32_t': 'u32', 'int8_t': 'i8', 'float': 'f32', 'double': 'f64'}
_CTYPES_KINDS = {ctypes.c_int32: 'i32', ctypes.c_int64: 'i64', ctypes.c_uint32: 'u32', ctypes.c_int8: 'i8', ctypes.c_float: 'f32',
                 ctypes.c_double: 'f64'}


def c_declarators(decl):
    """'const float* a, b[2]' -> [('a', 'ptr', None), ('b', 'f32', 2)]. Pointers and p3d_stream_t are 'ptr'."""
    base, rest = re.fullmatch(r'\s*((?:unsigned\s+)?\w+)(.*)', re.sub(r'\bconst\b', '', decl), flags=re.S).groups()
    out = []
    for part in rest.split(','):
        stars, name, n = re.fullmatch(r'\s*(\**)\s*(\w+)\s*(?:\[(\d+)\])?\s*', part).groups()
        kind = 'ptr' if (stars or base == 'p3d_stream_t') else _C_KINDS[base]
        out.append((name, kind, None if n is None else int(n)))
    return out


def ctypes_kind(t):
    if t in (ctypes.c_void_p, ctypes.c_char_p) or issubclass(t, ctypes._Pointer):
        return 'ptr'
    return _CTYPES_KINDS[t]


def header_prototypes():
    """name -> (return kind, parameter kinds, whether the last parameter is the stream) for every p3d_* prototype of the
    header; an array parameter is a pointer."""
    protos = {}
    for ret, name, params in re.findall(r'([\w\s*]+?)\b(p3d_\w+)\s*\(([^)]*)\)\s*;', header_source()):
        ret = re.sub(r'\bconst\b', '', ret).strip()
        params = [] if params.strip() == 'void' else params.split(',')
        kinds = ['ptr' if n else kind for p in params for _, kind, n in c_declarators(p)]
        protos[name] = ('ptr' if '*' in ret else _C_KINDS[ret], kinds, bool(params) and 'p3d_stream_t' in params[-1])
    return protos


def header_structs():
    """name -> [(field, kind, array length or None)] for every `typedef struct {...} p3d_*_t;` of the header."""
    return {name: [f for decl in body.split(';') if decl.strip() for f in c_declarators(decl)]
            for body, name in re.findall(r'typedef\s+struct\s*\{(.*?)\}\s*(p3d_\w+_t)\s*;', header_source(), flags=re.S)}


def test_header_declares_entry_points():
    syms = declared_symbols()
    for must in ('p3d_render_fwd', 'p3d_bias_act', 'p3d_upfirdn2d', 'p3d_ray_sampler', 'p3d_run_model'):
        assert must in syms


def test_library_exports_all_declared_symbols():
    from pix2pix3d_b200 import _lib
    if not _lib.available():
        pytest.skip('libp3d.so not built (run python -m pix2pix3d_b200.build)')
    handle = ctypes.CDLL(_lib.LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(handle, s)]
    assert not missing, missing
    assert handle.p3d_abi_version() == _lib.ABI_VERSION


def test_ctypes_table_covers_header():
    from pix2pix3d_b200 import _lib
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared_symbols()


def test_ctypes_signatures_match_header_prototypes():
    """Every entry of _lib._SIGNATURES has the header's parameter count, the same kind (pointer, int, int64_t, uint32_t, float,
    double) at each position and the same return kind; exactly the entries without a trailing stream are query entries."""
    from pix2pix3d_b200 import _lib
    protos = header_prototypes()
    assert sorted(protos) == declared_symbols()
    bad = []
    for name, (ret, kinds, has_stream) in protos.items():
        restype, argtypes, launches = _lib._SIGNATURES[name]
        if [ctypes_kind(t) for t in argtypes] != kinds:
            bad.append((name, 'argtypes', [ctypes_kind(t) for t in argtypes], kinds))
        if ctypes_kind(restype) != ret:
            bad.append((name, 'restype', ctypes_kind(restype), ret))
        if (launches is None) == has_stream:
            bad.append((name, 'launches', launches))
    assert not bad, bad


def test_struct_mirrors_match_the_header_layout():
    """Every struct of include/p3d.h has a ctypes mirror in _lib.STRUCTS (p3d_mesh_view_t crosses as a float array,
    test_mesh_render_cpu.py) with the header's fields in the header's order, of the same kinds, at the offsets and sizes
    a C compiler gives them, and of the same total size."""
    import subprocess
    import tempfile
    from pix2pix3d_b200 import _lib
    structs = header_structs()
    assert sorted(_lib.STRUCTS) == sorted(n for n in structs if n != 'p3d_mesh_view_t')
    lines = ['#include <stddef.h>', '#include <stdio.h>', '#include "p3d.h"', 'int main(void) {']
    for sname in _lib.STRUCTS:
        lines.append(f'printf("{sname} %zu\\n", sizeof({sname}));')
        for f, _, _ in structs[sname]:
            lines.append(f'printf("{sname}.{f} %zu %zu\\n", offsetof({sname}, {f}), sizeof((({sname}*)0)->{f}));')
    lines += ['return 0;', '}']
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, 't.c'), os.path.join(td, 't')
        with open(src, 'w') as fh:
            fh.write('\n'.join(lines) + '\n')
        subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), src, '-o', exe])
        out = subprocess.check_output([exe], text=True)
    layout = {key: tuple(int(v) for v in vals) for key, *vals in (ln.split() for ln in out.splitlines())}
    for sname, mirror in _lib.STRUCTS.items():
        assert [n for n, _ in mirror._fields_] == [f for f, _, _ in structs[sname]], sname
        for (f, kind, n), (_, t) in zip(structs[sname], mirror._fields_):
            got = (ctypes_kind(t._type_), t._length_) if issubclass(t, ctypes.Array) else (ctypes_kind(t), None)
            assert got == (kind, n), (sname, f)
            assert (getattr(mirror, f).offset, getattr(mirror, f).size) == layout[f'{sname}.{f}'], (sname, f)
        assert (ctypes.sizeof(mirror),) == layout[sname], sname


class _StubLib:
    """Stands in for the ctypes handle: every entry records its arguments and returns `status`."""

    def __init__(self):
        self.calls, self.status = [], 0

    def p3d_status_string(self, status):
        return b'stub message'

    def __getattr__(self, name):
        def entry(*args):
            self.calls.append((name, args))
            return self.status
        return entry


def test_call_passes_pointers_appends_the_stream_and_applies_the_status_policy(monkeypatch):
    import torch
    from pix2pix3d_b200 import _lib
    stub, order = _StubLib(), []

    class Guard:
        def __init__(self, device):
            self.device = device

        def __enter__(self):
            order.append(('enter', self.device))

        def __exit__(self, *exc):
            order.append('exit')

    monkeypatch.setattr(_lib, '_lib', stub)
    monkeypatch.setattr(_lib, 'launch_count', 0)
    monkeypatch.setattr(_lib, 'stream_ptr', lambda device=None: order.append('stream') or 'STREAM')
    monkeypatch.setattr(torch.cuda, 'device', Guard)
    x, y, dims = torch.arange(4.0), torch.empty(3), (ctypes.c_int32 * 2)(7, 8)

    assert _lib.call('p3d_ray_sampler', x, y, 2, 0.5, None, dims, device=None) is True
    (name, args), = stub.calls
    assert name == 'p3d_ray_sampler'
    assert args[:5] == (x.data_ptr(), y.data_ptr(), 2, 0.5, None) and args[5] is dims and args[6] == 'STREAM'
    assert order == [('enter', None), 'stream', 'exit']          # the stream is the current one of the guarded device
    assert _lib.launch_count == 1
    _lib.call('p3d_decoder_mlp_bwd', x, device=None)              # two kernels per call
    assert _lib.launch_count == 3 == 1 + _lib._SIGNATURES['p3d_decoder_mlp_bwd'][2]

    stub.status = -2                                              # P3D_BAD_ARG
    with pytest.raises(RuntimeError, match='p3d_fma failed: stub message'):
        _lib.call('p3d_fma', x, device=None)
    stub.status = -1                                              # P3D_UNSUPPORTED
    with pytest.raises(RuntimeError, match='p3d_conv_gemm failed'):
        _lib.call('p3d_conv_gemm', x, device=None)
    assert _lib.call('p3d_conv_gemm', x, device=None, unsupported_ok=True) is False
    stub.status = -2
    with pytest.raises(RuntimeError, match='p3d_conv_gemm failed'):
        _lib.call('p3d_conv_gemm', x, device=None, unsupported_ok=True)
    assert _lib.launch_count == 3

    n_calls = len(stub.calls)
    for name in ('p3d_abi_version', 'p3d_build_info', 'p3d_status_string', 'p3d_decoder_mlp_bwd_workspace_floats',
                 'p3d_marching_cubes_workspace_bytes'):
        with pytest.raises(ValueError, match='query entry'):
            _lib.call(name, device=None)
    assert len(stub.calls) == n_calls and _lib.launch_count == 3


def test_cuda_ops_fail_loudly_without_library(monkeypatch):
    from pix2pix3d_b200 import _lib
    monkeypatch.setattr(_lib, 'LIB_PATH', '/nonexistent/libp3d.so')
    monkeypatch.setattr(_lib, '_lib', None)
    with pytest.raises(RuntimeError, match='missing'):
        _lib.lib()


def test_library_exports_nothing_undeclared():
    """Every `p3d_*` symbol the shared library exports is declared in include/p3d.h (no entry points outside the documented ABI)."""
    import shutil
    import subprocess
    from pix2pix3d_b200 import _lib
    if not _lib.available() or not shutil.which('nm'):
        pytest.skip('needs the built library and nm')
    out = subprocess.check_output(['nm', '-D', '--defined-only', _lib.LIB_PATH], text=True)
    exported = sorted({ln.split()[-1] for ln in out.splitlines() if ln.split() and re.fullmatch(r'p3d_[a-z0-9_]+', ln.split()[-1])})
    assert exported == declared_symbols()
