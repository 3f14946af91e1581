"""CPU: the C-ABI library loads and exports every symbol include/mcb200.h declares; argument validation that runs
before any CUDA call reports through mc_last_error_string (no compute without a GPU)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT
from modelcompression_b200 import _lib


def declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'mcb200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(mc_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 20
    for name in names:
        assert hasattr(lib, name), "libmcb200.so does not export %s" % name
    assert set(names) == set(_lib.EXPORTED_SYMBOLS), "ctypes prototypes out of sync with include/mcb200.h"


def test_version_and_error_string():
    lib = _lib.load()
    assert lib.mc_version() == 100
    assert isinstance(lib.mc_last_error_string(), bytes)


def test_argument_validation_without_gpu():
    lib = _lib.load()
    rc = lib.mc_conv_fwd(None, None)
    assert rc == -1 and b'null descriptor' in lib.mc_last_error_string()
    d = _lib.mc_conv_desc()
    d.d_in = d.d_wpack = d.d_scale = d.d_shift = d.d_out = 16
    d.ksize = 5
    rc = lib.mc_conv_fwd(ctypes.byref(d), None)
    assert rc == -1 and b'ksize' in lib.mc_last_error_string()
    rc = lib.mc_kth_abs_select(None, None, 0, 0, 0.0, None, None, 0, None)
    assert rc == -1
    with pytest.raises(_lib.McError):
        _lib.check(rc, "mc_kth_abs_select")
    assert lib.mc_workspace_bytes_kth_abs_select(1000) >= 4000


def test_conv_desc_layout_matches_header():
    # field order of the ctypes mirror == struct mc_conv_desc in the header
    text = open(os.path.join(ROOT, 'include', 'mcb200.h')).read()
    body = text[text.index('typedef struct mc_conv_desc {') + len('typedef struct mc_conv_desc {'):
                text.index('} mc_conv_desc;')]
    body = re.sub(r'/\*.*?\*/', '', body, flags=re.S)
    fields = []
    for decl in body.split(';'):
        for piece in decl.split(','):
            names = re.findall(r'[A-Za-z_][A-Za-z_0-9]*', piece)
            if names:
                fields.append(names[-1])
    assert fields == [f[0] for f in _lib.mc_conv_desc._fields_]


def test_cpu_tensor_fails_loudly(cfg_path):
    import torch
    import modelcompression_b200 as mc
    model = mc.Darknet(cfg_path).eval()
    with pytest.raises(RuntimeError, match="no CPU"):
        model(torch.zeros(1, 3, 416, 416))
    with pytest.raises(RuntimeError, match="no CPU"):
        mc.weight_prune(model, 50.)


def test_conv_desc_offsets_match_the_c_compiler(tmp_path):
    """The ctypes mirror of mc_conv_desc must have the C compiler's layout (size and every field offset): a field added
    on one side only would silently shift the descriptor the kernels read."""
    import subprocess
    fields = [f[0] for f in _lib.mc_conv_desc._fields_]
    src = tmp_path / "layout.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "mcb200.h"', 'int main(void) {',
             '  printf("%zu\\n", sizeof(mc_conv_desc));']
    for f in fields:
        lines.append('  printf("%%zu\\n", offsetof(mc_conv_desc, %s));' % f)
    lines += ['  return 0;', '}']
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include')
    subprocess.run(['gcc', '-I', inc, str(src), '-o', str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert out[0] == ctypes.sizeof(_lib.mc_conv_desc)
    for f, off in zip(fields, out[1:]):
        assert getattr(_lib.mc_conv_desc, f).offset == off, f


def test_bn_pool_pass_contract_without_gpu():
    """The BatchNorm / pool passes (train_ops.cu) move 8 channels per 16-byte access: C > 2048, pitches or ch_off that
    are not multiples of 8, pointers that are not 16-byte aligned and B*(H+1)*(W+1) >= 2^31 are argument errors,
    reported before any CUDA call.  (Pointers are fake addresses: nothing may be launched.)"""
    lib = _lib.load()
    P, Q = 1 << 20, (1 << 20) + 2  # 16-byte aligned / misaligned device addresses
    f = ctypes.c_void_p(P)

    def col_stats(C=64, ld=64, ch_off=0, z=P, rows=100):
        return lib.mc_col_stats(z, rows, C, ld, ch_off, f, f, None)

    def bn_apply(C=64, ld_z=64, ld_out=64, ch_off=0, z=P, out=P, B=2, H=8, W=8):
        return lib.mc_bn_apply(z, ld_z, B, H, W, C, f, f, 1, out, ld_out, ch_off, 0, None)

    def bn_backward(C=64, ld_z=64, ld_da=64, ld_dz=64, ch_off=0, z=P, da=P, dz=P, B=2, H=8, W=8):
        return lib.mc_bn_backward(z, ld_z, da, ld_da, ch_off, 0, B, H, W, C, f, f, f, f, 1, f, f, dz, ld_dz, None)

    def pool_backward(C=64, ld_a=64, ld_dp=64, ld_df=64, a=P, dp=P, df=P, B=2, H=8, W=8):
        return lib.mc_maxpool2x2_backward(a, ld_a, dp, ld_dp, B, H, W, C, df, ld_df, 0, None)

    def bn_apply_pool(C=64, ld_z=64, ld_p=64, z=P, p=P, B=2, H=8, W=8):
        return lib.mc_bn_apply_pool(z, ld_z, B, H, W, C, f, f, 1, p, ld_p, None)

    def bn_pool_backward(C=64, ld_z=64, ld_dp=64, ld_dz=64, z=P, dp=P, dz=P, B=2, H=8, W=8):
        return lib.mc_bn_pool_backward(z, ld_z, dp, ld_dp, B, H, W, C, f, f, f, f, f, f, 1, f, f, dz, ld_dz, None)

    big = dict(B=1 << 13, H=511, W=511)  # 2^13 * 512 * 512 = 2^31 rows
    cases = [
        (col_stats, dict(C=2056, ld=2056)), (col_stats, dict(ld=68)), (col_stats, dict(ch_off=4, ld=72)),
        (col_stats, dict(z=Q)), (col_stats, dict(rows=1 << 31)),
        (bn_apply, dict(C=2056, ld_z=2056, ld_out=2056)), (bn_apply, dict(ld_out=68)), (bn_apply, dict(ch_off=4, ld_out=72)),
        (bn_apply, dict(z=Q)), (bn_apply, dict(out=Q)), (bn_apply, big),
        (bn_backward, dict(C=2056, ld_z=2056, ld_da=2056, ld_dz=2056)), (bn_backward, dict(ld_z=68)),
        (bn_backward, dict(ld_da=68)), (bn_backward, dict(ld_dz=68)), (bn_backward, dict(ch_off=4, ld_da=72)),
        (bn_backward, dict(z=Q)), (bn_backward, dict(da=Q)), (bn_backward, dict(dz=Q)), (bn_backward, big),
        (pool_backward, dict(C=2056, ld_a=2056, ld_dp=2056, ld_df=2056)), (pool_backward, dict(ld_a=68)),
        (pool_backward, dict(ld_dp=68)), (pool_backward, dict(ld_df=68)), (pool_backward, dict(a=Q)),
        (pool_backward, dict(dp=Q)), (pool_backward, dict(df=Q)), (pool_backward, dict(B=1 << 13, H=510, W=511)),
        (bn_apply_pool, dict(C=4096, ld_z=4096, ld_p=4096)), (bn_apply_pool, dict(ld_z=68)), (bn_apply_pool, dict(p=Q)),
        (bn_apply_pool, dict(B=1 << 13, H=510, W=511)),
        (bn_pool_backward, dict(C=4096, ld_z=4096, ld_dp=4096, ld_dz=4096)), (bn_pool_backward, dict(ld_dz=68)),
        (bn_pool_backward, dict(dz=Q)), (bn_pool_backward, dict(B=1 << 13, H=510, W=511)),
    ]
    for fn, kw in cases:
        rc = fn(**kw)
        msg = lib.mc_last_error_string()
        assert rc == -1 and msg.startswith(b'mc_'), "%s(%s): rc %d, %r" % (fn.__name__, kw, rc, msg)
