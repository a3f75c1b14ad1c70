"""The leaf table of the small operand kernels (small_kernel_leaves.py) against the library: every kernel instantiation compiled from
conv_pack.cu, fir_packed.cu, conv_thin.cu and reduce.cu has a launch case, and every case names an instantiation that exists."""
import os
import shutil
import subprocess

import pytest

from small_kernel_leaves import KERNELS, LEAVES, base_name, leaf_name

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, 'pasta-gan-plusplus_b200', 'lib', 'libpgpp_sm100a.so')


def _cuda_tool(name):
    for d in (os.environ.get('CUDA_HOME'), '/usr/local/cuda'):
        if d and os.path.isfile(os.path.join(d, 'bin', name)):
            return os.path.join(d, 'bin', name)
    return None


def test_leaf_name_normalises_symbols_and_profiler_names():
    assert leaf_name('void pgpp::mul_reduce_kernel<(int)256>(pgpp::MulReduceArgs)') == 'mul_reduce_kernel<256>'
    assert leaf_name('pgpp::mul_reduce_kernel<256>(pgpp::MulReduceArgs)') == 'mul_reduce_kernel<256>'
    assert leaf_name('void pgpp::pack_nchw_kernel<__half, (bool)1, (bool)0>(pgpp::PackArgs, pgpp::TileGeom)') == 'pack_nchw_kernel<__half,1,0>'
    assert leaf_name('void pgpp::pack_nchw_kernel<__half, true, false>(pgpp::PackArgs, pgpp::TileGeom)') == 'pack_nchw_kernel<__half,1,0>'
    assert leaf_name('void pgpp::sum_hw_kernel<float, (int)32>(const T1 *, float *, long long, long long)') == 'sum_hw_kernel<float,32>'
    assert leaf_name('pgpp::demod_kernel(const float *, const float *, float *, int, int, int, int, float)') == 'demod_kernel'
    assert leaf_name('void pgpp::conv_direct_kernel<3, 3, 1, 2, false>(pgpp::DirectArgs, pgpp::TileGeom, long long)') == \
        'conv_direct_kernel<3,3,1,2,0>'
    assert base_name('conv1x1_thin_kernel<8,32,1,3>') == 'conv1x1_thin_kernel'


def test_every_compiled_instantiation_has_a_case():
    cuobjdump, cufilt = _cuda_tool('cuobjdump'), _cuda_tool('cu++filt')
    if cuobjdump is None or cufilt is None:
        pytest.skip('cuobjdump / cu++filt not found in $CUDA_HOME/bin or /usr/local/cuda/bin')
    assert os.path.isfile(LIB), f'{LIB} not built'
    syms = subprocess.run([cuobjdump, '-symbols', LIB], check=True, capture_output=True, text=True).stdout
    demangled = subprocess.run([cufilt], input=syms, check=True, capture_output=True, text=True).stdout
    entries = [line.split('STO_ENTRY', 1)[1].strip() for line in demangled.splitlines() if 'STO_ENTRY' in line]
    compiled = {leaf_name(e) for e in entries}
    ours = {leaf for leaf in compiled if base_name(leaf) in KERNELS}
    assert {base_name(leaf) for leaf in ours} == KERNELS
    assert sorted(ours - LEAVES) == [], 'instantiations without a launch case'
    assert sorted(LEAVES - ours) == [], 'cases that name no compiled instantiation'
    assert len(ours) == 71
