"""CPU-side checks of the drop-in boundary: the library builds, loads and
exports exactly the symbols include/pygp_b200.h declares; the host package
mirrors the reference's constructors and error behaviour.  No compute calls."""

import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'pygp_b200.h')


@pytest.fixture(scope='module')
def built():
    import __graft_entry__ as g
    g.build()
    from pygp_b200 import _lib
    return _lib


def header_symbols():
    text = open(HEADER).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(pgp_[a-z0-9_]+)\s*\(', text)))


def test_header_symbols_exported(built):
    out = subprocess.check_output(['nm', '-D', '--defined-only', built.LIB_PATH]).decode()
    exported = set(re.findall(r' T (pgp_\w+)', out))
    declared = header_symbols()
    assert len(declared) >= 30
    missing = [s for s in declared if s not in exported]
    assert not missing, 'declared in the header but not exported: %s' % missing
    # and the ctypes table covers the same set
    assert sorted(built.SIGNATURES) == declared


def test_library_is_sm100a_only(built):
    out = subprocess.check_output(['cuobjdump', '-lelf', built.LIB_PATH]).decode()
    archs = set(re.findall(r'sm_(\d+a?)', out))
    assert archs == {'100a'}, archs


def test_gemm_uses_fp64_tensor_pipe(built):
    sass = subprocess.check_output(['cuobjdump', '-sass', built.LIB_PATH]).decode()
    funcs = sass.split('Function : ')
    gemm = [f for f in funcs if 'gemm_kernel' in f.split('\n', 1)[0]]
    assert len(gemm) >= 4, 'NT / NN / TN forms of gemm_kernel expected in the library'
    for f in gemm:
        assert f.count("DMMA.8x8x4") >= 64       # one k-tile of FP64 tensor-core work per warp
        assert 'LDGSTS' in f                     # cp.async staging


def test_gram_tiles_are_staged_by_the_bulk_copy_engine(built):
    """The Gram / trace tile kernels stage their inputs with cp.async.bulk + mbarrier (the TMA engine):
    UBLKCP (bulk copy global -> shared) and SYNCS (mbarrier arrive / try_wait) in their SASS."""
    sass = subprocess.check_output(['cuobjdump', '-sass', built.LIB_PATH]).decode()
    funcs = sass.split('Function : ')
    tiles = [f for f in funcs if f.split('\n', 1)[0].split('(')[0].find('gram_kernel') >= 0 or 'trace_kernel' in f.split('\n', 1)[0]]
    assert len(tiles) >= 20
    for f in tiles:
        assert 'UBLKCP' in f, f.split('\n', 1)[0]
        assert 'SYNCS' in f, f.split('\n', 1)[0]


def test_no_cpu_fallback(built):
    """Without a device the product path must fail loudly."""
    import torch
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    import pygp_b200 as pygp
    k = pygp.kernels.SE(1.0, 0.5)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        k.get(np.zeros((3, 1)))


def test_product_does_not_import_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'pygp_b200')):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, f


def test_spec_serialisation():
    import pygp_b200 as pygp
    pk = pygp.kernels
    k = pk.SE(1.0, [0.5, 0.6]) * pk.Matern(0.5, [0.4, 0.3], 5) + pk.RQ(0.5, 0.4, 0.3, ndim=2)
    s = k._spec()
    assert (s.ndim, s.nhyper, s.n_parts, s.n_ops) == (2, 9, 3, 5)
    assert [(s.ops[i].op, s.ops[i].arg) for i in range(5)] == [(0, 0), (0, 1), (2, 2), (0, 2), (1, 2)]
    assert [(p.type, p.iso, p.hyper_offset, p.nhyper) for p in list(s.parts)[:3]] == \
        [(0, 0, 0, 3), (3, 0, 3, 3), (5, 1, 6, 3)]
    # associative flattening (_combo.py:151-160)
    k3 = pk.SE(1, 1, ndim=2) + pk.SE(2, 1, ndim=2) + pk.SE(3, 1, ndim=2)
    assert len(k3._parts) == 3 and k3._spec().n_ops == 4
    assert sum(p[1] for p in k._params()) == k.nhyper


def test_constructor_errors():
    # reference tests/test_kernels.py:243-273, tests/test_inference.py:215-230
    import pygp_b200 as pygp
    pk = pygp.kernels
    with pytest.raises(ValueError):
        pk.SE(1, 1, ndim=1) + pk.SE(1, 1, ndim=2)
    with pytest.raises(ValueError):
        pk.SE(1, 1, ndim=1) * pk.SE(1, 1, ndim=2)
    for K, args in [(pk.SE, (1, [1, 1])), (pk.Matern, (1, [1, 1])), (pk.RQ, (1, [1, 1], 1))]:
        with pytest.raises(ValueError):
            K(*args, ndim=1)
    with pytest.raises(ValueError):
        pk.Matern(1, 1, d=12)
    with pytest.raises(ValueError):
        pygp.BasicGP(1, 1, 1, 0, 2, 'foo')
    gp = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(1), pk.Periodic(1, 1, 1), 0)
    with pytest.raises(ValueError):
        pygp.BasicGP.from_gp(gp)


def test_hyper_roundtrip_and_names():
    import pygp_b200 as pygp
    gp = pygp.BasicGP(0.1, 1.0, [0.5, 0.6], 0.3)
    assert [p[0] for p in gp._params()] == ['sn', 'sf', 'ell', 'mu']
    np.testing.assert_allclose(gp.get_hyper(), [np.log(0.1), 0.0, np.log(0.5), np.log(0.6), 0.3])
    gp.set_hyper(gp.get_hyper() + 0.1)         # no data: no device call
    np.testing.assert_allclose(gp.get_hyper()[-1], 0.4)
    g2 = pygp.inference.ExactGP(pygp.likelihoods.Gaussian(0.1),
                                pygp.kernels.SE(1, 1, ndim=2) + pygp.kernels.RQ(1, 1, 1, ndim=2), 0)
    assert [p[0] for p in g2._params()] == ['like.sigma', 'kern.part0.sf', 'kern.part0.ell',
                                            'kern.part1.sf', 'kern.part1.ell', 'kern.part1.alpha', 'mean']
    assert repr(gp).startswith('BasicGP(sn=')


def _build_c_client(built, tmp_path):
    exe = str(tmp_path / 'c_smoke')
    libdir = os.path.dirname(built.LIB_PATH)
    subprocess.check_call(['gcc', '-std=c99', '-Wall', '-Wextra', '-pedantic', '-Werror', '-I', os.path.join(ROOT, 'include'),
                           os.path.join(ROOT, 'tests', 'c_abi', 'smoke.c'), '-o', exe, '-L', libdir, '-lpygp_b200',
                           '-Wl,-rpath,' + libdir, '-lm'])
    return exe


def test_header_is_plain_c_and_links(built, tmp_path):
    """include/pygp_b200.h is a C header (strict C99, no torch / C++ types) and a
    plain-C client links against the library; without a device it fails loudly."""
    import torch
    exe = _build_c_client(built, tmp_path)
    if torch.cuda.is_available():
        pytest.skip('a GPU is present (tests/test_exact_gpu.py runs the client)')
    p = subprocess.run([exe], capture_output=True, text=True)
    assert p.returncode == 2
    assert 'no CPU fallback' in p.stderr
