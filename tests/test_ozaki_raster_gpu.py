"""The residue products of the emulated V V^T (pygp_b200/csrc/ozaki.cu) at the orders where their work
order matters: tiles handed out from a global counter in bands of row blocks, the output cut into several
strips.  tools/bin/ozaki_check strips checks that the order visits every tile of a strip once, compares the
residue bytes of sampled tiles (first and last of every strip, diagonal tiles, the last partial row block,
random ones; all 16 moduli) bit for bit against an independent dp4a product of the same residue rows, and
H against the DMMA product."""

import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHECK = os.path.join(ROOT, 'tools', 'bin', 'ozaki_check')

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def check():
    import __graft_entry__ as g
    g.build()
    return CHECK


# (n, most tiles per strip): 32768 has 16512 lower tiles, 20077 (157 row blocks, the last one partial) 6241
@pytest.mark.parametrize('n,tiles', [(32768, 5000), (20000 + 77, 2000)])
def test_products_in_strips_bit_exact(check, n, tiles):
    p = subprocess.run([CHECK, 'strips', str(n), str(tiles)], capture_output=True, text=True)
    out = p.stdout + p.stderr
    assert p.returncode == 0, out
    f = dict(re.findall(r'(\w+)=(\S+)', out))
    assert int(f['strips']) >= 3, out
    assert int(f['order_errors']) == 0 and int(f['residue_mismatches']) == 0, out
    assert int(f['tiles_checked']) > 3 * int(f['strips']), out
    assert float(f['max_rel_dH']) <= 1e-13, out
