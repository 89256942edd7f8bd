"""CPU: the oracle restatement against known-answer vectors generated from the reference
(SURVEY.md section 8c KAT1/1b/2/3, produced with the reference's own compiled torchac.cpp) and against
the committed golden fixtures (tests/golden, produced by oracle/gen_golden.py from the unmodified
reference Python).  The C oracle is pinned byte-for-byte against stored outputs of the reference's compiled
coder (tests/golden/torchac_pin.npz, oracle/pin_oracle.py)."""
import hashlib
import struct

import numpy as np
import pytest
import torch

from oracle import ac, model as om
from tests import util


def test_kat_uniform_rows():
    row = ac.uniform_cdf_row(25)
    assert row.tolist() == [0, 2621, 5243, 7864, 10486, 13107, 15729, 18350, 20972, 23593, 26214, 28836,
                            31457, 34079, 36700, 39322, 41943, 44564, 47186, 49807, 52429, 55050, 57672,
                            60293, 62915, 0]
    row256 = ac.uniform_cdf_row(256)
    assert row256.tolist() == [256 * i for i in range(256)] + [0]


def test_kat_streams():
    row25, row256 = ac.uniform_cdf_row(25), ac.uniform_cdf_row(256)
    cases = [(row25, [0, 1, 2, 3, 24, 23, 12, 12], '0071e1d840'),
             (row256, [0, 255, 128, 1, 254, 77], '00ff8001fe4d40'),
             (row25, [0], '04'), (row25, [24], 'f8')]
    for row, sym, want in cases:
        sym = np.array(sym, np.int16)
        got = ac.encode(row, sym)
        assert got.hex() == want
        assert (ac.decode(row, got, len(sym)) == sym).all()


def test_kat2_mixture():
    """K=2, 1x4 pixels, L=25 (SURVEY.md KAT2): CDF rows + stream."""
    targets = torch.linspace(-1 - 1 / 24, 1 + 1 / 24, 26).numpy()
    mu = np.array([[-0.5, 0, 0.25, 0.9], [0.5, 0.1, -0.25, -0.9]], np.float32)
    ls = np.array([[-2, -1, -3, -7], [-1.5, -2.5, 0, -4]], np.float32)
    pi = torch.softmax(torch.tensor([[0., 1, -1, 2], [0, 0, 0, 0]]), 0).numpy()
    cdf = ac.mixture_cdf(targets, mu, ls, pi)
    row0 = [620, 1120, 2001, 3505, 5934, 9525, 14187, 19327, 24090, 27895, 30678, 32712, 34352, 35903,
            37592, 39572, 41920, 44628, 47599, 50662, 53616, 56285, 58555, 60390, 61812, 62879]
    assert np.abs(cdf[0].astype(int) - np.array(row0)).max() <= 1
    assert cdf[3, :6].tolist()[0] == 3 and abs(int(cdf[3, 1]) - 311) <= 1
    sym = np.array([6, 12, 15, 1], np.int16)
    data = ac.encode(cdf, sym)
    assert (ac.decode(cdf, data) == sym).all()
    if (cdf[0] == np.array(row0)).all():
        assert data.hex() == '401c'


def test_decoder_zero_fills_short_input():
    row = ac.uniform_cdf_row(25)
    sym = np.arange(20, dtype=np.int16) % 25
    data = ac.encode(row, sym)
    out = ac.decode(row, data[:2], 20)          # truncated: must not crash, prefix still right
    assert out.shape == (20,) and (out[:2] == sym[:2]).all()
    assert ac.decode(row, b'', 5).shape == (5,)


def test_pinned_against_compiled_reference():
    """the C oracle reproduces the compiled reference coder's streams and garbage-input decodes
    (tests/golden/torchac_pin.npz; also against oracle/_ref itself when that is built)."""
    from oracle import pin_oracle
    assert pin_oracle.main() == 0


@pytest.mark.parametrize('name,cfg', [('l3c_32x32_i0', 'cr'), ('l3c_40x28_i1', 'cr'), ('rgbs_64x64_i0', 'cr_rgb_shared')])
def test_oracle_reproduces_reference_goldens(name, cfg):
    """oracle/model.py (weights from the product's seed-0 module tree) == the unmodified
    reference: container bytes, symbols, parameters, theoretical bpsp; and it decodes them.
    Container bytes: the DMLL scales need the CPU convs to round exactly as on the host that made the
    goldens (oneDNN picks other kernels on other CPUs, e.g. AVX2 ones), so byte identity and the decode of the
    reference's own file are asserted where this host reproduces the file; the uniform-prior scale is pure
    integer arithmetic and is decoded from the reference's file on every host."""
    g = util.golden_npz(name)
    summ = util.golden_summary()[name]
    bp = util.blueprint(cfg, device='cpu')
    sd = util.cpu_state_dict(bp)
    ocfg = util.oracle_cfg(cfg)
    img = torch.from_numpy(g['img'])
    data, dbg = om.encode_image(sd, ocfg, img, 'torch', return_debug=True)
    ref = g['container'].tobytes()
    out = dbg['out']
    assert (out.S[1].numpy() == g['S1']).all()
    if cfg == 'cr':
        assert (out.S[2].numpy() == g['S2']).all() and (out.S[3].numpy() == g['S3']).all()
        np.testing.assert_allclose(out.P[2].numpy(), g['P2'], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(out.P[1].numpy()[:, :, ::2, ::2], g['P1'], rtol=1e-4, atol=1e-4)
        th = om.theoretical_bpsps(ocfg, out)
        np.testing.assert_allclose(th, g['theory_bpsps'], rtol=1e-4)
    np.testing.assert_allclose(out.P[0].numpy()[:, :, ::4, ::4], g['P0'], rtol=1e-4, atol=1e-3)
    assert len(data) == summ['ref_bytes']
    if data == ref:     # bit-identical conv numerics (same CPU kernels as the generating run)
        assert hashlib.sha256(data).hexdigest() == summ['ref_sha256']
    # the reference's streams of the coarsest scale (first in the container, after the padding tuple)
    top = g['S%d' % ocfg.num_scales]
    C, h, w = struct.unpack_from('<BHH', ref, 8)
    assert (C, h, w) == top.shape[1:]
    row, pos = ac.uniform_cdf_row(om.dmlls(ocfg)[1].L), 13
    for c in range(C):
        n, = struct.unpack_from('<I', ref, pos)
        assert (ac.decode(row, ref[pos + 4:pos + 4 + n], h * w) == top[0, c].reshape(-1)).all(), c
        pos += 4 + n
    # the whole file: where data == ref this is the reference's own file
    dec = om.decode_image(sd, ocfg, data, 'torch')
    assert (dec[0] == img.long()).all()


def test_oracle_weights_equal_the_reference_default_init():
    """oracle/weights.py (plain torch module tree, used by `bench.py --impl reference`) reproduces the
    seed-0 default init of the UNMODIFIED reference: same keys, order and values (sha256 recorded by
    oracle/gen_golden.py from the reference's own MultiscaleBlueprint)."""
    import hashlib
    import json
    import os
    from oracle import model as om, weights
    with open(os.path.join(os.path.dirname(__file__), 'golden', 'summary.json')) as f:
        g = json.load(f)
    for cfg, key in [(om.CFG_L3C, 'l3c'), (om.CFG_RGB_SHARED, 'rgbs')]:
        sd = weights.default_init_state_dict(cfg)
        h = hashlib.sha256()
        for k in sd:
            h.update(k.encode())
            h.update(sd[k].contiguous().numpy().tobytes())
        assert h.hexdigest() == g[key + '_sd_sha256'], key
        assert sum(v.numel() for v in sd.values()) == g[key + '_sd_numel']


def test_reference_arm_of_the_bench_never_touches_the_product():
    """VERDICT r1: the reference arm's process must map only the checker's native code."""
    import ast
    import os
    src = open(os.path.join(os.path.dirname(os.path.dirname(__file__)), 'bench.py')).read()
    tree = ast.parse(src)
    for fn in tree.body:
        if isinstance(fn, ast.FunctionDef) and fn.name in ('run_reference', '_ref_roundtrip', '_ref_init',
                                                           'cpu_roundtrips', '_reference_sample', 'make_images'):
            seg = ast.get_source_segment(src, fn)
            assert 'l3c_pytorch_b200' not in seg and 'import l3c' not in seg, fn.name
    # and nothing at module level pulls it in
    top = [n for n in tree.body if isinstance(n, (ast.Import, ast.ImportFrom))]
    assert all('l3c' not in ast.get_source_segment(src, n) for n in top)
    for mod in ('model.py', 'weights.py', 'ac.py'):
        assert 'l3c_pytorch_b200' not in open(os.path.join(os.path.dirname(os.path.dirname(__file__)), 'oracle', mod)).read().replace(
            'not import l3c_pytorch_b200', '')
