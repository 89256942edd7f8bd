"""Pins ac_oracle.c against the reference's own torchac.cpp: KATs of SURVEY.md section 8c + seeded random
tables, byte-for-byte.  TEST INFRASTRUCTURE ONLY.

The reference's outputs on the seeded cases are stored in tests/golden/torchac_pin.npz, so the pin holds on
any checkout.  Where the reference's coder is compiled into oracle/_ref (build_ref.py) it is also run live and
must still agree with the stored outputs.

    python oracle/pin_oracle.py                  # pin against the stored outputs (and oracle/_ref if built)
    python oracle/pin_oracle.py --write-golden   # regenerate tests/golden/torchac_pin.npz from oracle/_ref
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ac, build_ref  # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden', 'torchac_pin.npz')


def _t_cdf(cdf):
    return torch.from_numpy(cdf.view(np.int16).copy()).reshape(1, 1, cdf.shape[0], cdf.shape[1])


def cases(reference_encode):
    """The seeded cases, in a fixed order: yields (cdf [n_sym, Lp] uint16, sym [n_sym] int16, want, junk).
    `want = reference_encode(i, cdf, sym)` is the reference's stream of case i; the length of the garbage
    input `junk` (None for the underflow cases) depends on it, and so does every case drawn after it."""
    rng = np.random.default_rng(7)
    i = 0
    for Lp, n_sym in [(26, 1), (26, 8), (26, 4097), (257, 3), (257, 5000), (6, 777), (2, 64)]:
        for trial in range(6):
            L = Lp - 1
            # random strictly increasing rows with >= 1 count per symbol, first entry may be > 0
            w = rng.integers(1, 4000 if trial % 2 else 40, size=(n_sym, L)).astype(np.float64)
            w = w / w.sum(1, keepdims=True) * (65536 - Lp - 40)
            c = np.floor(np.cumsum(w, 1)).astype(np.int64) + np.arange(1, L + 1)
            lead = rng.integers(0, 30, size=(n_sym, 1))
            cdf = np.concatenate([lead, c[:, :-1] + lead, np.zeros((n_sym, 1), np.int64)], 1)
            cdf = cdf.astype(np.uint16)
            assert (np.diff(cdf[:, :-1].astype(np.int64), axis=1) > 0).all()
            sym = rng.integers(0, L, size=n_sym).astype(np.int16)
            want = reference_encode(i, cdf, sym)
            # truncated / garbage input: the decoder zero-fills, must still agree with the reference
            junk = bytes(rng.integers(0, 256, size=max(1, len(want) // 2)).astype(np.uint8))
            yield cdf, sym, want, junk
            i += 1
    # long underflow runs: every symbol straddles the midpoint, the owed ("pending") bits pile up far
    # beyond 32 and across many symbols before a release or the terminator flushes them
    # (torchac.cpp:196-206, 209-219) -- the path the GPU encoder's batched emission must reproduce
    for n_sym in (5, 33, 1000, 4099):
        for trial in range(3):
            half = 32768
            rows = np.zeros((n_sym, 4), np.int64)
            for k in range(n_sym):
                rows[k, :3] = [0, half - int(rng.integers(1, 200)), half + int(rng.integers(1, 200))]
            sym = np.ones(n_sym, np.int16)
            if trial < 2:
                for k in rng.integers(0, n_sym, size=max(1, n_sym // 37)):
                    sym[k] = int(rng.integers(0, 3))
            cdf = rows.astype(np.uint16)
            yield cdf, sym, reference_encode(i, cdf, sym), None
            i += 1


def reference_outputs(ref):
    """Runs the compiled reference on every case -> the arrays tests/golden/torchac_pin.npz stores:
    the concatenated streams with their offsets, the concatenated decodes of the garbage inputs with theirs,
    and the sha256 of every input (a changed random stream fails loudly instead of as a mismatch)."""
    streams, junk_dec, h = [], [], hashlib.sha256()

    def encode(i, cdf, sym):
        want = ref.encode_cdf(_t_cdf(cdf), torch.from_numpy(sym.copy()))
        assert (ref.decode_cdf(_t_cdf(cdf), want).numpy() == sym).all(), 'reference round trip, case %d' % i
        return want

    for cdf, sym, want, junk in cases(encode):
        streams.append(np.frombuffer(want, np.uint8))
        h.update(cdf.tobytes() + sym.tobytes())
        if junk is not None:
            junk_dec.append(ref.decode_cdf(_t_cdf(cdf), junk).numpy().astype(np.int16))
            h.update(junk)
    return {'streams': np.concatenate(streams),
            'stream_offsets': np.cumsum([0] + [len(s) for s in streams]).astype(np.int64),
            'junk_decoded': np.concatenate(junk_dec),
            'junk_offsets': np.cumsum([0] + [len(d) for d in junk_dec]).astype(np.int64),
            'inputs_sha256': np.array(h.hexdigest())}


def check(gold):
    """The C oracle against the reference's outputs `gold` on every case, and the KATs.
    -> (number of cases, number of underflow cases)"""
    so, jo = gold['stream_offsets'], gold['junk_offsets']
    h = hashlib.sha256()
    n_cases = n_under = n_junk = 0
    for cdf, sym, want, junk in cases(lambda i, cdf, sym: gold['streams'][so[i]:so[i + 1]].tobytes()):
        h.update(cdf.tobytes() + sym.tobytes())
        assert ac.encode(cdf, sym) == want, ('case', n_cases, cdf.shape, len(want))
        assert (ac.decode(cdf, want) == sym).all(), ('case', n_cases)
        if junk is None:
            n_under += 1
        else:
            h.update(junk)
            assert (ac.decode(cdf, junk) == gold['junk_decoded'][jo[n_junk]:jo[n_junk + 1]]).all(), ('junk', n_cases)
            n_junk += 1
        n_cases += 1
    assert n_cases == len(so) - 1 and n_junk == len(jo) - 1
    assert h.hexdigest() == str(gold['inputs_sha256']), 'the seeded inputs differ from the ones the goldens were made of'
    # KATs (SURVEY.md section 8c)
    row25 = ac.uniform_cdf_row(25)
    assert row25.tolist()[:4] == [0, 2621, 5243, 7864] and row25[-1] == 0 and row25[-2] == 62915
    assert ac.encode(row25, np.array([0, 1, 2, 3, 24, 23, 12, 12], np.int16)).hex() == '0071e1d840'
    row256 = ac.uniform_cdf_row(256)
    assert ac.encode(row256, np.array([0, 255, 128, 1, 254, 77], np.int16)).hex() == '00ff8001fe4d40'
    assert ac.encode(row25, np.array([0], np.int16)).hex() == '04'
    assert ac.encode(row25, np.array([24], np.int16)).hex() == 'f8'
    return n_cases, n_under


def main(argv=()):
    ref = build_ref.load()
    if '--write-golden' in argv:
        if ref is None:
            print('oracle/_ref is not built (build_ref.py): nothing to write the goldens from')
            return 1
        np.savez_compressed(GOLDEN, **reference_outputs(ref))
        print('wrote', os.path.relpath(GOLDEN, ROOT))
    with np.load(GOLDEN) as f:
        gold = dict(f)
    n_cases, n_under = check(gold)
    if ref is not None:
        live = reference_outputs(ref)
        assert all(np.array_equal(live[k], gold[k]) for k in gold), 'oracle/_ref disagrees with ' + GOLDEN
    print('pinned: %d random cases (incl. %d long-underflow ones) + KAT1/1b/3 byte-identical to the reference%s'
          % (n_cases, n_under, ' (stored outputs and oracle/_ref)' if ref is not None else ' (stored outputs)'))
    return 0


if __name__ == '__main__':
    sys.exit(main(sys.argv[1:]))
