"""Record runs of the UNMODIFIED original jpeg2png into tests/golden/reference_runs.npz.

Needs the original's sources compiled into oracle/_ref (oracle/Makefile, `make -C oracle ref
REF=<path to the sources>`); then:

    python tests/golden/make_reference_runs.py

For every run the file keeps the inputs (`struct coef` contents and solver parameters) and, per
output plane of the original's compute() (SIMD build = what ships), the SHA-256 of its float32 bits
and a fixed sample of its values (tests/golden_io.py); for the 8x8 transforms, the input blocks and
the CRC-32 of each output block.  tests/test_oracle.py checks the restatement
against these records, so the comparison needs no copy of the original.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from jpeg2png_b200 import synth  # noqa: E402
from tests import helpers as H  # noqa: E402
from tests.golden_io import REFERENCE_RUNS, block_crc, record_image, record_planes  # noqa: E402
from tests.test_oracle import REFERENCE_CONFIGS  # noqa: E402


def sweep_config(seed):
    """Randomised configuration: plane sizes, sampling factors up to 3x4, zero and non-zero weights,
    single-plane and joint mode, planes smaller than the frame."""
    rng = np.random.default_rng(1000 + seed)
    nplanes = 3
    samp = [(1, 1)] + [(int(rng.integers(1, 4)), int(rng.integers(1, 5))) for _ in range(2)]
    fw, fh = 8 * int(rng.integers(2, 9)), 8 * int(rng.integers(2, 7))
    dims = []
    for (sw, sh) in samp:
        cw, ch = -(-fw // sw), -(-fh // sh)
        cw, ch = -(-cw // 8) * 8, -(-ch // 8) * 8
        if rng.random() < 0.3 and cw > 8:
            cw -= 8                                               # a plane that does not cover the frame
        dims.append((cw, ch))
    img = synth.random_coefs(dims, samp, seed=seed, amplitude=int(rng.integers(5, 60)), qmax=int(rng.integers(2, 80)))
    joint = rng.random() < 0.6
    channels = [0, 1, 2] if joint else [int(rng.integers(0, nplanes))]
    weight = float(rng.choice([0.0, 0.1, 0.3, 1.0]))
    pw = [float(rng.choice([0.0, 0.001, 0.05])) for _ in channels]
    iters = int(rng.integers(1, 25))
    return img, channels, weight, pw, iters


def runs():
    """name -> (image, channels, weight, pweights, iterations)"""
    out = {'simd_vs_scalar': (synth.synth_coefs(96, 64, 10, '4:2:0', 11), [0, 1, 2], 0.3, [0.001] * 3, 25)}
    for i, (w, h, q, ss, channels, weight, pw, iters) in enumerate(REFERENCE_CONFIGS):
        out[f'config{i}'] = (synth.synth_coefs(w, h, q, ss, seed=1234 + w + h), channels, weight, pw, iters)
    for seed in range(5):
        img = synth.random_coefs([(40, 24), (24, 16), (16, 8)], [(1, 1), (2, 2), (3, 4)], seed)
        out[f'random_planes{seed}'] = (img, [0, 1, 2], 0.4, [0.001] * 3, 12)
    for seed in range(16):
        out[f'sweep{seed}'] = sweep_config(seed)
    return out


def main():
    H.build_oracle_libs()
    assert H.have_ref(), 'the original jpeg2png is not compiled into oracle/_ref (see oracle/Makefile)'
    blob = {}
    for name, (img, channels, weight, pw, iters) in runs().items():
        f = H.decode_planes(img, channels)
        out = H.run_compute('ref', img, channels, weight, pw, iters, [p.copy() for p in f])
        p = f'{name}.'
        blob.update(record_image(p, img))
        blob.update({p + 'channels': np.array(channels), p + 'weight': np.float32(weight),
                     p + 'pweight': np.array(pw, np.float32), p + 'iterations': np.int64(iters)})
        blob.update(record_planes(p, out))
        if name == 'simd_vs_scalar':
            scalar = H.run_compute('ref_c', img, channels, weight, pw, iters, [p.copy() for p in f])
            H.assert_bit_identical(out, scalar, 'reference SIMD vs scalar build')
            blob.update(record_planes(p + 'scalar_', scalar))
    # 8x8 transforms: random blocks over many magnitudes, and extreme ones (denormals)
    ref = H.load_ref()
    rng = np.random.default_rng(5)
    blocks = [rng.normal(0, s, 64).astype(np.float32) for s in (1e-3, 1.0, 50.0, 1e4, 1e-30) for _ in range(40)]
    blocks += [np.zeros(64, np.float32), np.full(64, 127.5, np.float32), -np.ones(64, np.float32) * 1e-42]
    blob['transforms.blocks'] = np.array(blocks)
    blob['transforms.dct_crc32'] = np.array([block_crc(H.transform8x8(ref.dct8x8s, b)) for b in blocks], np.uint32)
    blob['transforms.idct_crc32'] = np.array([block_crc(H.transform8x8(ref.idct8x8s, b)) for b in blocks], np.uint32)
    np.savez_compressed(REFERENCE_RUNS, **blob)
    print(REFERENCE_RUNS, os.path.getsize(REFERENCE_RUNS), 'bytes,', len(blob), 'arrays')


if __name__ == '__main__':
    main()
