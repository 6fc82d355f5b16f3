"""CPU tests: the oracle restatement against the golden vectors and against recorded runs of the
original jpeg2png (tests/golden/reference_runs.npz).  Bit-exact everywhere: the path is fp32/fp64
arithmetic in a fixed IEEE operation order, so "equal" means equal bit patterns."""
import os

import numpy as np
import pytest

from jpeg2png_b200 import synth
from tests import helpers as H
from tests.golden_io import (assert_matches_recorded, block_crc, golden_cases, load_case, load_reference_run,
                             load_reference_transforms)

needs_ref = pytest.mark.skipif(not (H.have_ref() or os.path.exists(H.REFERENCE_SRC)),
                               reason='compiled reference (oracle/_ref) not available on this machine')


@pytest.fixture(scope='module', autouse=True)
def _build():
    H.build_oracle_libs()


@pytest.mark.parametrize('name', golden_cases())
def test_oracle_matches_golden(name):
    g = load_case(name)
    out = H.run_compute('oracle', g['img'], g['channels'], g['weight'], g['pweight'], g['iterations'], g['fdata'])
    H.assert_bit_identical(out, g['out'], f'golden {name}')


@pytest.mark.parametrize('name', golden_cases())
def test_oracle_decode_matches_golden(name):
    """The conventional decode (jpeg.c:83-92 + unbox) that produced the fixtures' fdata."""
    g = load_case(name)
    dec = H.decode_planes(g['img'], g['channels'])
    H.assert_bit_identical(dec, g['fdata'], f'decode {name}')


@needs_ref
@pytest.mark.parametrize('name', golden_cases())
def test_reference_reproduces_golden(name):
    """Guards the fixtures themselves: the reference build still returns what was recorded."""
    g = load_case(name)
    out = H.run_compute('ref', g['img'], g['channels'], g['weight'], g['pweight'], g['iterations'], g['fdata'])
    H.assert_bit_identical(out, g['out'], f'ref {name}')


def test_reference_simd_equals_scalar():
    """The reference's own invariant (compute_simd_step.c:103-104, :223-224): its SIMD and scalar
    builds were recorded on the same frame; the restatement must reproduce both bit for bit."""
    run = load_reference_run('simd_vs_scalar')
    out = H.run_compute('oracle', run['img'], run['channels'], run['weight'], run['pweight'], run['iterations'])
    assert_matches_recorded(out, run['out'], 'oracle vs reference SIMD build')
    assert_matches_recorded(out, run['scalar_out'], 'oracle vs reference scalar build')


# (w, h, quality, subsampling, channels, weight, pweights, iterations); the frames were synthesised
# with seed 1234 + w + h and the original's outputs recorded by tests/golden/make_reference_runs.py
REFERENCE_CONFIGS = [
    (256, 256, 10, '4:2:0', [0, 1, 2], 0.3, [0.001] * 3, 50),      # BASELINE config 1
    (256, 256, 10, '4:2:0', [2], 0.3, [0.001], 50),                # config 1, separate mode, chroma
    (200, 120, 30, '4:2:0', [0, 1, 2], 0.3, [0.001] * 3, 30),      # luma grid narrower/shorter than the frame
    (136, 72, 50, '4:4:4', [0, 1, 2], 0.7, [0.001, 0.0, 0.01], 40),
    (64, 64, 90, '4:4:4', [0, 1, 2], 0.0, [0.0] * 3, 20),          # TV only
]


@pytest.mark.parametrize('w,h,q,ss,channels,weight,pw,iters', REFERENCE_CONFIGS)
def test_oracle_matches_reference(w, h, q, ss, channels, weight, pw, iters):
    run = load_reference_run(f'config{REFERENCE_CONFIGS.index((w, h, q, ss, channels, weight, pw, iters))}')
    assert (run['img'].width, run['img'].height, run['channels'], run['iterations']) == (w, h, channels, iters)
    ora = H.run_compute('oracle', run['img'], channels, weight, pw, iters)
    assert_matches_recorded(ora, run['out'], 'ref vs oracle')


def test_oracle_matches_reference_random_planes():
    for seed in range(5):
        run = load_reference_run(f'random_planes{seed}')
        ora = H.run_compute('oracle', run['img'], [0, 1, 2], 0.4, [0.001] * 3, 12)
        assert_matches_recorded(ora, run['out'], f'random seed {seed}')


def test_transforms_match_reference():
    """8x8 DCT / IDCT restatement vs ooura/dct.c on random and extreme blocks (denormals included)."""
    ora = H.load_oracle()
    blocks, want_dct, want_idct = load_reference_transforms()
    for i, (b, wd, wi) in enumerate(zip(blocks, want_dct, want_idct)):
        assert block_crc(H.transform8x8(ora.oracle_dct8x8, b)) == wd, f'DCT of block {i}'
        assert block_crc(H.transform8x8(ora.oracle_idct8x8, b)) == wi, f'IDCT of block {i}'


def test_oracle_objective_log_decreases():
    """Sanity of the logged objective (compute.c:271-272): finite, and lower at the end than at the start."""
    img = synth.synth_coefs(64, 64, 10, '4:2:0', 3)
    _, log = H.run_compute('oracle', img, [0, 1, 2], 0.3, [0.001] * 3, 30, want_log=True)
    assert np.isfinite(log).all()
    assert log[-1, 0] < log[0, 0]
    assert log[0, 1] == 0.0           # first step: DCT distance is exactly zero (cos == data*q)


def test_rgb_conversion_restatement():
    """png.c:39-62 restatement: truncation, clamping, 8 and 16 bit packing."""
    ora = H.load_oracle()
    y = np.array([[0.0, 255.0, 128.4, 300.0, -5.0, 16.999]], np.float32)
    cb = np.array([[0.0, 0.0, 10.0, 0.0, 0.0, -20.5]], np.float32)
    cr = np.array([[0.0, 0.0, -10.0, 0.0, 0.0, 30.25]], np.float32)
    out8 = np.zeros(6 * 3, np.uint8)
    ora.oracle_ycc_to_rgb(6, 1, 8, y.ctypes.data, 6, cb.ctypes.data, 6, cr.ctypes.data, 6, out8.ctypes.data)
    out8 = out8.reshape(6, 3)
    assert tuple(out8[0]) == (0, 0, 0) and tuple(out8[1]) == (255, 255, 255)
    assert tuple(out8[3]) == (255, 255, 255) and tuple(out8[4]) == (0, 0, 0)
    r = min(255.0, max(0.0, float(np.float32(128.4)) + 1.402 * -10.0))
    assert out8[2, 0] == int(np.float32(r))
    out16 = np.zeros(6 * 6, np.uint8)
    ora.oracle_ycc_to_rgb(6, 1, 16, y.ctypes.data, 6, cb.ctypes.data, 6, cr.ctypes.data, 6, out16.ctypes.data)
    v = out16.reshape(6, 3, 2)
    assert (int(v[1, 0, 0]) << 8 | int(v[1, 0, 1])) == 255 * 256


@pytest.mark.parametrize('seed', range(16))
def test_oracle_matches_reference_random_sweep(seed):
    """Randomised configurations (plane sizes, sampling factors up to 3x4, zero and non-zero weights,
    single-plane and joint mode, planes smaller than the frame; drawn by
    tests/golden/make_reference_runs.py): restatement == recorded reference."""
    run = load_reference_run(f'sweep{seed}')
    img = run['img']
    b = H.run_compute('oracle', img, run['channels'], run['weight'], run['pweight'], run['iterations'])
    assert_matches_recorded(b, run['out'], f"sweep seed {seed}: samp {[(p.w_samp, p.h_samp) for p in img.planes]} "
                                           f"dims {[(p.w, p.h) for p in img.planes]} channels {run['channels']} "
                                           f"w {run['weight']} p {run['pweight']} i {run['iterations']}")
