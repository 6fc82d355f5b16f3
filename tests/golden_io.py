"""Load tests/golden/case_*.npz back into a CoefImage + parameters, and the recorded runs of the
original jpeg2png in tests/golden/reference_runs.npz (written by tests/golden/make_reference_runs.py)."""
import glob
import hashlib
import os
import zlib

import numpy as np

from jpeg2png_b200.synth import CoefImage, Plane

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
REFERENCE_RUNS = os.path.join(GOLDEN_DIR, 'reference_runs.npz')
SAMPLE = 64             # output samples kept beside each plane's digest, to locate a mismatch


def golden_cases():
    return sorted(os.path.basename(p)[5:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, 'case_*.npz')))


def load_case(name):
    z = np.load(os.path.join(GOLDEN_DIR, f'case_{name}.npz'))
    planes = []
    for k in range(3):
        w, h, sw, sh = (int(v) for v in z[f'p{k}_dims'])
        planes.append(Plane(w=w, h=h, w_samp=sw, h_samp=sh, data=z[f'p{k}_data'], quant=z[f'p{k}_quant']))
    img = CoefImage(width=int(z['width']), height=int(z['height']), planes=planes)
    channels = [int(c) for c in z['channels']]
    fdata = [z[f'fdata{k}'] for k in range(len(channels))]
    out = [z[f'out{k}'] for k in range(len(channels))]
    return dict(img=img, channels=channels, weight=float(z['weight']), pweight=[float(v) for v in z['pweight']],
                iterations=int(z['iterations']), fdata=fdata, out=out)


def plane_digest(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype='<f4').tobytes()).digest()


def sample_index(size):
    """Positions of the recorded samples of a flattened plane: SAMPLE evenly spaced ones."""
    return np.linspace(0, size - 1, min(size, SAMPLE)).astype(np.int64)


def record_image(prefix, img):
    """The `struct coef` contents of img as npz fields (inputs are stored, not regenerated: the
    synthetic images go through numpy's transcendental functions, whose last bits vary by CPU)."""
    blob = {f'{prefix}size': np.array([img.width, img.height]),
            f'{prefix}dims': np.array([[p.w, p.h, p.w_samp, p.h_samp] for p in img.planes]),
            f'{prefix}quant': np.array([p.quant for p in img.planes], np.uint16)}
    for k, p in enumerate(img.planes):
        blob[f'{prefix}data{k}'] = np.asarray(p.data, np.int16)
    return blob


def record_planes(prefix, planes):
    """Output planes as npz fields: shapes, SHA-256 of the float32 bits, a few sampled values."""
    planes = [np.ascontiguousarray(p, np.float32) for p in planes]
    return {f'{prefix}out_shape': np.array([p.shape for p in planes]),
            f'{prefix}out_sha256': np.array([np.frombuffer(plane_digest(p), np.uint8) for p in planes]),
            f'{prefix}out_values': np.array([p.reshape(-1)[sample_index(p.size)] for p in planes])}


def _planes(z, prefix):
    return [dict(shape=tuple(int(v) for v in shape), sha256=sha.tobytes(), values=values)
            for shape, sha, values in zip(z[prefix + 'out_shape'], z[prefix + 'out_sha256'], z[prefix + 'out_values'])]


def load_reference_run(name):
    """One recorded compute() call of the original jpeg2png: inputs, parameters and output planes.
    'scalar_out' is present when the run was also recorded from the build without SIMD."""
    z = np.load(REFERENCE_RUNS)
    p = f'{name}.'
    channels = [int(c) for c in z[p + 'channels']]
    dims = z[p + 'dims']
    img = CoefImage(width=int(z[p + 'size'][0]), height=int(z[p + 'size'][1]),
                    planes=[Plane(w=int(dims[k][0]), h=int(dims[k][1]), w_samp=int(dims[k][2]), h_samp=int(dims[k][3]),
                                  data=z[f'{p}data{k}'], quant=z[p + 'quant'][k]) for k in range(3)])
    run = dict(img=img, channels=channels, weight=float(z[p + 'weight']), pweight=[float(v) for v in z[p + 'pweight']],
               iterations=int(z[p + 'iterations']), out=_planes(z, p))
    if p + 'scalar_out_sha256' in z.files:
        run['scalar_out'] = _planes(z, p + 'scalar_')
    return run


def block_crc(a):
    return zlib.crc32(np.ascontiguousarray(a, dtype='<f4').tobytes())


def load_reference_transforms():
    """Blocks, and the CRC-32 of the bits the original's 8x8 DCT and IDCT (ooura/dct.c) turned each into."""
    z = np.load(REFERENCE_RUNS)
    return z['transforms.blocks'], z['transforms.dct_crc32'], z['transforms.idct_crc32']


def assert_matches_recorded(got, recorded, what=''):
    """Bit for bit against a recorded run: every plane's digest must match; on a mismatch the
    recorded sample tells where the planes differ and by how much."""
    assert len(got) == len(recorded), f'{what}: {len(got)} planes vs {len(recorded)} recorded'
    for k, (p, r) in enumerate(zip(got, recorded)):
        assert p.shape == r['shape'], f'{what} plane {k}: shape {p.shape} vs recorded {r["shape"]}'
        if plane_digest(p) == r['sha256']:
            continue
        idx = sample_index(p.size)
        vals = np.ascontiguousarray(p, np.float32).reshape(-1)[idx]
        bad = np.flatnonzero(vals.view(np.uint32) != r['values'].view(np.uint32))
        detail = 'all recorded samples agree'
        if bad.size:
            i = bad[0]
            pos = tuple(int(v) for v in np.unravel_index(idx[i], p.shape))
            diff = np.abs(vals[bad].astype(np.float64) - r['values'][bad].astype(np.float64))
            detail = (f'{bad.size} of {vals.size} recorded samples differ; first at {pos}: {vals[i]!r} vs '
                      f'{r["values"][i]!r}; max abs diff among them {float(diff.max())}')
        raise AssertionError(f'{what} plane {k}: bits differ from the recorded run ({detail})')
