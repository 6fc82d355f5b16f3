"""Row strips of one frame over several B200s (pytest -m gpu on a box with >= 2 GPUs): the product's
strip sessions against the CHECKER (the compiled reference's compute() when it travelled, else the
oracle restatement) — not merely against the single-GPU product.  Skipped on a single-GPU box.

Three drivers of the same iteration are covered:
  torchdist  jpeg2png_b200/strips.py drives both exchanges with torch.distributed (NCCL)
  native     j2p_session_iterate_strip with the peer-memory protocol (default): the exchanges
             happen inside the two solver kernels over NVLink, cudaIpc mappings
  nccl       the same entry point with J2P_STRIP_P2P=0: NCCL launches between the kernels
  unfused    peer memory, but the border rows travel in the stand-alone halo kernel
             (J2P_STRIP_FUSED_HALO=0; what frames with uncovered columns use)
  tma        peer memory with the luma plane projected by the TMA kernel (J2P_PROJ_TMA=1), whose
             warp tiles deliver the fused border rows"""
import os
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CASES = {
    # several CTAs per row band and per tile row, ragged right edge, 25 iterations
    'c420': dict(w=640, h=512, q=20, ss='4:2:0', weight=0.3, pw=[0.001] * 3, iters=25, tile=None),
    'c444': dict(w=712, h=384, q=40, ss='4:4:4', weight=0.3, pw=[0.001, 0.002, 0.0], iters=20, tile=None),
    # luma 1928 wide in a 1936-wide frame: stepped-only columns at the strip borders -> stand-alone halo kernel
    'uncovered': dict(w=1928, h=256, q=30, ss='4:2:0', weight=0.3, pw=[0.001] * 3, iters=12, tile=None),
}
MODES = {'torchdist': {}, 'native': {}, 'nccl': {'J2P_STRIP_P2P': '0'}, 'unfused': {'J2P_STRIP_FUSED_HALO': '0'},
         'tma': {'J2P_PROJ_TMA': '1'}}


def _frame(case):
    from jpeg2png_b200 import synth
    if case['tile']:
        base = synth.synth_coefs(-(-case['w'] // 64) * 16, -(-case['h'] // 64) * 16, case['q'], case['ss'], seed=1238)
        return synth.tile_coefs(base, 4, 4, case['w'], case['h'])
    return synth.synth_coefs(case['w'], case['h'], case['q'], case['ss'], seed=777)


def _worker(rank, world, init_file, out_dir, mode, case):
    for k, v in MODES[mode].items():
        os.environ[k] = v
    import torch
    import torch.distributed as dist
    from jpeg2png_b200 import abi, strips
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', init_method=f'file://{init_file}', rank=rank, world_size=world,
                            device_id=torch.device('cuda', rank))
    try:
        lib = abi.load_product()
        img = _frame(case)
        mcu = 8 * max(p.h_samp for p in img.planes)
        row0, rows = strips.plan_strips(img.frame_h, mcu, world)[rank]
        be = strips.ProductStrip(lib, img, case['weight'], case['pw'], case['iters'], row0, rows, rank)
        if mode == 'torchdist':
            strips.solve_strips(be, dist, rank, world, case['iters'])
        else:
            # the library's own loop, in two calls to cover the continuation path, then once more
            # from a re-armed session (sequence numbers keep running across solves)
            comm = strips.native_comm(be, dist, rank, world)
            first = max(1, case['iters'] // 3)
            strips.solve_strips_native(be, comm, first)
            strips.solve_strips_native(be, comm, case['iters'] - first)
            run1 = [be.download(c) for c in range(3)]
            assert lib.j2p_session_reset(be.s) == 0
            strips.solve_strips_native(be, comm, case['iters'])
            for c in range(3):
                assert (run1[c].view(np.uint32) == be.download(c).view(np.uint32)).all(), 'second solve differs from the first'
        np.savez(os.path.join(out_dir, f'rank{rank}.npz'), rows=rows, **{f'p{c}': be.download(c) for c in range(3)})
        if mode != 'torchdist':
            assert lib.j2p_comm_status(comm) == 0, lib.j2p_last_error().decode()
            want_protocol = 0 if mode == 'nccl' or world > 8 else 1
            assert lib.j2p_comm_protocol(comm) == want_protocol, f'protocol {lib.j2p_comm_protocol(comm)}, expected {want_protocol}'
            lib.j2p_comm_destroy(comm)
        be.close()
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _run(world, mode, case, tmp_path, iters_check=None):
    import torch
    import torch.multiprocessing as mp
    from tests import helpers as H
    if torch.cuda.device_count() < world:
        pytest.skip(f'needs {world} GPUs')
    init_file = tempfile.mktemp(dir=str(tmp_path))
    mp.spawn(_worker, args=(world, init_file, str(tmp_path), mode, case), nprocs=world, join=True)
    img = _frame(case)
    checker = 'ref' if H.have_ref() else 'oracle'
    want = H.run_compute(checker, img, [0, 1, 2], case['weight'], case['pw'], case['iters'])
    parts = [np.load(os.path.join(str(tmp_path), f'rank{r}.npz')) for r in range(world)]
    got = [np.concatenate([p[f'p{c}'] for p in parts], axis=0) for c in range(3)]
    H.assert_bit_identical(got, want, f'{world} strips ({mode}) vs {checker}')


@pytest.mark.parametrize('mode', list(MODES))
@pytest.mark.parametrize('world', [2, 4, 8])
def test_strips_match_reference(world, mode, tmp_path):
    _run(world, mode, CASES['c420'], tmp_path)


@pytest.mark.parametrize('name', ['c444', 'uncovered'])
def test_strips_other_geometries(name, tmp_path):
    _run(2, 'native', CASES[name], tmp_path)


@pytest.mark.parametrize('world', [2, 8])
def test_8k_strips_match_reference(world, tmp_path):
    """BASELINE config 4's frame (7680x4320 4:2:0) in row strips, 10 iterations, against the
    compiled reference: the strong-scaling workload of bench.py at the size it is measured on."""
    case = dict(w=7680, h=4320, q=10, ss='4:2:0', weight=0.3, pw=[0.001] * 3, iters=10, tile=True)
    _run(world, 'native', case, tmp_path)
