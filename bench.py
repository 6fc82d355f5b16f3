#!/usr/bin/env python
"""bench.py — headline benchmark of the jpeg2png solver hot path on B200.

Workload (BASELINE.json metric, configs[2]): one 3840x2160 Q50 4:4:4 frame, all three planes
optimised jointly, `-i 100 -w 0.3 -p 0.001` (reference defaults).  A *step* is one complete solve
of one frame = 100 solver iterations = 200 kernel launches.  Metric: Mpixel-iterations/s =
image_w * image_h * iterations / t / 1e6, whole job over all N GPUs.

  value     solve with the coefficient planes ALREADY resident in HBM (session layer); the timed
            region includes re-arming the iterate (reference aux_init) but no host traffic.
  e2e       the same solve through the drop-in `compute()` with HOST `struct coef` buffers
            (malloc-family memory, as the reference contract requires): H2D of data + quant +
            conventional decode, 100 iterations, D2H of the three result planes, all timed.
  roofline  the dominant kernel's ALGORITHMIC bytes per launch / its mean launch duration measured
            live with CUDA events on the session stream (j2p_session_profile), against the
            measured HBM copy bandwidth in MEASURED_PEAKS.json.
  cpu_baseline  the unmodified reference compute() (oracle/_ref, SSE2+OpenMP build) — or the
            oracle port where that is absent — timed on this box's host cores on a bounded sample.

N > 1 (torchrun): the path shards by independent frames (reference jpeg2png.c:330 file loop,
BASELINE config 5 style): every rank solves its own frame on its own GPU, no data-path
collective; NCCL is only used for the barrier and the max-over-ranks of the device time.
Scaling is therefore "weak".

  strong    (beside the weak-scaling `value`) ONE 7680x4320 4:2:0 frame cut into N row strips, the
            only multi-GPU mode that communicates: device time per iteration, speed-up over the
            whole frame on one GPU measured in the same run, bit-identity with that 1-GPU result.
  parity_at_size  N=1: the product's first 20 iterations of the bench frame against the
            reference's, bit for bit (the cpu_baseline call produces the reference planes anyway).

`--impl reference` times the reference CPU implementation instead (rank 0 only).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WIDTH, HEIGHT, QUALITY, SUBSAMPLING, ITERATIONS = 3840, 2160, 50, '4:4:4', 100
WEIGHT, PWEIGHT = 0.3, 0.001
SEED = 1234 + 3
WORKLOAD = '3840x2160 Q50 4:4:4 synthetic JPEG coefficients, joint 3 planes, -i 100 -w 0.3 -p 0.001'
METRIC = 'Mpixel-iterations/s'
FALLBACK_HBM_GBS = 6650.0
DUMP_BYTES = 64 * 10**6          # --dump-outputs writes at most this much in all
DUMP_SEED = 20240601


def algorithmic_bytes(img, nchannel=3):
    """Bytes one launch of each kernel must move (DESIGN.md §4), per frame.

    Per plane-pixel with s = w_samp*h_samp:
      k_gradient: read x_k 4 + x_{k-1} 4 + gp 4/s, write g 4                      = 12 + 4/s
      k_project : read x_k 4 + x_{k-1} 4 + g 4 + data 2/s, write x_{k+1} 4 + gp 4/s = 16 + 6/s
    (SURVEY.md §8d's two-pass figure is 28 + 12/s; this design needs 28 + 10/s because the
    DCT-distance gradient is produced inside k_project and k_gradient never reads `data`.)
    """
    n = img.frame_w * img.frame_h
    grad = proj = 0.0
    for p in img.planes[:nchannel]:
        s = p.w_samp * p.h_samp
        cover = (p.w * p.h) / (n / s) if n else 1.0      # planes whose grid is smaller than the frame
        grad += n * 12 + n / s * 4 * cover
        proj += n * 16 + n / s * 6 * cover
    return grad, proj


def sample_clocks(stop, out, device):
    """nvidia-smi clocks + throttle reasons during the timed region."""
    q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    try:
        p = subprocess.Popen(['nvidia-smi', f'--id={device}', f'--query-gpu={q}', '--format=csv,noheader,nounits', '-lms', '100'],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except OSError:
        return

    def reader():
        for line in p.stdout:
            out.append(line.strip())
    t = threading.Thread(target=reader, daemon=True)
    t.start()
    stop.wait()
    p.terminate()
    try:
        p.wait(timeout=2)
    except Exception:
        p.kill()


def summarise_clocks(lines):
    sm, mx, reasons = [], [], set()
    names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
    for ln in lines:
        f = [x.strip() for x in ln.split(',')]
        if len(f) < 7:
            continue
        try:
            sm.append(float(f[0]))
            mx.append(float(f[1]))
        except ValueError:
            continue
        for name, v in zip(names, f[3:7]):
            if v.lower().startswith('active'):
                reasons.add(name)
    if not sm:
        return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
    busy = sorted(sm)[len(sm) // 2:]           # upper half = samples taken under load
    return {'sm_mhz': float(np.median(busy)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons), 'samples': len(sm)}


def measured_peak():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        return FALLBACK_HBM_GBS, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def recorded_traffic(kernel):
    """dram bytes per launch from the committed ncu --set full capture (profiles/), or None."""
    path = os.path.join(ROOT, 'profiles', 'traffic.json')
    try:
        with open(path) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


def emit(line, world):
    """Rank 0's one JSON line.  Under torchrun on the GPU boxes the workers' stdout has been seen
    arriving on the launcher's stderr (gpurun_out/bench_n2.* in round 1), so for N > 1 the same
    line is written to both streams; the two copies are identical."""
    text = json.dumps(line)
    print(text, flush=True)
    if world > 1:
        print(text, file=sys.stderr, flush=True)


def dump_outputs(directory, arrays):
    """Write each float32 array as DIR/<name>.npy.  When they are larger than DUMP_BYTES together,
    each is replaced by the same fixed, seeded sample of its flattened elements (positions sorted),
    so two runs with the same arguments write files that compare element for element."""
    os.makedirs(directory, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, np.float32) for k, v in arrays.items()}
    header = 128                                  # .npy header of a 1-D or 2-D float32 array
    if sum(a.nbytes + header for a in arrays.values()) > DUMP_BYTES:
        keep = (DUMP_BYTES // len(arrays) - header) // 4
        for k, a in arrays.items():
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(a.size, size=min(keep, a.size), replace=False))
            arrays[k] = a.reshape(-1)[idx]
        print(f'bench.py: outputs sampled to {keep} of their elements each (seed {DUMP_SEED})', file=sys.stderr, flush=True)
    for k, a in arrays.items():
        np.save(os.path.join(directory, f'{k}.npy'), a)


def make_frame(seed):
    from jpeg2png_b200 import synth
    return synth.synth_coefs(WIDTH, HEIGHT, QUALITY, SUBSAMPLING, seed)


# ---------------------------------------------------------------------------------------------
# reference arm / cpu baseline
# ---------------------------------------------------------------------------------------------
def cpu_solve_rate(img, fdata, iterations, kind, keep=None):
    """Time ONE compute() call of `iterations` iterations with the CPU checker (host marshalling
    excluded); returns (Mpix-it/s, seconds).  keep: a list that receives the result planes."""
    from tests import helpers as H
    timer = {}
    out = H.run_compute(kind, img, [0, 1, 2], WEIGHT, [PWEIGHT] * 3, iterations, fdata, timer=timer)
    if keep is not None:
        keep.extend(out)
    dt = timer['seconds']
    return img.width * img.height * iterations / dt / 1e6, dt


def usable_cpus():
    """CPUs this process may really use: the affinity mask capped by the cgroup CPU quota (the GPU
    boxes show 128 hardware threads but grant 16 CPUs; an OpenMP team wider than the quota spins
    itself into being throttled, which would make the CPU arm look slower than it is)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        quota, period = open('/sys/fs/cgroup/cpu.max').read().split()[:2]
        if quota != 'max':
            n = min(n, max(1, -(-int(quota) // int(period))))
    except (OSError, ValueError):
        pass
    return max(1, n)


def cpu_kind_and_cores():
    """Which CPU checker is the baseline, and with how many threads.  The OpenMP team is set
    explicitly to the CPUs this process may use: torchrun exports OMP_NUM_THREADS=1 to its workers,
    which would otherwise silently shrink the reference arm at N > 1."""
    from tests import helpers as H
    if H.have_ref():
        lib = H.load_ref()
        cores = usable_cpus()
        lib.ref_glue_set_threads(cores)
        return 'ref', 'reference', cores
    H.build_oracle_libs()
    return 'oracle', 'port', 1


def cpu_separate_mode_rate(img, fdata, iterations, kind):
    """The reference's -s mode (jpeg2png.c:147-152): three concurrent compute(1, ...) calls, one
    per plane, weights {w, 0, 0}.  Three host threads here (ctypes releases the GIL)."""
    from tests import helpers as H
    weights = [WEIGHT, 0.0, 0.0]
    t0 = time.perf_counter()
    ts = [threading.Thread(target=H.run_compute, args=(kind, img, [c], weights[c], [PWEIGHT], iterations, [fdata[c]])) for c in range(3)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    dt = time.perf_counter() - t0
    return img.width * img.height * iterations / dt / 1e6, dt


def cpu_file_parallel_rate(img, fdata, iterations, kind, nfiles):
    """The reference's file loop (jpeg2png.c:330): `nfiles` frames solved concurrently, each in
    joint mode.  Aggregate Mpix-it/s over all of them."""
    from tests import helpers as H
    t0 = time.perf_counter()
    ts = [threading.Thread(target=H.run_compute, args=(kind, img, [0, 1, 2], WEIGHT, [PWEIGHT] * 3, iterations, fdata)) for _ in range(nfiles)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    dt = time.perf_counter() - t0
    return nfiles * img.width * img.height * iterations / dt / 1e6, dt


def cpu_warmup(kind):
    """OpenMP cold start (about 1 s on first use) must not land in a timed call."""
    from jpeg2png_b200 import synth
    from tests import helpers as H
    small = synth.synth_coefs(64, 64, 50, '4:4:4', 1)
    H.run_compute(kind, small, [0, 1, 2], WEIGHT, [PWEIGHT] * 3, 2)


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    kind, label, cores = cpu_kind_and_cores()
    img = make_frame(SEED)
    cpu_warmup(kind)
    # bounded sample: per-iteration cost does not depend on the iteration count, so every step
    # solves the same frame for `it` iterations, sized so the whole run stays within ~3 minutes
    budget_s = 120.0
    per_iter_s = 0.65
    it = int(max(1, min(ITERATIONS, budget_s / ((args.steps + args.warmup) * per_iter_s))))
    from tests import helpers as H
    fdata = H.decode_planes(img)
    for _ in range(args.warmup):
        cpu_solve_rate(img, fdata, it, kind)
    dt = 0.0
    planes = []
    for k in range(args.steps):
        dt += cpu_solve_rate(img, fdata, it, kind, keep=planes if k == args.steps - 1 else None)[1]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {f'plane{c}': p for c, p in enumerate(planes)})
    value = img.width * img.height * it * args.steps / dt / 1e6
    sample = f'{WIDTH}x{HEIGHT} 4:4:4 frame, {it} of {ITERATIONS} iterations per step (per-iteration cost is iteration-count independent)'
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'Mpix-it/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'sample': sample},
        'cpu_baseline': {'value': value, 'unit': 'Mpix-it/s', 'cores': cores, 'kind': label, 'sample': sample},
        'e2e': {'value': value, 'unit': 'Mpix-it/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# product arm
# ---------------------------------------------------------------------------------------------
def run_product_arm(args, rank, local_rank, world):
    import torch
    from jpeg2png_b200 import abi

    if not torch.cuda.is_available():
        raise RuntimeError('bench.py: no CUDA device; the solver has no CPU path to fall back to')
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    lib = abi.load_product()

    img = make_frame(SEED + rank)               # every rank solves its own frame
    W, H = img.frame_w, img.frame_h

    def barrier():
        if dist is not None:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- resident session -------------------------------------------------------------------
    d = abi.FrameDesc()
    d.nchannel = 3
    for c, p in enumerate(img.planes):
        d.plane_w[c], d.plane_h[c], d.w_samp[c], d.h_samp[c] = p.w, p.h, p.w_samp, p.h_samp
        d.pweight[c] = PWEIGHT
    d.weight = WEIGHT
    d.iterations = ITERATIONS
    s = C.c_void_p()
    if lib.j2p_session_create(C.byref(s), local_rank, C.byref(d)) != 0:
        raise RuntimeError(lib.j2p_last_error().decode())
    for c, p in enumerate(img.planes):
        data = np.ascontiguousarray(p.data)
        quant = np.ascontiguousarray(p.quant)
        # fdata = NULL: the conventional decode runs on the device (jpeg.c:83-92 restated in k_decode)
        if lib.j2p_session_upload(s, c, data.ctypes.data, quant.ctypes.data, None) != 0:
            raise RuntimeError(lib.j2p_last_error().decode())
    stream = torch.cuda.ExternalStream(lib.j2p_session_stream(s), device=torch.device('cuda', local_rank))

    def solve_resident():
        if lib.j2p_session_iterate(s, 0, ITERATIONS) != 0:
            raise RuntimeError(lib.j2p_last_error().decode())

    for _ in range(max(args.warmup, 3)):
        solve_resident()
    lib.j2p_session_sync(s)

    clock_lines, stop = [], threading.Event()
    sampler = None
    if rank == 0:
        sampler = threading.Thread(target=sample_clocks, args=(stop, clock_lines, local_rank), daemon=True)
        sampler.start()
        time.sleep(0.3)

    launches0 = lib.j2p_session_launches(s)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        solve_resident()
    ev1.record(stream)
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    launches = int(lib.j2p_session_launches(s) - launches0)
    if args.dump_outputs and rank == 0:
        # the three frame planes the last timed solve left in HBM, before anything else runs on the session
        planes = {}
        for c in range(3):
            planes[f'plane{c}'] = np.empty((H, W), np.float32)
            if lib.j2p_session_download(s, c, planes[f'plane{c}'].ctypes.data) != 0:
                raise RuntimeError(lib.j2p_last_error().decode())
        dump_outputs(args.dump_outputs, planes)

    # ---- per-kernel live timing for the roofline (rank 0, N=1 semantics: one GPU's kernels) ----
    mg, mp = C.c_float(), C.c_float()
    if lib.j2p_session_profile(s, 20, C.byref(mg), C.byref(mp)) != 0:
        raise RuntimeError(lib.j2p_last_error().decode())
    lib.j2p_session_sync(s)

    # result checksum of the resident solve (kept out of the timed region)
    solve_resident()
    out = np.empty((H, W), np.float32)
    lib.j2p_session_download(s, 0, out.ctypes.data)
    checksum = float(np.float64(out).sum())
    lib.j2p_session_destroy(s)

    # The clock sampler covers the device-timed region above.  It is stopped before the end-to-end
    # leg: a polling nvidia-smi takes driver locks that stall the CUDA API calls of this process,
    # and the e2e leg is exactly the host-API path (measured: 65 ms per 4K solve with the poller
    # running, 36 ms without; profiles/r01_notes.md).  J2P_BENCH_SAMPLE_E2E=1 keeps it running.
    keep_sampling = os.environ.get('J2P_BENCH_SAMPLE_E2E') == '1'
    if sampler is not None and not keep_sampling:
        stop.set()
        sampler.join(timeout=3)

    # ---- end to end through compute() with host buffers --------------------------------------
    # the conventional decode the caller of compute() owns (jpeg2png.c:127-139): produced once,
    # outside the timed region, by the product's own device decode
    fdata = device_decode(lib, img, local_rank)
    h2d = sum(p.data.nbytes + p.quant.nbytes + p.w * p.h * 4 for p in img.planes)
    d2h = 3 * W * H * 4
    n_e2e = args.steps
    arrays = [abi.CoefArray(img, [0, 1, 2], fdata) for _ in range(n_e2e + 1)]
    pw = (C.c_float * 3)(PWEIGHT, PWEIGHT, PWEIGHT)
    lg = abi.Logger(None, b'', 3, 0)
    os.environ['J2P_DEVICE'] = str(local_rank)
    lib.compute(3, arrays[0].arr, C.byref(lg), None, C.c_float(WEIGHT), pw, ITERATIONS)     # warm-up
    barrier()
    t0 = time.perf_counter()
    for k in range(n_e2e):
        lib.compute(3, arrays[1 + k].arr, C.byref(lg), None, C.c_float(WEIGHT), pw, ITERATIONS)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e_checksum = float(np.float64(arrays[1].result(0)).sum())
    for a in arrays:
        a.release()
    if sampler is not None and keep_sampling:
        stop.set()
        sampler.join(timeout=3)

    strong = None
    if os.environ.get('J2P_BENCH_STRONG', '1') != '0':
        strong = run_strong(lib, torch, dist, rank, local_rank, world)

    if rank == 0:
        pix_it = WIDTH * HEIGHT * ITERATIONS
        value = world * pix_it * args.steps / (ms_total * 1e-3) / 1e6
        e2e_value = world * pix_it * n_e2e / e2e_s / 1e6
        peak, peak_src = measured_peak()
        gb, pb = algorithmic_bytes(img)
        kernels = [
            {'name': 'k_gradient', 'ms': float(mg.value), 'bytes': gb},
            {'name': 'k_project', 'ms': float(mp.value), 'bytes': pb},
        ]
        for k in kernels:
            k['gbs'] = k['bytes'] / (k['ms'] * 1e-3) / 1e9
            k['frac'] = k['gbs'] / peak
            k['traffic'] = recorded_traffic(k['name'])
        dom = max(kernels, key=lambda k: k['ms'])
        roofline = {'bound': 'hbm', 'kernel': dom['name'], 'achieved': dom['gbs'], 'peak': peak, 'unit': 'GB/s',
                    'frac': dom['frac'], 'traffic': dom['traffic'], 'peak_source': peak_src,
                    'algorithmic_bytes_per_launch': dom['bytes'], 'ms_per_launch': dom['ms'],
                    'kernels': kernels,
                    # the two kernels of an iteration, each timed on its own (events around every launch)
                    'iteration': {'bytes': gb + pb, 'ms': float(mg.value + mp.value),
                                  'gbs': (gb + pb) / ((mg.value + mp.value) * 1e-3) / 1e9,
                                  'frac': (gb + pb) / ((mg.value + mp.value) * 1e-3) / 1e9 / peak},
                    # the same bytes over the iteration's share of the timed region (`value`): kernels queued
                    # back to back, launch gaps included — the whole-iteration figure of SURVEY.md §8(d)
                    'iteration_in_solve': {'bytes': gb + pb, 'ms': ms_total / args.steps / ITERATIONS,
                                           'gbs': (gb + pb) / (ms_total / args.steps / ITERATIONS * 1e-3) / 1e9,
                                           'frac': (gb + pb) / (ms_total / args.steps / ITERATIONS * 1e-3) / 1e9 / peak}}
        cpu = None
        parity_at_size = None
        if world == 1:
            kind, label, cores = cpu_kind_and_cores()
            cpu_warmup(kind)
            sample_it = 20
            ref_planes = []
            rate, secs = cpu_solve_rate(img, fdata, sample_it, kind, keep=ref_planes)
            # parity AT THE BENCHMARKED SIZE: the product's first `sample_it` iterations of the same
            # frame through compute(), bit for bit against what the reference just produced
            from tests import helpers as checker        # (H is the frame height in this function)
            got = checker.run_compute('product', img, [0, 1, 2], WEIGHT, [PWEIGHT] * 3, sample_it, fdata)
            same = all((checker.bits(a) == checker.bits(b)).all() for a, b in zip(got, ref_planes))
            parity_at_size = {'result': 'bit-identical' if same else 'MISMATCH', 'against': label,
                              'what': f'{WIDTH}x{HEIGHT} 4:4:4 joint, first {sample_it} iterations, all three planes'}
            if not same:
                parity_at_size['max_abs_diff'] = float(max(np.max(np.abs(a.astype(np.float64) - b)) for a, b in zip(got, ref_planes)))
            del got, ref_planes
            sep_rate, sep_secs = cpu_separate_mode_rate(img, fdata, 10, kind)
            nfiles = max(1, min(4, cores // 3))
            fp_rate, fp_secs = cpu_file_parallel_rate(img, fdata, 5, kind, nfiles)
            cpu = {'value': rate, 'unit': 'Mpix-it/s', 'cores': cores, 'kind': label,
                   'sample': f'{WIDTH}x{HEIGHT} 4:4:4 joint, {sample_it} of {ITERATIONS} iterations, one call, {secs:.1f} s '
                             '(joint mode threads over the 3 planes only; TV/TGV passes are serial, compute.c:233,253,260)',
                   'separate_mode': {'value': sep_rate, 'unit': 'Mpix-it/s',
                                     'sample': f'-s mode, 3 concurrent compute(1,..) (jpeg2png.c:147-152), 10 iterations, {sep_secs:.1f} s'},
                   'file_parallel': {'value': fp_rate, 'unit': 'Mpix-it/s',
                                     'sample': f'{nfiles} frames solved concurrently, joint mode (jpeg2png.c:330), 5 iterations each, {fp_secs:.1f} s'}}
        line = {
            'metric': METRIC, 'value': value, 'unit': 'Mpix-it/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': ms_total / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'frames_per_step': world, 'sharding': 'one frame per GPU, no data-path collective',
                       'l2': 'working set ~0.75 GB per frame >> 126 MB L2 (no flush needed)',
                       'frame': [W, H], 'iterations': ITERATIONS},
            'clocks': dict(summarise_clocks(clock_lines), region='device-timed region' + (' and e2e leg' if keep_sampling else ' (poller stopped before the e2e leg)')),
            'e2e': {'value': e2e_value, 'unit': 'Mpix-it/s', 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                    'ms_per_step': e2e_s / n_e2e * 1e3, 'host_memory': 'pageable malloc-family buffers (reference struct coef contract)',
                    'api': 'compute(3, coefs, log, NULL, 0.3, pweights, 100) via libjpeg2png_b200.so'},
            'gpu_launches': launches,
            'roofline': roofline,
            'cpu_baseline': cpu,
            'parity_at_size': parity_at_size,
            'strong': strong,
            'checksum': {'resident': checksum, 'e2e': e2e_checksum},
        }
        line['roofline']['iteration_frac'] = roofline['iteration_in_solve']['frac']
        emit(line, world)
    if dist is not None:
        dist.destroy_process_group()


STRONG = dict(width=7680, height=4320, quality=10, subsampling='4:2:0', iterations=100, seed=1238)


def run_strong(lib, torch, dist, rank, local_rank, world):
    """Strong scaling of ONE frame (BASELINE config 4's frame: 7680x4320 Q10 4:2:0, joint, 100
    iterations here): the frame is cut into `world` MCU-aligned row strips, one per GPU
    (j2p_session_create_strip); an iteration is the two solver kernels with the exchanges inside
    them over NVLink peer memory (j2p_session_iterate_strip, DESIGN.md §7).  Device time with CUDA
    events on the session streams, max over ranks.  In the same run rank 0 also solves the whole
    frame on its own GPU: that is the 1-GPU time the speed-up is quoted against, and the bits every
    strip must reproduce (CRC32 of every rank's rows against the same rows of the 1-GPU result).
    Collective: every rank calls it.  Returns the block on rank 0, None elsewhere."""
    import zlib
    from jpeg2png_b200 import abi, strips, synth
    W, H, it = STRONG['width'], STRONG['height'], STRONG['iterations']
    base = synth.synth_coefs(-(-W // 64) * 16, -(-H // 64) * 16, STRONG['quality'], STRONG['subsampling'], STRONG['seed'])
    img = synth.tile_coefs(base, 4, 4, W, H)     # a quarter-size cartoon tiled 4x4 at block level: seconds of host time, same statistics
    mcu = 8 * max(p.h_samp for p in img.planes)
    plan = strips.plan_strips(img.frame_h, mcu, world)
    dev = torch.device('cuda', local_rank)

    def barrier():
        if dist is not None:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    # ---- the whole frame on one GPU (rank 0) ------------------------------------------------
    single_ms, ref_crcs = None, None
    if rank == 0:
        d = abi.FrameDesc()
        d.nchannel = 3
        for c, p in enumerate(img.planes):
            d.plane_w[c], d.plane_h[c], d.w_samp[c], d.h_samp[c] = p.w, p.h, p.w_samp, p.h_samp
            d.pweight[c] = PWEIGHT
        d.weight = WEIGHT
        d.iterations = it
        s = C.c_void_p()
        if lib.j2p_session_create(C.byref(s), local_rank, C.byref(d)) != 0:
            raise RuntimeError(lib.j2p_last_error().decode())
        for c, p in enumerate(img.planes):
            data, quant = np.ascontiguousarray(p.data), np.ascontiguousarray(p.quant)
            if lib.j2p_session_upload(s, c, data.ctypes.data, quant.ctypes.data, None) != 0:
                raise RuntimeError(lib.j2p_last_error().decode())
        stream = torch.cuda.ExternalStream(lib.j2p_session_stream(s), device=dev)
        for _ in range(2):
            lib.j2p_session_iterate(s, 0, 10)                      # warm-up
        lib.j2p_session_sync(s)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        if lib.j2p_session_iterate(s, 0, it) != 0:
            raise RuntimeError(lib.j2p_last_error().decode())
        e1.record(stream)
        lib.j2p_session_sync(s)
        single_ms = e0.elapsed_time(e1)
        ref_crcs = []
        for c in range(3):
            out = np.empty((img.frame_h, img.frame_w), np.float32)
            lib.j2p_session_download(s, c, out.ctypes.data)
            ref_crcs.append([zlib.crc32(out[r0:r0 + rows].tobytes()) for r0, rows in plan])
        lib.j2p_session_destroy(s)
    if world == 1:
        pix = W * H * it
        return {'workload': f"{W}x{H} Q{STRONG['quality']} {STRONG['subsampling']} synthetic JPEG coefficients, joint 3 planes, {it} iterations",
                'n_gpus': 1, 'us_per_iteration': single_ms / it * 1e3, 'mpix_it_s': pix / (single_ms * 1e-3) / 1e6,
                'single_gpu_us_per_iteration': single_ms / it * 1e3, 'speedup_vs_1gpu': 1.0}

    # ---- the same frame in `world` row strips -----------------------------------------------
    barrier()
    row0, rows = plan[rank]
    be = strips.ProductStrip(lib, img, WEIGHT, [PWEIGHT] * 3, it, row0, rows, local_rank)
    comm = strips.native_comm(be, dist, rank, world)
    strips.solve_strips_native(be, comm, 5)                         # warm-up: binds the peer memory, first-use costs
    lib.j2p_session_sync(be.s)
    barrier()
    if lib.j2p_session_reset(be.s) != 0:
        raise RuntimeError(lib.j2p_last_error().decode())
    lib.j2p_session_sync(be.s)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(be.stream)
    strips.solve_strips_native(be, comm, it)
    e1.record(be.stream)
    lib.j2p_session_sync(be.s)
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    strip_ms = float(t.item())
    status = int(lib.j2p_comm_status(comm))
    protocol = int(lib.j2p_comm_protocol(comm))
    crcs = [zlib.crc32(be.download(c).tobytes()) for c in range(3)]
    gathered = [None] * world
    dist.all_gather_object(gathered, (crcs, status))
    lib.j2p_comm_destroy(comm)
    be.close()
    barrier()
    if rank != 0:
        return None
    same = all(gathered[r][0][c] == ref_crcs[c][r] for r in range(world) for c in range(3))
    pix = W * H * it
    return {'workload': f"{W}x{H} Q{STRONG['quality']} {STRONG['subsampling']} synthetic JPEG coefficients, joint 3 planes, {it} iterations, "
                        f'ONE frame in {world} MCU-aligned row strips',
            'n_gpus': world, 'us_per_iteration': strip_ms / it * 1e3, 'mpix_it_s': pix / (strip_ms * 1e-3) / 1e6,
            'single_gpu_us_per_iteration': single_ms / it * 1e3, 'speedup_vs_1gpu': single_ms / strip_ms,
            'protocol': 'peer memory: both exchanges inside the solver kernels (NVLink stores + flags)' if protocol == 1 else 'NCCL all-gather + send/recv between the kernels',
            'exchange_status': 'ok' if all(g[1] == 0 for g in gathered) else 'TIMEOUT',
            'bit_identical_to_1gpu': bool(same),
            'timing': 'CUDA events on the session streams, max over ranks; the 1-GPU time is rank 0 solving the whole frame in the same run'}


def device_decode(lib, img, device):
    """Conventional decode of all planes on the device (session upload with fdata=NULL, 0 iterations)."""
    from jpeg2png_b200 import abi
    planes = []
    for c, p in enumerate(img.planes):
        d = abi.FrameDesc()
        d.nchannel = 1
        d.plane_w[0], d.plane_h[0], d.w_samp[0], d.h_samp[0] = p.w, p.h, 1, 1
        d.iterations = 0
        s = C.c_void_p()
        if lib.j2p_session_create(C.byref(s), device, C.byref(d)) != 0:
            raise RuntimeError(lib.j2p_last_error().decode())
        data = np.ascontiguousarray(p.data)
        quant = np.ascontiguousarray(p.quant)
        if lib.j2p_session_upload(s, 0, data.ctypes.data, quant.ctypes.data, None) != 0:
            raise RuntimeError(lib.j2p_last_error().decode())
        out = np.empty((p.h, p.w), np.float32)
        lib.j2p_session_download(s, 0, out.ctypes.data)
        lib.j2p_session_destroy(s)
        planes.append(out)
    return planes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the planes the last step computed as DIR/<name>.npy '
                         f'(float32; a fixed seeded sample when larger than {DUMP_BYTES // 10**6} MB in all)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if world != args.gpus and world > 1:
        args.gpus = world
    if args.impl == 'reference':
        run_reference_arm(args, rank, world)
    else:
        run_product_arm(args, rank, local_rank, world)


if __name__ == '__main__':
    main()
