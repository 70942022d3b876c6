#!/usr/bin/env python3
"""bench.py -- headline benchmark of the B200-native SG-SLAM tracking hot path (driver contract in the task statement).

  python bench.py --gpus N --steps K --warmup W [--impl ours|reference] [--config s2|720p|hamming] [--dump-outputs DIR]

config s2 (default; BASELINE.json configs[1], the configuration `metric` is quoted on): one "step" = one pass of the hot path over a batch of
synthetic 640x480 frames per GPU,

    colour frame -> Detector2D::detect (MobileNetV3-SSDLite, tcgen05 GEMMs) ------------------------\\
    gray frame   -> ORB extract -> LK to the previous frame -> (join) findFundamentalMat -> dyn-reject (boxes + epipolar) -> SearchByProjection(cur, last)

the detector's person boxes are produced on the device and consumed by the F estimate and the rejection in stream order (src/Frame.cc:474-500 joins
the detector thread at the same place).  Frames of independent streams are sharded over ranks with no data-path collective (weak scaling); one
ncclBroadcast of the shared vocabulary happens at start-up, untimed.
config 720p (configs[2]): the same step at 1280x720 / 2000 features.   config hamming (configs[4]): brute-force 256-bit Hamming sweep 1k..64k.

  value : whole-job frames/s with all inputs resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e   : the same step through sgs_tracker_step with HOST (pinned) buffers, H2D / D2H inside the timed region
  roofline     : dominant kernel's algorithmic bytes / its CUDA-event time vs the measured HBM copy peak (MEASURED_PEAKS.json)
  cpu_baseline : the reference's CPU path (oracle port, C++ worker threads pinned one per core) on this box's host cores, bounded sample
  --impl reference : that CPU path alone, on the same workload / frames per step
"""
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
for p in (os.path.join(ROOT, 'sg-slam_b200'), os.path.join(ROOT, 'oracle')):
    if p not in sys.path:
        sys.path.insert(0, p)

TH = 15.0                              # Tracking.cc:919-923 (RGB-D)
MODEL = os.path.join(ROOT, 'oracle', '_ref', 'ncnn_model', 'mobilenetv3_ssdlite_voc')      # the reference's trained model, staged by build()
DET_GFLOP = 1.115                      # SURVEY 8(d): 557.37 MMAC per 300x300 inference
CONFIGS = {
    's2':   dict(W=640, H=480, NFEAT=1000, batch=512, cam_scale=1.0, name='S2 walking_xyz-shaped synthetic 640x480 stream (BASELINE configs[1])'),
    '720p': dict(W=1280, H=720, NFEAT=2000, batch=192, cam_scale=2.0, name='S3 synthetic 1280x720 stream, 2000 features (BASELINE configs[2])'),
}
# launches of one tracker step: extract (7 resize, FAST, quadtree, blur, describe) + LK (3 pyrDown, 4 Scharr, 4 border, track) + RANSAC F + depth lookup + dyn-reject/compact (2) + match
TRACKER_LAUNCHES = 11 + 12 + 1 + 1 + 2 + 1


def alg_bytes(W, H, nk):
    """Algorithmic bytes per frame (SURVEY 8d): every stage reads its input once and writes its output once."""
    lv = [(W, H)]
    sf = 1.0
    for _ in range(7):
        sf *= 1.2
        lv.append((int(round(W / np.float32(sf))), int(round(H / np.float32(sf)))))
    px = [w * h for w, h in lv]
    pyr = sum(px[i - 1] + px[i] for i in range(1, 8))
    extract = pyr + sum(px) + 160 * nk + 749 * nk + 2 * sum(px) + 544 * nk + 28 * nk
    lk_pyr = int(W * H * (1 + 1 / 4 + 1 / 16 + 1 / 64) * 6 + W * H * (1 / 4 + 1 / 16 + 1 / 64) * 4)
    return dict(pyramid=pyr, fast=sum(px), blur=2 * sum(px), describe=(749 + 544 + 60) * nk, extract=extract, lk_pyr=lk_pyr, lk_track=nk * 4 * 2 * 529,
                fm=16 * nk + 72, track=76 * nk + 56 * nk + 44 * 8 * nk)


_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly one JSON line: everything libraries print there (e.g. the NCCL version banner) is sent to stderr instead."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + '\n').encode())


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# synthetic workload (S2/S3/S4 of SURVEY 8d): `nbatch` frames = streams of consecutive frames, identical bytes for CPU and GPU
# ----------------------------------------------------------------------------------------------------------------------
def make_frames(nbatch, seed, W, H, unique=32):
    from pysgs import synth
    unique = min(unique, nbatch)
    base, boxes = synth.stream_s2(unique, W, H, seed=seed, tex_w=int(1.6 * W), tex_h=int(1.6 * H))
    frames = np.zeros((nbatch, H, W), np.uint8)
    bx = np.zeros((nbatch, 4), np.float32)
    for i in range(nbatch):
        rep, k = divmod(i, unique)
        if rep == 0:
            frames[i] = base[k]; bx[i] = boxes[k]
        else:   # further streams: the same camera path seen through a cyclic shift (distinct pixels, same statistics)
            dx, dy = 7 * rep, 5 * rep
            frames[i] = np.roll(np.roll(base[k], dy, 0), dx, 1)
            bx[i] = boxes[k]; bx[i, 0] = (boxes[k, 0] + dx) % W; bx[i, 1] = (boxes[k, 1] + dy) % H
    return frames, bx, unique


def prev_index(nbatch, unique):
    """Index (inside the batch) of the previous frame of the same stream; the first frame of a stream is its own predecessor."""
    f = np.arange(nbatch, dtype=np.int32)
    return np.where(f % unique != 0, f - 1, f).astype(np.int32)


def camera_dict(scale):
    from pysgs import synth
    c = dict(synth.TUM3)
    for k in ('fx', 'fy', 'cx', 'cy'):
        c[k] = c[k] * scale
    return c


def make_track_inputs(kps, desc, counts, boxes, cap, point_cap, pidx, W, H, cam):
    """Per-frame inputs of the dyn-reject + match stage (host side, untimed): ground-truth person boxes (used by the tracker-only legs; the full
    step takes the detector's), u_right from a synthetic depth plane, and the last-frame map points = keypoints of the previous frame
    back-projected with that depth (Tracking::UpdateLastFrame state)."""
    from pysgs import synth
    B = len(counts)
    depth = synth.depth_s1(W, H)
    ur = np.full((B, cap), -1, np.float32)
    nb = np.ones(B, np.int32); have = np.ones(B, np.uint8)
    bx = np.zeros((B, 4, 4), np.float32); bx[:, 0] = boxes
    lxyz = np.zeros((B, point_cap, 3), np.float32); ldesc = np.zeros((B, point_cap, 32), np.uint8)
    lflags = np.zeros((B, point_cap), np.uint8); loct = np.zeros((B, point_cap), np.int32); lang = np.zeros((B, point_cap), np.float32)
    ln = np.zeros(B, np.int32)
    T = np.tile(np.eye(4, dtype=np.float32).reshape(1, 16), (B, 1))
    for f in range(B):
        n = counts[f]
        k = kps[f, :n]
        z = depth[np.clip(k['y'].astype(np.int64), 0, H - 1), np.clip(k['x'].astype(np.int64), 0, W - 1)]
        ur[f, :n] = k['x'] - np.float32(cam['bf']) / z
        g = pidx[f]
        m = min(counts[g], point_cap)
        kk = kps[g, :m]
        zz = depth[np.clip(kk['y'].astype(np.int64), 0, H - 1), np.clip(kk['x'].astype(np.int64), 0, W - 1)]
        lxyz[f, :m] = np.stack([(kk['x'] - cam['cx']) * zz / cam['fx'], (kk['y'] - cam['cy']) * zz / cam['fy'], zz], 1)
        ldesc[f, :m] = desc[g, :m]; loct[f, :m] = kk['octave']; lang[f, :m] = kk['angle']
        lflags[f, :m] = 1 | (2 * ((np.arange(m) % 5) != 0))                              # every 5th point is a temporal point (0 observations)
        ln[f] = m
    return dict(ur=ur, boxes=bx, nb=nb, have=have, lxyz=lxyz, ldesc=ldesc, lflags=lflags, loct=loct, lang=lang, ln=ln, T=T, sf=synth.scale_factors(),
                pidx=np.ascontiguousarray(pidx, np.int32))


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clock / throttle-reason sampler for the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def run(self):
        q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + q, '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(',')])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 7 and r[0].replace('.', '').isdigit()]
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        sm = sorted(float(r[0]) for r in rows)
        load = [v for v in sm if v >= 0.6 * sm[-1]] or sm      # "under load": idle gaps do not drag the median down
        reasons = []
        for i, name in ((3, 'hw_slowdown'), (4, 'hw_thermal_slowdown'), (5, 'sw_thermal_slowdown'), (6, 'sw_power_cap')):
            if any(r[i].lower().startswith('active') for r in rows):
                reasons.append(name)
        return {'sm_mhz': load[len(load) // 2], 'sm_max_mhz': float(rows[0][1]), 'reasons': reasons, 'samples': len(rows),
                'power_w_max': max(float(r[2]) for r in rows if r[2].replace('.', '').isdigit())}


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))), 'measured'
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback'


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's per-frame chain inside the C++ oracle (oracle/chain.cpp), worker threads pinned one per core
# ----------------------------------------------------------------------------------------------------------------------
def cpu_chain_rates(frames, pidx, ti, cam, cap, nfeat, nframes, want_outputs=False):
    """(all-cores frames/s, single-thread frames/s, cores, Chain).  Single thread = the reference's actual execution model (one tracking thread)."""
    import oracle as O
    cores = O.online_cpus()
    ch = O.Chain(frames, pidx, ti, cam, cap, nfeatures=nfeat, th=TH, want_outputs=want_outputs)
    ch.run(0, min(nframes, cores), nthreads=cores)                           # warm-up: page in, spin the threads once
    t0 = time.perf_counter(); ch.run(0, nframes, nthreads=cores); dt_all = time.perf_counter() - t0
    n1 = min(4, nframes)
    t0 = time.perf_counter(); ch.run(0, n1, nthreads=1); dt_one = time.perf_counter() - t0
    return nframes / dt_all, n1 / dt_one, cores, ch


def cpu_detector(threads):
    """Detector2D::detect on the CPU for the baseline legs: the FP32 restatement evaluated on chunks of 16 frames with PyTorch-CPU tensors in channels-last
    layout on all host threads (oracle/detector_batched.py; same graph walk as the parity checker oracle/detector_oracle.py, which interprets one frame layer
    by layer through numpy and is ~7x slower) -- NOT ncnn, which is not installable here.  Returns run(frames) -> list of detections."""
    import detector_batched as DB
    import ncnn_model as NM
    import torch
    torch.set_num_threads(threads)                        # the CPUs this process may really use (affinity mask capped by the cgroup quota)
    layers = NM.parse_param(MODEL + '.param'); NM.load_weights(layers, MODEL + '.bin')
    bd = DB.BatchedDetector(layers)
    return lambda frames: bd.detect(frames)


def detector_cpu_rate(rgb_frames):
    """frames/s of cpu_detector over the sample (after a warm-up on its first chunk)."""
    import oracle as O
    run = cpu_detector(O.online_cpus())
    run(rgb_frames[:16])
    t0 = time.perf_counter()
    run(rgb_frames)
    return len(rgb_frames) / (time.perf_counter() - t0)


def combine_rates(chain_fps, det_fps):
    """Both run on the same cores (the reference's detector is one more CPU thread): CPU time per frame adds up."""
    return 1.0 / (1.0 / chain_fps + (1.0 / det_fps if det_fps else 0.0))


def run_reference(args, cfg):
    """--impl reference: the reference's own CPU path on this box's host cores.  The reference cannot be compiled here (needs OpenCV/Eigen/ncnn/ROS,
    DESIGN.md), so this times the CPU oracle port: the C++ per-frame chain on one pinned worker thread per core over the SAME number of frames
    per step as the GPU arm, plus the detector restatement on a bounded sample of those frames (scaled to the step)."""
    if int(os.environ.get('RANK', '0')) != 0:
        return
    import oracle as O
    from pysgs import synth
    if args.config == 'hamming':
        return run_reference_hamming(args)
    W, H, NF = cfg['W'], cfg['H'], cfg['NFEAT']
    NB = args.batch or cfg['batch']
    cam = camera_dict(cfg['cam_scale'])
    frames, boxes, unique = make_frames(NB, 2, W, H)
    pidx = prev_index(NB, unique)
    cap = NF + 64
    O.lib()
    # inputs of the match stage need the keypoints once (untimed): extraction of the unique frames on all cores
    ti0 = make_track_inputs(np.zeros((NB, cap), O.KP_DTYPE), np.zeros((NB, cap, 32), np.uint8), np.zeros(NB, np.int32), boxes, cap, cap, pidx, W, H, cam)
    ch0 = O.Chain(frames, pidx, ti0, cam, cap, nfeatures=NF, th=TH, want_outputs=True)
    cores = O.online_cpus()
    ch0.run(0, NB, nthreads=cores)
    ti = make_track_inputs(ch0.out['kps'], ch0.out['desc'], ch0.out['counts'], boxes, cap, cap, pidx, W, H, cam)
    ch = O.Chain(frames, pidx, ti, cam, cap, nfeatures=NF, th=TH, want_outputs=False)
    # Every timed step really runs both parts on the same bounded sample of S frames of the batch (no extrapolation: steps x ms_per_step is the wall time
    # of the timed region): the tracking chain on all cores, then the detector restatement in chunks of 16 frames on all cores.  S is sized from a probe so that a
    # step takes about two seconds.
    with_det = os.path.exists(MODEL + '.param') and not args.no_detector
    det_run = None
    if with_det:
        det_fn = cpu_detector(cores)
        rgb = synth.gray_to_rgb(frames[:min(NB, 256)])

        def det_run(n):
            det_fn([rgb[f % len(rgb)] for f in range(n)])
        det_run(16)
    ch.run(0, min(NB, cores), nthreads=cores)
    t0 = time.perf_counter(); ch.run(0, min(NB, 2 * cores), nthreads=cores); probe_chain = (time.perf_counter() - t0) / min(NB, 2 * cores)
    probe_det = 0.0
    if with_det:
        t0 = time.perf_counter(); det_run(16); probe_det = (time.perf_counter() - t0) / 16
    S = int(max(8, min(NB, round(2.0 / max(1e-6, probe_chain + probe_det)))))
    if S >= cores:
        S = max(cores, int(round(S / cores)) * cores)  # whole rounds of the worker threads
    t_chain = t_det = 0.0

    def ref_step(timed):
        nonlocal t_chain, t_det
        a = time.perf_counter(); ch.run(0, S, nthreads=cores); b = time.perf_counter()
        if with_det:
            det_run(S)
        c = time.perf_counter()
        if timed:
            t_chain += b - a; t_det += c - b
    for _ in range(args.warmup):
        ref_step(False)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref_step(True)
    dt_step = (time.perf_counter() - t0) / args.steps
    t0 = time.perf_counter(); ch.run(0, 4, nthreads=1); one_fps = 4 / (time.perf_counter() - t0)
    fps = S / dt_step
    line = {'impl': 'reference', 'metric': 'frames/sec ORB extract+match+dyn-reject %dx%d' % (W, H), 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt_step, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
            'config': {'workload': workload_name(cfg, with_det), 'frames_per_gpu_per_step': NB, 'sample_frames_per_step': S,
                       'note': 'CPU oracle port of the reference path (the reference itself needs OpenCV/ROS/ncnn: unbuildable here).  Every step runs %d frames of the %d-frame batch through the tracking chain (C++ worker threads pinned one per core) and through the detector (PyTorch-CPU FP32 restatement, chunks of 16 frames in channels-last layout on all threads); both inside the timed region' % (S, NB)},
            'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port', 'sample': '%d frames per step x %d steps, chain + detector both run on every frame of the sample' % (S, args.steps),
                             'tracking_chain_all_cores': S * args.steps / t_chain if t_chain > 0 else None, 'tracking_chain_single_thread': one_fps,
                             'tracking_chain_per_core': (S * args.steps / t_chain / cores) if t_chain > 0 else None,
                             'detector_all_cores': (S * args.steps / t_det) if t_det > 0 else None},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    emit(line)


def workload_name(cfg, with_detector):
    return '%s, ORB %d features / 8 levels / 1.2: %sextract + LK(21x21, 4 levels) + findFundamentalMat(FM_RANSAC 1.0/0.99) + dyn-reject(boxes + epipolar) + SearchByProjection(th=15)' % (
        cfg['name'], cfg['NFEAT'], 'Detector2D::detect (MobileNetV3-SSDLite 300x300) + ' if with_detector else '')


# ----------------------------------------------------------------------------------------------------------------------
# config hamming (BASELINE configs[4]): brute-force 256-bit Hamming matching, N = M in {1k .. 64k}, queries sharded over the ranks
# ----------------------------------------------------------------------------------------------------------------------
HAMMING_SIZES = [1024, 2048, 4096, 8192, 16384, 32768, 65536]


def run_reference_hamming(args):
    import oracle as O
    from pysgs import synth
    cores = O.online_cpus()
    n = 8192
    t = synth.descriptors_s5(n, 5); q = synth.descriptors_near(t[:2048], 6)
    from concurrent.futures import ThreadPoolExecutor
    chunks = np.array_split(np.arange(len(q)), cores)
    O.bf_match(q[:64], t)

    def one():
        with ThreadPoolExecutor(cores) as ex:
            list(ex.map(lambda idx: O.bf_match(q[idx], t) if len(idx) else None, chunks))      # ctypes releases the GIL inside the C++ loops
    for _ in range(args.warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one()
    dt = (time.perf_counter() - t0) / args.steps
    pairs = len(q) * n / dt
    emit({'impl': 'reference', 'metric': 'descriptor pairs/sec brute-force Hamming 256-bit', 'value': pairs, 'unit': 'pairs/s', 'n_gpus': args.gpus, 'steps': args.steps,
          'warmup': args.warmup, 'ms_per_step': 1e3 * dt, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
          'config': {'workload': 'S5 brute-force Hamming (BASELINE configs[4]); CPU sample: %d queries x %d train descriptors per step' % (len(q), n)},
          'cpu_baseline': {'value': pairs, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port', 'sample': '%d x %d pairs per step' % (len(q), n)},
          'e2e': {'value': pairs, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}})


def run_hamming(args):
    import torch
    from pysgs import binding as B
    from pysgs import synth
    world = int(os.environ.get('WORLD_SIZE', '1')); rank = int(os.environ.get('RANK', '0')); local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    NMAX = HAMMING_SIZES[-1]
    train = torch.from_numpy(synth.descriptors_s5(NMAX, 5) if rank == 0 else np.zeros((NMAX, 32), np.uint8)).cuda()
    if dist is not None:
        dist.broadcast(train, 0)                 # the database descriptors reach every rank through one ncclBroadcast
    torch.cuda.synchronize()
    rs = np.random.RandomState(6)
    train_h = train.cpu().numpy()
    flips = np.unpackbits(train_h, axis=1) ^ (rs.uniform(size=(NMAX, 256)) < 0.06)
    query = torch.from_numpy(np.packbits(flips, axis=1)).cuda()
    st = torch.cuda.Stream()
    warm = max(args.warmup, 3)
    rows = []
    sampler = ClockSampler(local); sampler.start(); time.sleep(0.2)
    flush = torch.empty(160 * 1024 * 1024, dtype=torch.uint8, device='cuda')           # > 126 MB L2: written between timed iterations
    for n in HAMMING_SIZES:
        nq = n // world                                                               # this rank's share of the queries; the train set is replicated
        q = query[rank * nq:(rank + 1) * nq]
        idx = torch.zeros(nq, dtype=torch.int32, device='cuda'); best = torch.zeros_like(idx); second = torch.zeros_like(idx)
        scratch = torch.zeros(max(1, B.hamming_bf_scratch_elems(nq, n)), dtype=torch.int64, device='cuda')
        run = lambda: B.hamming_bf_device(q.data_ptr(), nq, train.data_ptr(), n, idx.data_ptr(), best.data_ptr(), second.data_ptr(), scratch.data_ptr(), st.cuda_stream)
        with torch.cuda.stream(st):
            for _ in range(warm):
                run()
            tot = 0.0
            for _ in range(args.steps):
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
                e0.record(st); run(); e1.record(st); e1.synchronize()
                tot += e0.elapsed_time(e1)
        ms = tot / args.steps
        if dist is not None:
            t_ = torch.tensor([ms], dtype=torch.float64, device='cuda'); dist.all_reduce(t_, op=dist.ReduceOp.MAX); ms = float(t_.item())
        ok = bool((idx.cpu().numpy() == np.arange(rank * nq, (rank + 1) * nq)).mean() > 0.999)          # planted neighbours are found
        rows.append({'n': n, 'ms': ms, 'pairs_per_s': n * float(n) / (ms * 1e-3), 'planted_neighbours_found': ok})
    clocks = sampler.stop()
    if rank == 0:
        peaks, kind = measured_peaks()
        top = rows[-1]
        sm_hz = (clocks.get('sm_mhz') or 1965.0) * 1e6
        popc_pairs = 148 * 16 * sm_hz / 8                          # 16 POPC / clk / SM, 8 32-bit words per pair
        for r in rows:
            r['frac_of_popc_rate'] = r['pairs_per_s'] / popc_pairs
            r['alg_gbs'] = (32 * 2 * r['n'] + 12 * r['n']) / (r['ms'] * 1e-3) / 1e9
        emit({'metric': 'descriptor pairs/sec brute-force Hamming 256-bit', 'value': top['pairs_per_s'], 'unit': 'pairs/s', 'n_gpus': world, 'steps': args.steps, 'warmup': warm,
              'ms_per_step': top['ms'], 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'u8', 'data': 'synthetic',
              'config': {'workload': 'S5 brute-force Hamming sweep N = M in {1k..64k} x 256 bit (BASELINE configs[4]); value = the 64k x 64k point', 'sweep': rows,
                         'sharding': 'queries split over the ranks, train descriptors replicated by one ncclBroadcast', 'l2_policy': 'a 160 MB buffer is written between timed iterations'},
              'clocks': clocks, 'gpu_launches': 2 * args.steps * len(HAMMING_SIZES),
              'roofline': {'bound': 'hbm', 'kernel': 'hamming_bf_kernel', 'achieved': top['alg_gbs'], 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': top['alg_gbs'] / peaks['hbm_gbs'],
                           'traffic': None, 'peak_kind': kind, 'binding_roof': 'POPC issue rate: %.2f of 148 SM x 16 POPC/clk' % top['frac_of_popc_rate'],
                           'note': 'all-pairs matching re-uses every descriptor N times from shared memory: the HBM fraction is reported as asked, the binding roof is the integer pipe'},
              'e2e': None, 'cpu_baseline': None})
    if dist is not None:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='s2', choices=['s2', '720p', 'hamming'])
    ap.add_argument('--batch', type=int, default=0, help='frames per GPU per step (default 512 at 640x480: 157 MB of gray input > the 126 MB L2)')
    ap.add_argument('--cpu-sample', type=int, default=0, help='frames of the cpu_baseline sample (0: four per host thread, at least 64)')
    ap.add_argument('--parity-frames', type=int, default=256, help='frames of the full-chain parity check against the pure oracle')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-pipeline', action='store_true', help='e2e: skip the steps-in-flight mode')
    ap.add_argument('--pipeline-handles', type=int, default=3, help='e2e: full-size handles taking whole steps in turn')
    ap.add_argument('--no-detector', action='store_true', help='tracker-only step with ground-truth boxes (the round-1 definition of the step)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed to DIR/<name>.npy (see dump_step_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.config == 'hamming'):
        ap.error('--dump-outputs writes the outputs of the GPU step: --impl ours with --config s2 or 720p')
    claim_stdout()
    cfg = CONFIGS.get(args.config)
    if args.impl == 'reference':
        return run_reference(args, cfg)
    if args.config == 'hamming':
        return run_hamming(args)

    import torch
    from pysgs import binding as B
    from pysgs import synth

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: there is no CPU fallback for the product path')
    torch.cuda.set_device(local)
    pin_rank_to_numa_node(local)
    dist = None
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')   # keep stdout to the single JSON line (NCCL prints its version banner to stdout)
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    W, H, NFEAT = cfg['W'], cfg['H'], cfg['NFEAT']
    NB = args.batch or cfg['batch']
    warm = max(args.warmup, 3)
    L = B.lib()
    v = C.c_void_p
    camd = camera_dict(cfg['cam_scale'])
    use_det = (not args.no_detector) and os.path.exists(MODEL + '.param')
    if not use_det and not args.no_detector:
        log('[bench] WARNING: %s.param not staged (build() copies it from the reference tree): the detector is left out of the step' % MODEL)

    # ---- workload + one-time set-up (untimed) -------------------------------------------------------------------------
    t_setup = time.time()
    frames, gt_boxes, unique = make_frames(NB, 2 + rank, W, H)
    pidx = prev_index(NB, unique)
    sf = synth.scale_factors()
    cam = B.make_camera(W, H, camd, sf)
    trk = B.Tracker(W, H, cam, NFEAT, 1.2, 8, 20, 7, max_batch=NB, point_cap=NFEAT + 64, max_boxes=4, device=local)
    cap, pcap = trk.cap, trk.point_cap
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
    h_frames = pin((NB, H, W), torch.uint8); h_frames.numpy()[:] = frames
    h_kps = pin((NB, cap, 28), torch.uint8); h_desc = pin((NB, cap, 32), torch.uint8); h_n = pin((NB,), torch.int32)
    d_frames = h_frames.cuda()
    d_pidx = torch.from_numpy(pidx).cuda()
    st = torch.cuda.Stream(); st_det = torch.cuda.Stream()
    det = None
    h_rgb = d_rgb = None
    if use_det:
        det = B.Detector(MODEL + '.param', MODEL + '.bin', max_frames=NB, det_thr=0.9, dyn_thr=0.01, device=local)
        h_rgb = pin((NB, H, W, 3), torch.uint8); h_rgb.numpy()[:] = synth.gray_to_rgb(frames)
        d_rgb = h_rgb.cuda()
    L.sgs_tracker_extractor.restype = C.c_void_p
    exh = v(L.sgs_tracker_extractor(trk.h))
    torch.cuda.synchronize()
    # set-up pass on the device: extract; the keypoints feed the host-side construction of u_right / last-frame points
    B.check(L.sgs_tracker_extract_device(trk.h, v(d_frames.data_ptr()), NB, C.c_size_t(W * H), W, v(st.cuda_stream)))
    B.check(L.sgs_extractor_fetch(exh, NB, v(h_kps.data_ptr()), v(h_desc.data_ptr()), cap, v(h_n.data_ptr()), v(st.cuda_stream)))
    kps0 = h_kps.numpy().reshape(NB, cap * 28).view(B.KP_DTYPE).reshape(NB, cap).copy(); desc0 = h_desc.numpy().copy(); n0 = h_n.numpy().copy()
    ti = make_track_inputs(kps0, desc0, n0, gt_boxes, cap, pcap, pidx, W, H, camd)
    keys_h = ['ur', 'boxes', 'nb', 'have', 'lxyz', 'ldesc', 'lflags', 'loct', 'lang', 'ln', 'T', 'pidx']
    hp = {k: torch.from_numpy(np.ascontiguousarray(ti[k])).pin_memory() for k in keys_h}
    dv = {k: t.cuda(non_blocking=True) for k, t in hp.items()}
    d_depth = torch.from_numpy(synth.depth_s1(W, H).astype(np.float32)).cuda()      # one synthetic depth plane shared by every frame
    bcast = vocabulary_broadcast(dist, rank, local, L, B, synth)
    h_out = dict(kps=pin((NB, cap, 28), torch.uint8), desc=pin((NB, cap, 32), torch.uint8), ur=pin((NB, cap), torch.float32), cnt=pin((NB,), torch.int32),
                 mp=pin((NB, cap), torch.int32), nm=pin((NB,), torch.int32), boxes=pin((NB, 4, 4), torch.float32), nb=pin((NB,), torch.int32), have=pin((NB,), torch.uint8))
    torch.cuda.synchronize()
    log('[bench] rank %d set-up %.1fs: %d frames/step %dx%d, mean %.0f keypoints/frame, detector %s' % (rank, time.time() - t_setup, NB, W, H, n0.mean(), 'in the step' if use_det else 'OFF'))

    S = st.cuda_stream

    def dev_extract():
        B.check(L.sgs_tracker_extract_device(trk.h, v(d_frames.data_ptr()), NB, C.c_size_t(W * H), W, v(S)))

    def dev_lk():
        B.check(L.sgs_tracker_lk_device(trk.h, v(d_frames.data_ptr()), NB, C.c_size_t(W * H), W, v(d_pidx.data_ptr()), v(S)))

    def dev_stereo():   # Frame::ComputeStereoFromRGBD on the device (u_right of the unfiltered keypoints)
        B.check(L.sgs_tracker_stereo_device(trk.h, NB, v(d_depth.data_ptr()), C.c_size_t(0), W, v(S)))

    def dev_fm(own_boxes):
        if own_boxes:   # boxes == NULL: the tracker's own arrays, written by the detector
            B.check(L.sgs_tracker_fundamental_device(trk.h, NB, v(0), v(0), v(0), v(d_pidx.data_ptr()), v(S)))
        else:
            B.check(L.sgs_tracker_fundamental_device(trk.h, NB, v(dv['boxes'].data_ptr()), v(dv['nb'].data_ptr()), v(dv['have'].data_ptr()), v(d_pidx.data_ptr()), v(S)))

    def dev_track(own_boxes):
        bx = [0, 0, 0] if own_boxes else [dv[k].data_ptr() for k in ('boxes', 'nb', 'have')]
        ptrs = [0, 0, 0] + bx + [dv[k].data_ptr() for k in ('lxyz', 'ldesc', 'lflags', 'loct', 'lang', 'ln', 'T', 'T')]      # prev_xy, u_right, F == NULL: the tracker's own
        B.check(L.sgs_tracker_track_device(trk.h, NB, *[v(p) for p in ptrs], C.c_float(TH), 0, 1, v(S)))

    def dev_detect():
        B.check(L.sgs_tracker_detect_device(trk.h, det.h, v(d_rgb.data_ptr()), C.c_int64(W * H * 3), W * 3, W, H, NB, v(st_det.cuda_stream)))

    def dev_step(with_det):
        if with_det:
            e_start = torch.cuda.Event(); e_start.record(st); st_det.wait_event(e_start)       # the detector's work belongs to this step's timed window
            dev_detect()
            e_det = torch.cuda.Event(); e_det.record(st_det)
        dev_extract(); dev_lk()
        if with_det:
            st.wait_event(e_det)                                                                # src/Frame.cc:478-481: join before the boxes are used
        dev_fm(with_det); dev_stereo(); dev_track(with_det)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_steps(with_det, nsteps):
        with torch.cuda.stream(st):
            for _ in range(warm):
                dev_step(with_det)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st):
            e0.record(st)
            for _ in range(nsteps):
                dev_step(with_det)
            e1.record(st)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---- device-resident leg (value): the whole step, detector included ---------------------------------------------------
    sampler = ClockSampler(local); sampler.start(); time.sleep(0.3)
    total_ms = timed_steps(use_det, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_step_outputs(args.dump_outputs, L, B, trk, NB, cap, use_det)
    value = world * NB * args.steps / (total_ms * 1e-3)
    # ---- the tracker-only step (ground-truth boxes as inputs: the round-1 definition), with per-stage device times -------
    B.check(L.sgs_extractor_set_profiling(exh, 1))
    L.sgs_tracker_lk.restype = C.c_void_p
    lkh = v(L.sgs_tracker_lk(trk.h))
    B.check(L.sgs_lk_set_profiling(lkh, 1))
    nprof = max(3, min(args.steps, 10))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4 * nprof + 1)]
    barrier()
    with torch.cuda.stream(st):
        ev[0].record(st)
        for i in range(nprof):
            dev_extract(); ev[4 * i + 1].record(st)
            dev_lk(); ev[4 * i + 2].record(st)
            dev_fm(False); ev[4 * i + 3].record(st)
            dev_stereo(); dev_track(False); ev[4 * i + 4].record(st)
    barrier()
    trk_ms = max_over_ranks(ev[0].elapsed_time(ev[4 * nprof])) / nprof
    extract_ms = sum(ev[4 * i].elapsed_time(ev[4 * i + 1]) for i in range(nprof)) / nprof
    lk_ms = sum(ev[4 * i + 1].elapsed_time(ev[4 * i + 2]) for i in range(nprof)) / nprof
    fm_ms = sum(ev[4 * i + 2].elapsed_time(ev[4 * i + 3]) for i in range(nprof)) / nprof
    track_ms = sum(ev[4 * i + 3].elapsed_time(ev[4 * i + 4]) for i in range(nprof)) / nprof
    ms5 = (C.c_double * 5)(); ncalls = C.c_int()
    B.check(L.sgs_extractor_stage_times(exh, ms5, C.byref(ncalls)))
    stage_ms = [ms5[i] / max(1, ncalls.value) for i in range(5)]
    B.check(L.sgs_extractor_set_profiling(exh, 0))
    ms2 = (C.c_double * 2)()
    B.check(L.sgs_lk_stage_times(lkh, ms2, C.byref(ncalls)))
    lk_pyr_ms, lk_track_ms = ms2[0] / max(1, ncalls.value), ms2[1] / max(1, ncalls.value)
    B.check(L.sgs_lk_set_profiling(lkh, 0))
    det_ms = None; det_fam = None; det_kinds = None
    if use_det:
        det.set_profiling(1)                                  # CUDA events around every kernel of the call, on the launching stream
        with torch.cuda.stream(st_det):
            dev_detect()
            ed0, ed1 = torch.cuda.Event(True), torch.cuda.Event(True)
            ed0.record(st_det)
            for _ in range(3):
                dev_detect()
            ed1.record(st_det)
        torch.cuda.synchronize()
        det_ms = ed0.elapsed_time(ed1) / 3
        kms, kcalls = det.kernel_times()
        det.set_profiling(0)
        det_fam, det_kinds = detector_gemm_table(det, kms, kcalls, NB)

    # ---- the rest of the tracking thread's chain (TrackWithMotionModel after the search + TrackLocalMap), timed beside the step ---------------------
    chain_info = None
    try:
        rngc = np.random.default_rng(17)
        mcap = (pcap // 2 + cap // 3 + 127) // 64 * 64
        with torch.cuda.stream(st):
            dev_step(use_det)
        torch.cuda.synchronize()
        pk, pd, pu, pc_, pm, pn, pnc = (C.c_void_p() for _ in range(7))
        B.check(L.sgs_tracker_results_device(trk.h, C.byref(pk), C.byref(pd), C.byref(pu), C.byref(pc_), C.byref(pm), C.byref(pn), C.byref(pnc)))
        nsamp = min(NB, 16)                                   # local maps are built on the host from a few frames and tiled over the batch
        ck = B.memcpy_d2h(np.zeros((NB, cap), B.KP_DTYPE), pk.value); cd = B.memcpy_d2h(np.zeros((NB, cap, 32), np.uint8), pd.value)
        cc = B.memcpy_d2h(np.zeros(NB, np.int32), pc_.value)
        lms = [make_local_map(f, ck[f], cd[f], int(cc[f]), ti, mcap, camd, sf, rngc, W, H) for f in range(nsamp)]
        tile = lambda k, dt: torch.from_numpy(np.ascontiguousarray(np.stack([lms[f % nsamp][k] for f in range(NB)]).astype(dt))).cuda()
        cm = dict(lid=tile('lid', np.int32), xyz=tile('xyz', np.float32), nrm=tile('nrm', np.float32), mn=tile('mn', np.float32), mx=tile('mx', np.float32),
                  dsc=tile('dsc', np.uint8), valid=tile('valid', np.uint8), obs=tile('obs', np.uint8),
                  n=torch.from_numpy(np.array([lms[f % nsamp]['n'] for f in range(NB)], np.int32)).cuda())
        co = dict(T1=torch.zeros((NB, 16), device='cuda'), T2=torch.zeros((NB, 16), device='cuda'), mp=torch.zeros((NB, cap), dtype=torch.int32, device='cuda'),
                  outl=torch.zeros((NB, cap), dtype=torch.uint8, device='cuda'), st=torch.zeros((NB, 8), dtype=torch.int32, device='cuda'))
        pa = B.PoseChainBatch()
        pa.last_xyz, pa.last_desc, pa.last_flags, pa.last_octave, pa.last_angle, pa.last_n = [dv[k].data_ptr() for k in ('lxyz', 'ldesc', 'lflags', 'loct', 'lang', 'ln')]
        pa.tcw_cur = pa.tcw_last = dv['T'].data_ptr(); pa.th, pa.mono, pa.check_orientation, pa.last_local_id = TH, 0, 1, cm['lid'].data_ptr()
        pa.mp_xyz, pa.mp_normal, pa.mp_min_dist, pa.mp_max_dist, pa.mp_desc, pa.mp_valid, pa.mp_obs, pa.mp_n, pa.mp_cap = [cm[k].data_ptr() for k in ('xyz', 'nrm', 'mn', 'mx', 'dsc', 'valid', 'obs', 'n')] + [mcap]
        pa.th_local, pa.nnratio_local = 3.0, 0.8
        for l in range(16): pa.inv_level_sigma2[l] = float(1.0 / (sf[l] * sf[l])) if l < len(sf) else 0.0
        pa.tcw_motion, pa.tcw_final, pa.f_mp, pa.outlier, pa.stats = co['T1'].data_ptr(), co['T2'].data_ptr(), co['mp'].data_ptr(), co['outl'].data_ptr(), co['st'].data_ptr()

        def dev_chain():
            B.check(L.sgs_tracker_pose_chain_device(trk.h, C.byref(pa), NB, v(S)))
        with torch.cuda.stream(st):
            dev_track(use_det); dev_chain()                     # warm-up (allocates the chain's scratch)
            ec = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
            for i in range(3):
                dev_track(use_det); ec[2 * i].record(st); dev_chain(); ec[2 * i + 1].record(st)
        torch.cuda.synchronize()
        chain_ms = sum(ec[2 * i].elapsed_time(ec[2 * i + 1]) for i in range(3)) / 3
        stc = co['st'].cpu().numpy()
        chain_info = {'call': 'sgs_tracker_pose_chain_device (2 th retry, PoseOptimization, outlier discard, SearchLocalPoints: frustum + scale + projection search, PoseOptimization, inlier count)',
                      'ms_per_step': chain_ms, 'frames_per_s': NB / chain_ms * 1e3, 'local_map_points_per_frame': float(np.mean([m['n'] for m in lms])),
                      'mean_matches_last_frame': float(stc[:, 2].mean()), 'mean_in_frustum': float(stc[:, 5].mean()), 'mean_matches_added': float(stc[:, 6].mean()),
                      'mean_inliers': float(stc[:, 7].mean()), 'not_in_value': 'timed beside the step: BASELINE metric = extract + match + dyn-reject'}
    except Exception as ex_:
        log('[bench] pose chain stage skipped: %r' % (ex_,))

    # ---- e2e leg: host buffers through the C ABI (sgs_tracker_step / sgs_tracker_extract + _track_lk), copies inside the timed region ----
    def host_ptrs(hpi, out, sl=slice(None)):
        ins = [hpi[k].data_ptr() for k in ('pidx', 'ur', 'lxyz', 'ldesc', 'lflags', 'loct', 'lang', 'ln', 'T', 'T')]
        outs = [out[k][sl].data_ptr() for k in ('kps', 'desc', 'ur', 'cnt', 'mp', 'nm', 'boxes', 'nb', 'have')]
        return ins, outs

    def step_host(tk, dt_, nb, fr, rgb, hpi, sl=slice(None), out=None):
        ins, outs = host_ptrs(hpi, h_out if out is None else out, sl)
        if dt_ is not None:
            B.check(L.sgs_tracker_step(tk.h, dt_.h, v(fr.data_ptr()), C.c_size_t(W * H), W, v(rgb.data_ptr()), C.c_size_t(W * H * 3), W * 3, nb, *[v(p) for p in ins],
                                       C.c_float(TH), 0, 1, *[v(p) for p in outs]))
        else:       # tracker only: two calls, ground-truth boxes as inputs
            tk.extract(fr.data_ptr(), nb, W * H, W, h_kps[sl].data_ptr(), 0, h_n[sl].data_ptr())
            B.check(L.sgs_tracker_track_lk(tk.h, nb, v(ins[0]), v(ins[1]), v(0), v(hpi['boxes'].data_ptr()), v(hpi['nb'].data_ptr()), v(hpi['have'].data_ptr()),
                                           *[v(p) for p in ins[2:]], C.c_float(TH), 0, 1, *[v(p) for p in outs[:6]]))

    e2e = None
    step_host(trk, det, NB, h_frames, h_rgb, hp)          # warm-up; its outputs feed the parity checks below
    res_gpu = {k: t.numpy().copy() for k, t in h_out.items()}
    if not args.no_e2e:
        step_host(trk, det, NB, h_frames, h_rgb, hp)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_host(trk, det, NB, h_frames, h_rgb, hp)
        torch.cuda.synchronize()
        dt1 = max_over_ranks(time.perf_counter() - t0)
        track_in = ['pidx', 'ur', 'lxyz', 'ldesc', 'lflags', 'loct', 'lang', 'ln', 'T', 'T'] + ([] if use_det else ['boxes', 'nb', 'have'])      # tcw_cur and tcw_last are both copied
        h2d = h_frames.numel() + (h_rgb.numel() if use_det else 0) + sum(hp[k].numel() * hp[k].element_size() for k in track_in)
        outs = ['kps', 'desc', 'ur', 'cnt', 'mp', 'nm'] + (['boxes', 'nb', 'have'] if use_det else [])
        d2h = sum(h_out[k].numel() * h_out[k].element_size() for k in outs) + (0 if use_det else h_kps.numel() + h_n.numel() * 4)
        dt, mode = dt1, 'one tracker handle, synchronous calls'
        if NB % (2 * unique) == 0 and NB >= 128:        # the same work split over two handles driven by two host threads: copies of one half overlap kernels of the other
            HB = NB // 2
            halves = []
            for hx in range(2):
                tk = B.Tracker(W, H, cam, NFEAT, 1.2, 8, 20, 7, max_batch=HB, point_cap=NFEAT + 64, max_boxes=4, device=local)
                dk = B.Detector(MODEL + '.param', MODEL + '.bin', max_frames=HB, det_thr=0.9, dyn_thr=0.01, device=local) if use_det else None
                sl = slice(hx * HB, (hx + 1) * HB)
                hpi = {k: hp[k][sl] for k in keys_h}
                hpi['pidx'] = torch.from_numpy(np.ascontiguousarray(pidx[sl] - hx * HB)).pin_memory()
                halves.append((tk, dk, sl, hpi))

            def worker(hx, nsteps, gate):
                torch.cuda.set_device(local)
                tk, dk, sl, hpi = halves[hx]
                gate.wait()
                for _ in range(nsteps):
                    step_host(tk, dk, HB, h_frames[sl], h_rgb[sl] if use_det else None, hpi, sl)

            def run_pair(nsteps):
                gate = threading.Barrier(3)
                th = [threading.Thread(target=worker, args=(hx, nsteps, gate)) for hx in range(2)]
                for t in th:
                    t.start()
                barrier()
                gate.wait()
                t0 = time.perf_counter()
                for t in th:
                    t.join()
                torch.cuda.synchronize()
                return time.perf_counter() - t0
            run_pair(2)
            same = bool(np.array_equal(res_gpu['cnt'], h_out['cnt'].numpy()) and np.array_equal(res_gpu['nm'], h_out['nm'].numpy()))
            dt2 = max_over_ranks(run_pair(args.steps))
            if not same:
                log('[bench] WARNING: two-handle e2e results differ from the single-handle ones')
            elif dt2 < dt1:
                dt, mode = dt2, 'two tracker (+ detector) handles, %d frames each per call, driven by two host threads' % HB
            for tk, dk, _, _ in halves:
                tk.close()
                if dk is not None:
                    dk.close()
        if use_det and args.steps >= 2 and not args.no_pipeline:
            # whole steps alternating over two full-size handles (two steps in flight): the copies of one step overlap the kernels of the other at the full
            # batch size of every launch
            NH = max(2, args.pipeline_handles)
            extra = [(B.Tracker(W, H, cam, NFEAT, 1.2, 8, 20, 7, max_batch=NB, point_cap=NFEAT + 64, max_boxes=4, device=local),
                      B.Detector(MODEL + '.param', MODEL + '.bin', max_frames=NB, det_thr=0.9, dyn_thr=0.01, device=local),
                      {k: pin(tuple(t.shape), t.dtype) for k, t in h_out.items()}) for _ in range(NH - 1)]

            def worker3(hx, nsteps, gate):
                torch.cuda.set_device(local)
                gate.wait()
                for _ in range(nsteps):
                    if hx == 0:
                        step_host(trk, det, NB, h_frames, h_rgb, hp)
                    else:
                        step_host(extra[hx - 1][0], extra[hx - 1][1], NB, h_frames, h_rgb, hp, out=extra[hx - 1][2])

            def run_alt(nsteps):
                gate = threading.Barrier(NH + 1)
                th = [threading.Thread(target=worker3, args=(hx, (nsteps + NH - 1 - hx) // NH, gate)) for hx in range(NH)]
                for t in th:
                    t.start()
                barrier()
                gate.wait()
                t0 = time.perf_counter()
                for t in th:
                    t.join()
                torch.cuda.synchronize()
                return time.perf_counter() - t0
            run_alt(NH)
            same3 = all(bool(np.array_equal(res_gpu['cnt'], e[2]['cnt'].numpy()) and np.array_equal(res_gpu['nm'], e[2]['nm'].numpy()) and np.array_equal(res_gpu['mp'], e[2]['mp'].numpy()))
                        for e in extra)
            dt3 = max_over_ranks(run_alt(args.steps))
            if not same3:
                log('[bench] WARNING: pipelined e2e results differ from the single-handle ones')
            elif dt3 < dt:
                dt, mode = dt3, '%d full-size tracker + detector handles taking whole steps in turn (%d steps in flight), one host thread each' % (NH, NH)
            for e in extra:
                e[0].close(); e[1].close()
        e2e = {'value': world * NB * args.steps / dt, 'unit': 'frames/s', 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
               'ms_per_step': 1e3 * dt / args.steps, 'mode': mode, 'single_handle_value': world * NB * args.steps / dt1,
               'note': ('sgs_tracker_step: host gray + colour frames and track inputs in, compacted keypoints / descriptors / matches / detector boxes out' if use_det else
                        'sgs_tracker_extract + sgs_tracker_track_lk (tracker only, ground-truth boxes as inputs)') + ', pinned host buffers'}

    # ---- roofline of the dominant kernel (timed live with CUDA events on the launching stream) ---------------------------------
    peaks, peak_kind = measured_peaks()
    nk = int(n0.mean())
    ab = alg_bytes(W, H, nk)
    names = ['pyramid(7 launches)', 'fast_warp_cells_kernel', 'quadtree_kernel', 'blur_tile_kernel', 'describe_kernel']
    alg = {'pyramid(7 launches)': ab['pyramid'], 'fast_warp_cells_kernel': ab['fast'] + 40 * nk, 'quadtree_kernel': 84 * nk, 'blur_tile_kernel': ab['blur'],
           'describe_kernel': ab['describe'], 'lk_pyramid+deriv(11 launches)': ab['lk_pyr'], 'lk_track_kernel': ab['lk_track'], 'fm_ransac_kernel': ab['fm'],
           'stereo+dynreject+compact+match(4 launches)': ab['track']}
    all_ms = dict(zip(names, stage_ms))
    all_ms.update({'lk_pyramid+deriv(11 launches)': lk_pyr_ms, 'lk_track_kernel': lk_track_ms, 'fm_ransac_kernel': fm_ms, 'stereo+dynreject+compact+match(4 launches)': track_ms})
    dom = max(('fast_warp_cells_kernel', 'quadtree_kernel', 'describe_kernel', 'lk_track_kernel', 'fm_ransac_kernel'), key=lambda k: all_ms[k])   # single-launch kernels
    dom_bytes = alg[dom] * NB
    achieved = dom_bytes / (all_ms[dom] * 1e-3) / 1e9
    step_alg = (ab['extract'] + ab['lk_pyr'] + ab['lk_track'] + ab['fm'] + ab['track']) * NB
    peak_note = 'measured copy bandwidth (MEASURED_PEAKS.json)' if peak_kind == 'measured' else 'fallback 6650 GB/s'
    tracker_dom = {'kernel': dom, 'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': achieved / peaks['hbm_gbs'],
                   'algorithmic_bytes_per_launch': int(dom_bytes), 'kernel_ms': all_ms[dom],
                   'note': 'largest single launch of the step; instruction-issue bound (exact OpenCV fixed-point arithmetic), the HBM fraction is reported as asked'}
    common = {'stage_ms': {k: round(x, 4) for k, x in all_ms.items()}, 'extract_ms': extract_ms, 'lk_ms': lk_ms, 'fundamental_ms': fm_ms, 'dynreject_match_ms': track_ms,
              'tracker_step_ms': trk_ms, 'detector_ms': det_ms,
              'per_kernel_alg_gbs': {k: round(alg[k] * NB / (all_ms[k] * 1e-3) / 1e9, 1) for k in all_ms},
              'extract_alg_gbs': ab['extract'] * NB / (extract_ms * 1e-3) / 1e9, 'extract_frac_of_hbm': ab['extract'] * NB / (extract_ms * 1e-3) / 1e9 / peaks['hbm_gbs'],
              'tracker_step_frac_of_hbm': step_alg / (trk_ms * 1e-3) / 1e9 / peaks['hbm_gbs'],
              'traffic': None, 'traffic_note': 'not measured in this run: the ncu --set full captures (dram__bytes_read/write per launch) are under profiles/'}
    if use_det and det_fam and det_fam['ms'] > all_ms[dom]:
        # with the detector in the step the kernel that takes most of it is the 1x1-convolution GEMM (one template, 66 launches of different shapes per call):
        # its algorithmic bytes per call / the sum of its launch durations, both for the NB frames of one step
        g_gbs = det_fam['bytes'] / (det_fam['ms'] * 1e-3) / 1e9
        g_tf = det_fam['flop'] / (det_fam['ms'] * 1e-3) / 1e12
        roofline = dict({'bound': 'hbm', 'kernel': 'conv1x1_tc_kernel (the detector\'s 1x1-convolution GEMM: %d launches per call, TMA + tcgen05/TMEM)' % det_fam['launches'],
                         'achieved': g_gbs, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': g_gbs / peaks['hbm_gbs'], 'peak_kind': peak_note,
                         'algorithmic_bytes_per_launch': int(det_fam['bytes'] / det_fam['launches']), 'algorithmic_bytes_per_call': int(det_fam['bytes']),
                         'kernel_ms': det_fam['ms'], 'launches': det_fam['launches'],
                         'tensor': {'achieved_fp32_equivalent': g_tf, 'tensor_pipe_tf32': 3 * g_tf, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s', 'frac_of_dense_bf16_peak': 3 * g_tf / peaks['bf16_tflops'],
                                    'note': 'K = 16..960 with FP32 activations: these layers stream (about %.0f FLOP per byte), the tensor pipe is never the bound' % (det_fam['flop'] / det_fam['bytes'])},
                         'detector_kernels_ms': det_kinds, 'tracker_dominant': tracker_dom,
                         'note': 'measured live: CUDA events around every kernel of sgs_detector_detect_device on its launching stream (sgs_detector_set_profiling), bytes = FP32 NHWC activations in + out + fused-tail tensor operands + weights'},
                        **common)
    else:
        roofline = dict({'bound': 'hbm', 'kernel': dom, 'achieved': achieved, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': achieved / peaks['hbm_gbs'], 'peak_kind': peak_note,
                         'algorithmic_bytes_per_launch': int(dom_bytes), 'kernel_ms': all_ms[dom],
                         'note': 'the tracker kernels are instruction-issue / latency bound (integer fixed-point OpenCV semantics): the HBM fraction is reported as asked'}, **common)
    det_info = None
    if use_det:
        tf = NB * DET_GFLOP / det_ms
        det_info = {'model': 'mobilenetv3_ssdlite_voc (the reference\'s trained ncnn model, 9.7 MB FP32 weights)', 'frames_per_call': NB, 'ms_per_call': det_ms, 'frames_per_s': NB / det_ms * 1e3,
                    'kernels_per_call': det.num_kernels,
                    'roofline': {'bound': 'tensor', 'achieved': tf, 'peak': peaks['bf16_tflops'], 'unit': 'TFLOP/s', 'frac': tf / peaks['bf16_tflops'],
                                 'note': '1.115 GFLOP per 300x300 inference (SURVEY 8d) counted once; the 66 1x1 convolutions (90 % of the MACs) are TMA-fed tcgen05 / TMEM GEMMs with error-compensated TF32 operands (3 tcgen05.mma per k-step: the tensor pipe does 3x these FLOPs), the rest FP32 FMA; the layers are streaming-bound (K = 16..960), peak = measured dense bf16'}}

    # ---- parity: (1) the whole chain against the PURE oracle (own LK, own F; the detector's boxes as inputs) ---------------------------------
    parity = None
    cpu = None
    if rank == 0 and world == 1:
        import oracle as O
        npar = min(args.parity_frames, NB)
        tp = dict(ti)
        if use_det:
            tp['boxes'] = res_gpu['boxes']; tp['nb'] = res_gpu['nb']; tp['have'] = res_gpu['have']
        ns = min(args.cpu_sample if args.cpu_sample > 0 else max(64, 4 * O.online_cpus()), NB)
        nrun = max(npar, ns)
        fps_all, fps_one, cores, ch = cpu_chain_rates(frames, pidx, tp, camd, cap, NFEAT, nrun, want_outputs=True)
        o = ch.out
        kps_g = res_gpu['kps'].reshape(NB, cap * 28).view(B.KP_DTYPE).reshape(NB, cap)
        same_extract = all(int(n0[f]) == int(o['counts'][f]) and kps0[f, :n0[f]].tobytes() == o['kps'][f, :n0[f]].tobytes() and np.array_equal(desc0[f, :n0[f]], o['desc'][f, :n0[f]])
                           for f in range(npar))
        keep_diff = []; match_diff = []; exact_frames = 0
        for f in range(npar):
            n = int(o['counts'][f])
            ko = np.ones(n, bool) if o['restored'][f] else o['keep'][f, :n].astype(bool)
            # GPU keep set: the surviving keypoints in order are a subsequence of the extracted ones -> recover the mask by matching positions
            ng = int(res_gpu['cnt'][f])
            kg = np.zeros(n, bool)
            src = kps0[f, :n]; dst = kps_g[f, :ng]
            j = 0
            for i in range(n):
                if j < ng and src[i] == dst[j]:
                    kg[i] = True; j += 1
            keep_diff.append(int((kg != ko).sum()))
            # matches: last-frame point index per original keypoint (-1: none / rejected)
            mo = np.full(n, -1, np.int64); mo[np.nonzero(ko)[0]] = o['match'][f, :int(ko.sum())]
            mg = np.full(n, -1, np.int64); mg[np.nonzero(kg)[0]] = res_gpu['mp'][f, :ng]
            match_diff.append(int((mo != mg).sum()))
            exact_frames += int(keep_diff[-1] == 0 and match_diff[-1] == 0)
        parity = {'frames': npar, 'extraction_bit_exact': bool(same_extract),
                  'keep_set_symmetric_difference': {'mean': float(np.mean(keep_diff)), 'max': int(np.max(keep_diff)), 'frames_identical': int(np.sum(np.array(keep_diff) == 0))},
                  'match_index_difference': {'mean': float(np.mean(match_diff)), 'max': int(np.max(match_diff)), 'frames_identical': int(np.sum(np.array(match_diff) == 0))},
                  'frames_identical_end_to_end': exact_frames, 'mean_keypoints': float(np.mean(o['counts'][:npar])),
                  'note': 'GPU chain (through sgs_tracker_step) against the pure CPU oracle chain (its own LK and its own F): per frame, keypoints whose keep / remove verdict differs and keypoints whose matched map point differs.  Differences come from LK (the GPU sums the window exactly, OpenCV in float order; <= 0.03 px) moving an epipolar distance across its threshold'}
        det_cpu = None
        if use_det:
            try:
                det_cpu = detector_cpu_rate([h_rgb.numpy()[f] for f in range(min(NB, 64))])
            except Exception as ex_:
                log('[bench] detector CPU baseline skipped: %r' % (ex_,))
        cpu = {'value': combine_rates(fps_all, det_cpu), 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
               'sample': '%d frames of the same batch on %d pinned C++ worker threads (tracking chain)%s' % (nrun, cores, '; detector restatement (PyTorch CPU, chunks of 16 frames, channels-last, all threads) on %d frames' % min(NB, 64) if use_det else ''),
               'tracking_chain_all_cores': fps_all, 'tracking_chain_single_thread': fps_one, 'tracking_chain_per_core': fps_all / cores, 'detector_all_cores': det_cpu}

    if rank == 0:
        line = {'metric': 'frames/sec ORB extract+match+dyn-reject %dx%d' % (W, H), 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
                'warmup': warm, 'ms_per_step': total_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u8',
                'data': 'synthetic',
                'config': {'workload': workload_name(cfg, use_det), 'frames_per_gpu_per_step': NB,
                           'l2_policy': 'inputs larger than L2: %d frames x %d B gray%s per step' % (NB, W * H, ' + %d B colour' % (W * H * 3) if use_det else ''),
                           'sharding': 'independent streams per rank, no data-path collective; one untimed ncclBroadcast of the vocabulary (35.6 MB of node descriptors + tree) at start-up',
                           'detector_in_step': bool(use_det),
                           'without_detector': {'value': world * NB / (trk_ms * 1e-3), 'unit': 'frames/s', 'ms_per_step': trk_ms,
                                                'note': 'the tracker-only step with ground-truth person boxes as inputs (the round-1 definition of the step)'},
                           'mean_keypoints': float(n0.mean()), 'mean_after_dynreject': float(res_gpu['cnt'].mean()), 'mean_matches': float(res_gpu['nm'].mean()),
                           'detector_person_boxes_per_frame': float(res_gpu['nb'].mean()) if use_det else None,
                           'detector': det_info, 'pose_chain': chain_info, 'full_chain_parity': parity},
                'clocks': clocks, 'e2e': e2e, 'gpu_launches': (TRACKER_LAUNCHES + (det.num_kernels if use_det else 0)) * args.steps, 'roofline': roofline, 'cpu_baseline': cpu}
        if bcast is not None:
            line['config']['startup_broadcast'] = bcast
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


DUMP_FRAMES = 128


def dump_step_outputs(out_dir, L, B, trk, nb, cap, with_det):
    """Writes what the last timed step left in the tracker -- what a caller of sgs_tracker_results_device (and sgs_tracker_boxes_device when the
    detector is in the step) receives -- as float32 / float64 .npy files under out_dir, at most 64 MB in all.  Per-frame arrays cover
    every frame; per-keypoint arrays cover a fixed sample of DUMP_FRAMES frames (seed 0, listed in sample_frames.npy), with the rows past a frame's
    count zeroed (they are scratch, not results).  The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    import torch
    torch.cuda.synchronize()
    p = [C.c_void_p() for _ in range(7)]
    B.check(L.sgs_tracker_results_device(trk.h, *[C.byref(x) for x in p]))
    counts = B.memcpy_d2h(np.zeros(nb, np.int32), p[3].value)
    sample = np.sort(np.random.default_rng(0).choice(nb, min(nb, DUMP_FRAMES), replace=False))
    valid = np.arange(cap)[None, :] < counts[sample, None]
    kps = B.memcpy_d2h(np.zeros((nb, cap), B.KP_DTYPE), p[0].value)[sample]
    out = {'counts': counts.astype(np.float64), 'nmatches': B.memcpy_d2h(np.zeros(nb, np.int32), p[5].value).astype(np.float64),
           'sample_frames': sample.astype(np.float64),
           'desc': np.where(valid[..., None], B.memcpy_d2h(np.zeros((nb, cap, 32), np.uint8), p[1].value)[sample], 0).astype(np.float32),
           'u_right': np.where(valid, B.memcpy_d2h(np.zeros((nb, cap), np.float32), p[2].value)[sample], 0).astype(np.float32),
           'cur_mp': np.where(valid, B.memcpy_d2h(np.zeros((nb, cap), np.int32), p[4].value)[sample], 0).astype(np.float64)}
    for f in B.KP_DTYPE.names:
        out['kp_' + f] = np.where(valid, kps[f], 0).astype(np.float32 if kps[f].dtype == np.float32 else np.float64)
    if with_det:
        pb, pn, ph = C.c_void_p(), C.c_void_p(), C.c_void_p()
        B.check(L.sgs_tracker_boxes_device(trk.h, C.byref(pb), C.byref(pn), C.byref(ph)))
        nboxes = B.memcpy_d2h(np.zeros(nb, np.int32), pn.value)
        boxes = B.memcpy_d2h(np.zeros((nb, trk.max_boxes, 4), np.float32), pb.value)
        boxes[np.arange(trk.max_boxes)[None, :] >= nboxes[:, None]] = 0
        out['boxes'], out['nboxes'] = boxes, nboxes.astype(np.float64)
        out['have_dyn'] = B.memcpy_d2h(np.zeros(nb, np.uint8), ph.value).astype(np.float64)
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)
    log('[bench] outputs of the last timed step written to %s (%.1f MB)' % (out_dir, sum(a.nbytes for a in out.values()) / 1e6))


def detector_gemm_table(det, kernel_ms, ncalls, nframes):
    """Joins the detector's kernel list (sgs_detector_describe) with its per-kernel times: algorithmic bytes and FLOPs of every 1x1-convolution GEMM for
    `nframes` frames -- activations in + out (FP32 NHWC), the weights once, the same-shape tensor operands of the fused tail (residual add, SE gate) --
    and the totals of the family."""
    import re
    ops = [l for l in det.describe().split('\n')[1:] if l]
    fam = {'launches': 0, 'ms': 0.0, 'bytes': 0.0, 'flop': 0.0}
    kinds = {}
    for j, op in enumerate(ops):
        kind = op.split()[0]
        t = kernel_ms[j + 1] / max(1, ncalls)
        kinds.setdefault(kind, [0, 0.0]); kinds[kind][0] += 1; kinds[kind][1] += t
        if kind != 'conv1x1':
            continue
        g = re.search(r'geom (\d+)x(\d+)x(\d+)->(\d+)x', op)
        cin, hh, ww, cout = [int(x) for x in g.groups()]
        npx = hh * ww * nframes
        tail = op.split('|', 1)[1] if '|' in op else ''
        ntensor = len(re.findall(r'(?:add|mul|sub|div)(?:\(rev\))? [0-9A-Za-z_]+ buf', tail))
        fam['launches'] += 1; fam['ms'] += t
        fam['bytes'] += (cin + cout + ntensor * cout) * 4.0 * npx + 4.0 * cin * cout
        fam['flop'] += 2.0 * cin * cout * npx
    kinds['preprocess'] = [1, kernel_ms[0] / max(1, ncalls)]
    kinds['detection_output'] = [2, (kernel_ms[-1] + kernel_ms[-2]) / max(1, ncalls)]
    return fam, {k: {'launches': v[0], 'ms': round(v[1], 4)} for k, v in kinds.items()}


def make_local_map(f, kps_c, desc_c, n_c, ti, mcap, cam, sf, rng, W, H):
    """Synthetic local map of frame f for the pose chain (sgs_tracker_pose_chain_device): every other last-frame point (those are 'seen' when matched), then
    points placed under every third keypoint of the current frame (candidates of the local search) with perturbed positions and descriptors; a few points
    are bad, a few have no observations, a few lie behind the camera.  Shared by tests/test_gpu_pose_chain.py."""
    from pysgs import synth
    depth = synth.depth_s1(W, H)
    m_last = int(ti['ln'][f])
    take_last = np.arange(0, m_last, 2)
    k = kps_c[:n_c]
    sel = np.arange(1, n_c, 3)
    kk = k[sel]
    z = depth[np.clip(kk['y'].astype(np.int64), 0, H - 1), np.clip(kk['x'].astype(np.int64), 0, W - 1)].astype(np.float32)
    xyz_new = np.stack([(kk['x'] - cam['cx']) * z / cam['fx'], (kk['y'] - cam['cy']) * z / cam['fy'], z], 1).astype(np.float32)
    xyz_new += rng.normal(0, 0.002, xyz_new.shape).astype(np.float32)
    d_new = desc_c[sel].copy()
    flip = rng.integers(0, 256, (len(sel), 6))
    np.bitwise_xor.at(d_new, (np.repeat(np.arange(len(sel)), 6), (flip >> 3).ravel()), (1 << (flip & 7)).astype(np.uint8).ravel())
    oct_new = kk['octave'].astype(np.int64)
    n = len(take_last) + len(sel)
    assert n <= mcap
    xyz = np.zeros((mcap, 3), np.float32); nrm = np.zeros((mcap, 3), np.float32); mn = np.zeros(mcap, np.float32); mx = np.zeros(mcap, np.float32)
    dsc = np.zeros((mcap, 32), np.uint8); valid = np.zeros(mcap, np.uint8); obs = np.zeros(mcap, np.uint8)
    xyz[:len(take_last)] = ti['lxyz'][f, take_last]; dsc[:len(take_last)] = ti['ldesc'][f, take_last]
    oct_all = np.concatenate([ti['loct'][f, take_last].astype(np.int64), oct_new])
    xyz[len(take_last):n] = xyz_new; dsc[len(take_last):n] = d_new
    dist = np.linalg.norm(xyz[:n], axis=1).astype(np.float32)
    mx[:n] = dist * sf[oct_all]; mn[:n] = mx[:n] / sf[-1]                # MapPoint::UpdateNormalAndDepth
    nrm[:n] = xyz[:n] / np.maximum(dist, 1e-6)[:, None]                   # mean viewing direction, camera at the origin
    valid[:n] = 1; valid[np.arange(5, n, 17)] = 0
    obs[:n] = 1; obs[np.arange(3, n, 11)] = 0
    xyz[np.arange(7, n, 29), 2] *= -1
    lid = np.full(ti['lxyz'].shape[1], -1, np.int32); lid[take_last] = np.arange(len(take_last))
    return dict(xyz=xyz, nrm=nrm, mn=mn, mx=mx, dsc=dsc, valid=valid, obs=obs, n=n, lid=lid)


def pin_rank_to_numa_node(local):
    """Host threads of this rank stay on the NUMA node of its GPU (pinned H2D from the far node halves the copy rate on 2-socket boxes)."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), 'pci_bus_id') else None
        node = None
        out = subprocess.run(['nvidia-smi', '-i', str(local), '--query-gpu=pci.bus_id', '--format=csv,noheader'], capture_output=True, text=True, timeout=10).stdout.strip()
        if out:
            p = '/sys/bus/pci/devices/%s/numa_node' % out.lower().replace('00000000:', '0000:')
            if os.path.exists(p):
                node = int(open(p).read().strip())
        if node is None or node < 0:
            return
        cpus = []
        for part in open('/sys/devices/system/node/node%d/cpulist' % node).read().strip().split(','):
            a, _, b = part.partition('-')
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            log('[bench] rank on GPU %d pinned to NUMA node %d (%d cpus)' % (local, node, len(allowed)))
        del bus
    except Exception as ex:
        log('[bench] NUMA pinning skipped: %r' % (ex,))


def vocabulary_broadcast(dist, rank, local, L, B, synth):
    """Shared read-only database: an ORBvoc-shaped vocabulary (k = 10, L = 6: 1,111,111 nodes x 32 B = 35.6 MB of node descriptors, SURVEY 8e).  Rank 0 owns
    it; with more than one rank it reaches the others through ONE ncclBroadcast at start-up (untimed, reported) and is consumed in place on the device."""
    import torch
    v = C.c_void_p
    VOC_K, VOC_L = 10, 6
    n = (VOC_K ** (VOC_L + 1) - 1) // (VOC_K - 1)
    desc = torch.from_numpy(synth.descriptors_s5(n, 5) if rank == 0 else np.zeros((n, 32), np.uint8)).cuda()
    info = None
    if dist is not None:
        warm_t = torch.zeros(1024, device='cuda'); dist.broadcast(warm_t, 0); torch.cuda.synchronize(); dist.barrier()      # communicator set up before timing
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record(); dist.broadcast(desc, 0); e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        info = {'bytes': int(desc.numel()), 'ms': ms, 'gb_per_s': desc.numel() / (ms * 1e-3) / 1e9}
    parent = ((np.arange(n, dtype=np.int64) - 1) // VOC_K).astype(np.int32); parent[0] = -1        # complete k-ary tree in breadth-first node order
    weight = np.zeros(n, np.float64); weight[(n - 1) // VOC_K:] = 1.0 + (np.arange(n - (n - 1) // VOC_K) % 7)
    h = v()
    B.check(L.sgs_vocabulary_create_device(local, VOC_K, VOC_L, n, parent.ctypes.data_as(v), v(desc.data_ptr()), weight.ctypes.data_as(v), C.byref(h)))
    L.sgs_vocabulary_destroy(h)
    return info


if __name__ == '__main__':
    main()
