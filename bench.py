#!/usr/bin/env python
"""bench.py -- frames/s of the DfM plane-sweep cost-volume path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # the CUDA path (default workload)
  python bench.py --impl reference ...                     # the reference's own CPU path
  python bench.py --workload waymo_mv | waymo_10sweep      # BASELINE.json configs[3] / [4]
  python bench.py ... --dump-outputs DIR                   # + last timed step's outputs, .npy

Workloads (one "step" = one pass of the hot path over one synthetic input):
  kitti          BASELINE.json configs[1]: one KITTI-shape pair, 370x1224 padded to 384x1248,
                 D=112 planes: DfMBackbone (warp + volume + 3-D aggregation + gate) + DepthHead
  waymo_mv       configs[3]: 5 views x [64,208,312] features -> lifting -> OutdoorImVoxelNeck
  waymo_10sweep  configs[4]: 2 frames x 5 views (the shipped 10-sweep config selects ONE
                 reference frame, SURVEY.md section 0) -> lifting (concat) -> DfMNeck

N > 1 is launched by torchrun, one rank per GPU: frames / samples are sharded over ranks
(independent; the reference cannot batch, dfm_backbone.py:160), no data-path collective,
"scaling": "weak" -- N replicas of the single-GPU path, not a partition of one frame.

One JSON line on stdout (rank 0).  Keys beyond the base contract:
  roofline            dominant kernel: algorithmic FLOPs (bytes) per launch / mean launch duration
                      (CUDA events inside the timed region, on the launching stream) vs the
                      measured peak in MEASURED_PEAKS.json
  cpu_baseline        the oracle (PyTorch-CPU port of the reference) on this host's cores
  gpu_eager_baseline  the same reference ops in PyTorch/cuDNN eager on this GPU, TF32 off / on
                      (protocol of tools/analysis_tools/benchmark.py:66-91: 5 warm-up frames)
  e2e                 same metric through the host-buffer C-ABI entry point a deployment
                      calls (pinned host inputs in, pinned host outputs out, H2D + D2H inside
                      the timed region)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, D, C = 384, 1248, 112, 32
HO, WO = H // 4, W // 4
ORI_SHAPE = (370, 1224, 3)
V = D * HO * WO
FLOPS_PER_FRAME = 521856.0 * V                       # SURVEY.md 8(d)
IO_BYTES_PER_FRAME = 2 * 32 * H * W * 4 + 5.25e6 + 33 * V * 4
KITTI_WORKLOAD = 'dfm_r34_1x8_kitti-3d-3class D=112 384x1248 batch=1'
# what one kitti step hands its caller: DfMBackbone's (cost, stereo, mono), DepthHead's 3 outputs
KITTI_OUTPUTS = ('cost', 'stereo_feat', 'mono_feat', 'depth_volumes', 'depth_volumes_softmax',
                 'depth_preds')
# --dump-outputs: an output with more elements than this is stored as a fixed, seeded sample;
# six outputs of at most 8 MiB each stay within DUMP_MAX_BYTES
DUMP_MAX_ELEMS = 1 << 21
DUMP_MAX_BYTES = 64 << 20
DUMP_SEED = 0
# dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel, from the
# committed `ncu --set full` capture (profiles/): kitti: conv_tc 32->32 full resolution
NCU_TRAFFIC = {'kitti': (973.0e6, 'profiles/r02_ncu_conv_tc_dominant_final.csv '
                                  '(587.1 MB read + 386.0 MB written per launch)')}
WAYMO = {
    'waymo_mv': dict(T=1, agg='mean', neck='OutdoorImVoxelNeck', flops=3.212e12,
                     name='multiview-dfm_r101_dcn_2x16_waymoD5 (5 views, 832x1248 input) '
                          'lifting + OutdoorImVoxelNeck, 1 sample'),
    'waymo_10sweep': dict(T=2, agg='concat', neck='DfMNeck', flops=7.649e12,
                          name='multiview-dfm_r101_dcn 10sweeps config (2 frames x 5 views) '
                               'lifting(concat) + DfMNeck, 1 sample'),
}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        j = json.load(open(p))
        return dict(bf16=j.get('bf16_tflops_sustained', j.get('bf16_tflops')),
                    hbm=j.get('hbm_gbs'), src='measured')
    return dict(bf16=1400.0, hbm=6650.0, src='fallback')  # B200_PROFILING.md


def dump_outputs(out_dir, arrays):
    """Writes each named output as ``<out_dir>/<name>.npy`` (float32 or float64), so that two
    builds run with the same arguments can be compared output for output.  An output with at
    most DUMP_MAX_ELEMS elements is written whole, in its own shape; a larger one as the 1-D
    array of its elements at DUMP_MAX_ELEMS flat indices drawn (with replacement, then sorted)
    from a CPU generator seeded with DUMP_SEED, which depend only on the output's size."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            g = torch.Generator().manual_seed(DUMP_SEED)
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=g).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        a = t.cpu().numpy()
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float32)
        total += a.nbytes
        if total > DUMP_MAX_BYTES:
            raise RuntimeError(f'--dump-outputs: more than {DUMP_MAX_BYTES} bytes at {name}')
        np.save(os.path.join(out_dir, name + '.npy'), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}',
                 '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 7 and r[0].isdigit()]
        if not rows:
            return None
        sm = [int(r[0]) for r in rows]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[3 + i] == 'Active' for r in rows)]
        return dict(sm_mhz=int(statistics.median(sm)), sm_max_mhz=int(rows[0][1]),
                    samples=len(rows), reasons=reasons)


# ------------------------------------------------------------------------------------
# the reference's own path (oracle port), on the host cores or in eager mode on the GPU
# ------------------------------------------------------------------------------------
def _oracle_kitti_frame(device, seed=0):
    """A closure running one whole reference frame (DfMBackbone.forward + DepthHead.forward,
    dfm_backbone.py:143-214, depth_head.py:190-212) on `device`."""
    import torch

    from depth_from_motion_b200 import synthetic as syn
    from oracle import dfm_oracle as O
    cur, prev, metas, params = syn.make_kitti_pair(seed, H, W, D, ori_shape=ORI_SHAPE)
    cfg = syn.depth_cfg_for(D)
    cur, prev = cur.to(device), prev.to(device)
    params = {k: v.to(device) for k, v in params.items()}
    samples = O.depth_samples(cfg).to(device)

    def frame():
        with torch.no_grad():
            cost, _, _ = O.dfm_backbone_forward(params, cur, prev, metas, cfg)
            return O.depth_head_forward(cost, samples)[2]
    return frame


def _oracle_waymo_sample(device, wl, seed=0):
    import numpy as np
    import torch

    from depth_from_motion_b200 import modules
    from depth_from_motion_b200 import synthetic as syn
    from oracle import dfm_oracle as O
    spec = WAYMO[wl]
    t, nv = spec['T'], 5
    feats, meta = syn.make_waymo_sample(seed, t, nv)
    rng = np.random.RandomState(seed + 1)
    mod = (modules.DfMNeck(64, 256, num_frames=2) if spec['neck'] == 'DfMNeck'
           else modules.OutdoorImVoxelNeck(64, 256))
    sd = {k: v.to(device) for k, v in syn.make_neck_params(rng, mod.state_dict()).items()}
    xs, ys, zs = modules.aligned_voxel_centers(syn.WAYMO_N_VOXELS, syn.WAYMO_RANGE)
    zz, yy, xx = torch.meshgrid(zs, ys, xs, indexing='ij')
    pts = torch.stack([xx, yy, zz], -1).reshape(-1, 3).to(device)
    l2i = [torch.tensor(m, dtype=torch.float32, device=device) for m in meta['ori_lidar2img']]
    feats = feats.to(device)
    sf = pts.new_tensor(meta['scale_factor'][:2])
    crop = pts.new_tensor(meta['img_crop_offset'])

    def sample():
        with torch.no_grad():
            vol = O.multiview_lift(feats, pts, syn.WAYMO_N_VOXELS, l2i, nv, t, sf, crop, False,
                                   meta['input_shape'], meta['img_shape'], spec['agg'])[None]
            if spec['neck'] == 'DfMNeck':
                return O.dfm_neck_forward(sd, vol, 64)[0]
            return O.imvoxel_neck_forward(sd, vol)[0]
    return sample


def _reference_step(workload, device):
    return _oracle_kitti_frame(device) if workload == 'kitti' else \
        _oracle_waymo_sample(device, workload)


def run_reference(args):
    """--impl reference: the reference's own PyTorch path on the host cores (the oracle port:
    the reference has no native code to compile and mmcv is not installable here, DESIGN.md
    section 6).  Every step is ONE WHOLE unit of the stated workload -- no extrapolation."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step = _reference_step(args.workload, 'cpu')
    for _ in range(args.warmup):
        step()
    ts = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        last = step()
        ts.append(time.perf_counter() - t0)
    if args.dump_outputs:
        name = 'depth_preds' if args.workload == 'kitti' else 'volume_feat'
        dump_outputs(args.dump_outputs, {name: last})
    per_step = sum(ts) / len(ts)
    fps = 1.0 / per_step
    name = KITTI_WORKLOAD if args.workload == 'kitti' else WAYMO[args.workload]['name']
    line = dict(
        impl='reference', metric='frames/sec', value=fps, unit='frames/s', n_gpus=args.gpus,
        steps=args.steps, warmup=args.warmup, ms_per_step=per_step * 1e3,
        higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
        data='synthetic', config=dict(workload=name),
        cpu_baseline=dict(value=fps, unit='frames/s', cores=cores, kind='port',
                          sample=f'every step is one whole unit of this workload through the '
                                 f'oracle (PyTorch-CPU restatement of the reference path); '
                                 f'{args.warmup} warm-up + {args.steps} timed, '
                                 f'median {statistics.median(ts):.2f} s, '
                                 f'min {min(ts):.2f} s, max {max(ts):.2f} s'),
        e2e=dict(value=fps, unit='frames/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


def gpu_eager_baseline(workload, nwarm=5, nrep=10):
    """The reference modules' own op sequence in PyTorch/cuDNN eager mode on this GPU (the
    same-box bar of SURVEY.md section 2.2 / 8d), cuDNN TF32 off (true fp32) and on (torch's
    default, what the reference's authors ran), tools/analysis_tools/benchmark.py:66-91."""
    import torch
    out = {}
    step = _reference_step(workload, 'cuda')
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        for key, tf32 in (('tf32_off', False), ('tf32_on', True)):
            torch.backends.cudnn.allow_tf32 = tf32
            for _ in range(nwarm):
                step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(nrep):
                step()
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) / nrep * 1e3
            out[key] = dict(ms_per_frame=round(ms, 3), frames_per_s=round(1e3 / ms, 2))
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    out['what'] = ('oracle/dfm_oracle.py (the reference ops, same order) on cuda tensors, '
                   f'{nwarm} warm-up + {nrep} timed frames, torch {torch.__version__}, cuDNN '
                   f'{torch.backends.cudnn.version()}')
    del step
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------
# the CUDA path
# ------------------------------------------------------------------------------------
def _setup_dist():
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a B200: there is no CPU path (use --impl reference)')
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL's INFO lines (if the caller set NCCL_DEBUG) must not interleave with the one
        # JSON line on stdout: send them to stderr's file unless the caller chose a file
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    return rank, world, local


def _timed_loop(step, args, world, rank, local, capi):
    """W warm-up steps, then exactly K timed steps between barrier + synchronize on both
    sides, CUDA events on the launching stream, clocks sampled during the timed region.
    Also returns what the last timed step returned."""
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for i in range(args.warmup):
            step(i)
        capi.sync_check()
        l0, tc0 = capi.launch_counters()
        capi.profile_enable(True)
        capi.profile_report()
        sampler = ClockSampler(local)
        barrier()
        if rank == 0:
            sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps - 1):
            step(i)
        last = step(args.steps - 1)
        e1.record()
        barrier()
        clocks = sampler.stop() if rank == 0 else None
        ms = e0.elapsed_time(e1)
        prof = capi.profile_report()
        capi.profile_enable(False)
        l1, tc1 = capi.launch_counters()
        capi.sync_check()
    from depth_from_motion_b200.sharding import reduce_step_time
    return reduce_step_time(ms, 'cuda'), prof, clocks, l1 - l0, tc1 - tc0, barrier, last


def _kernel_table(prof, steps):
    return {k: dict(launches=v['launches'] // steps, ms=round(v['ms'] / steps, 4),
                    tflops=round(v['flops'] / max(v['ms'], 1e-9) / 1e9, 1))
            for k, v in sorted(prof.items(), key=lambda kv: -kv[1]['ms'])}


def run_kitti(args):
    import torch
    import torch.distributed as dist

    from depth_from_motion_b200 import capi, modules
    from depth_from_motion_b200 import synthetic as syn
    from depth_from_motion_b200.sharding import reduce_step_time

    rank, world, local = _setup_dist()
    capi.lib()

    # two different pairs per rank so consecutive steps never re-read the same inputs;
    # the per-step working set (~7 GB of activations) is far larger than the 126 MB L2
    pairs = []
    for i in range(2):
        cur, prev, metas, params = syn.make_kitti_pair(100 + 2 * rank + i, H, W, D,
                                                       ori_shape=ORI_SHAPE)
        metas[0]['cam2img'] = syn.KITTI_P2.astype('float32').tolist()
        pairs.append((cur.cuda(), prev.cuda(), metas, cur.pin_memory(), prev.pin_memory()))
    cfg = syn.depth_cfg_for(D)
    model = modules.DfMBackbone(in_channels=C, depth_cfg=cfg).cuda().eval()
    model.load_state_dict(params, strict=True)
    model.downsampled_depth = _depths(cfg, 4)
    head = modules.DepthHead(
        depth_cfg=dict(mode='UD', num_bins=cfg['num_bins'], min_depth=2, max_depth=59.6),
        with_convs=False, num_views=1, depth_loss=dict(type='ce', loss_weight=1.0))
    head.depth_samples = _depths(cfg, 1)
    head.downsample_factor = 4

    def step(i):
        cur, prev, metas, _, _ = pairs[i % 2]
        cost, stereo, mono = model(cur, prev, metas)
        return (cost, stereo, mono) + tuple(head(cost))

    ms_total, prof, clocks, launches, tc_launches, barrier, last = _timed_loop(
        step, args, world, rank, local, capi)
    fps = world * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(KITTI_OUTPUTS, last)))
    del last

    # ---- e2e: DfM.simple_test's hot-path segment through the host-buffer C-ABI call -------
    # pinned host (cur, prev, sem) in -> voxel features + depth_preds out (what the BEV stage
    # consumes, detectors/dfm.py:416-429); every step copies one pair H2D (the NEXT pair, on a
    # side stream, overlapped with this step's compute) and its outputs D2H, all inside the
    # timed region
    fc = syn.make_frustum_case(7 + rank, H, W, D, (288, 304, 20))
    frustum = modules.FrustumToVoxel().eval()
    frustum.load_state_dict(fc['params'], strict=True)
    frustum = frustum.cuda()
    frustum.coordinates_3d = fc['coordinates_3d']
    frustum.depth_cfg = cfg
    h_sem = fc['sem'].contiguous().pin_memory()
    pipe = modules.HotPathPipeline(model, head, frustum)
    del fc
    use_prefetch = [False]

    def e2e_sync_step(i):
        _, _, metas, hc, hp = pairs[i % 2]
        return pipe(hc, hp, h_sem, metas)

    def e2e_submit(i):
        # start copying the NEXT pair (side stream), enqueue this frame (its pair was staged one
        # step earlier), then collect the PREVIOUS frame's outputs, whose device->host copy ran
        # underneath this frame's compute
        _, _, metas, hc, hp = pairs[i % 2]
        if use_prefetch[0]:
            nxt = pairs[(i + 1) % 2]
            pipe.prefetch(nxt[3], nxt[4], h_sem)
        pipe.submit(hc, hp, h_sem, metas)

    # self-check: the asynchronous, prefetched path must reproduce the plain synchronous call
    ref_vox = e2e_sync_step(0)[0].clone()
    try:
        pipe.prefetch(pairs[0][3], pairs[0][4], h_sem)
        use_prefetch[0] = True
        e2e_submit(0)
        if not torch.allclose(pipe.wait()[0], ref_vox, rtol=1e-5, atol=1e-6):
            raise RuntimeError('asynchronous / prefetched result differs')
    except RuntimeError as exc:
        print(f'[bench] prefetch path disabled: {exc}', file=sys.stderr)
        use_prefetch[0] = False
    nwarm = min(args.warmup, 3)
    e2e_submit(1)
    for i in range(2, 1 + nwarm):
        e2e_submit(i)
        pipe.wait()
    barrier_host = pipe.wait     # drain before timing
    barrier_host()
    barrier()
    t0 = time.perf_counter()
    ee0, ee1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ee0.record()
    first = 1 + nwarm
    e2e_submit(first)
    for i in range(first + 1, first + args.steps):
        e2e_submit(i)
        pipe.wait()              # outputs of frame i-1 are in host memory
    pipe.wait()                  # ... and of the last frame
    ee1.record()
    barrier()
    e2e_ms = reduce_step_time(max(ee0.elapsed_time(ee1), (time.perf_counter() - t0) * 1e3),
                              'cuda')
    e2e_fps = world * args.steps / (e2e_ms * 1e-3)
    vox_out, pred_out = pipe._out
    h2d = 2 * C * H * W * 4 + h_sem.numel() * 4 + D * 4 * 4
    d2h = (vox_out.numel() + pred_out.numel()) * 4

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    dom_key = f'conv_tc<32->32,s1,src>@{D}x{HO}x{WO}'
    roof = None
    tc_ms = sum(v['ms'] for k, v in prof.items() if k.startswith('conv_tc'))
    conv_ms = sum(v['ms'] for k, v in prof.items() if k.startswith('conv_'))
    if dom_key in prof:
        r = prof[dom_key]
        per_launch_flops = r['flops'] / r['launches']
        per_launch_s = r['ms'] * 1e-3 / r['launches']
        ach = per_launch_flops / per_launch_s / 1e12
        roof = dict(bound='tensor', kernel=dom_key, achieved=round(ach, 2), peak=pk['bf16'],
                    unit='TFLOP/s', frac=round(ach / pk['bf16'], 4),
                    traffic=NCU_TRAFFIC['kitti'][0], traffic_source=NCU_TRAFFIC['kitti'][1],
                    algorithmic_bytes=2 * V * 32 * 4,
                    executed_bf16_tflops=round(3 * ach, 1),
                    executed_frac_of_peak=round(3 * ach / pk['bf16'], 4),
                    peak_source=pk['src'] + ' bf16 dense (sustained)',
                    launches_per_step=r['launches'] / args.steps,
                    ms_per_launch=round(per_launch_s * 1e3, 4),
                    note='achieved = algorithmic fp32 conv FLOPs (2*V*27*Cin*Cout); the kernel '
                         'executes 3 bf16 MMAs per product (hi/lo split) for fp32-class '
                         'accuracy, so the tensor pipe runs at 3x this rate',
                    share_of_step=round(r['ms'] / ms_total, 4))
    else:
        simt = {k: v for k, v in prof.items() if k.startswith('conv_simt')}
        if simt:
            k, r = max(simt.items(), key=lambda kv: kv[1]['ms'])
            ach = r['flops'] / (r['ms'] * 1e-3) / 1e12
            roof = dict(bound='tensor', kernel=k, achieved=round(ach, 2), peak=pk['bf16'],
                        unit='TFLOP/s', frac=round(ach / pk['bf16'], 4), traffic=None,
                        peak_source=pk['src'])
    # HBM-bound kernels of the step against the measured copy bandwidth (algorithmic bytes)
    hbm_rows = {}
    alg = {'depth_head': 2 * (4 * D) * H * W * 4 + V * 4,
           'cout1_logits': V * 32 * 4 + V * 4,
           'gate': 3 * V * 4,
           'presplit': 3 * V * 32 * 4}     # two fp32 terms read, one pre-split tensor written
    for key, nbytes in alg.items():
        rows = [v for k, v in prof.items() if k == key or k.startswith(key)]
        if rows:
            ms = sum(v['ms'] for v in rows) / args.steps
            if key in ('cout1_logits', 'presplit'):   # stereo (D planes) + shortened mono (40)
                nbytes = nbytes * (1 + 40.0 / D)
            hbm_rows[key] = dict(ms=round(ms, 4), algorithmic_gb=round(nbytes / 1e9, 3),
                                 gbs=round(nbytes / ms / 1e6, 1),
                                 frac_of_hbm_peak=round(nbytes / ms / 1e6 / pk['hbm'], 3))
    cores = os.cpu_count() or 1
    cpu = eager = None
    if world == 1 and not args.no_cpu_baseline:
        import torch as _t
        _t.set_num_threads(cores)
        frame = _oracle_kitti_frame('cpu')
        frame()                                   # warm-up (thread pool, allocator)
        t0 = time.perf_counter()
        frame()
        t_cpu = time.perf_counter() - t0
        cpu = dict(value=1.0 / t_cpu, unit='frames/s', cores=cores, kind='port',
                   sample=f'one whole frame of this workload (D={D}, {H}x{W}) through the '
                          f'oracle (PyTorch-CPU restatement of the reference path) after one '
                          f'warm-up frame, {t_cpu:.1f} s')
    if world == 1 and not args.no_gpu_eager:
        eager = gpu_eager_baseline('kitti')
    line = dict(
        metric='frames/sec', value=fps, unit='frames/s', n_gpus=world, steps=args.steps,
        warmup=args.warmup, ms_per_step=ms_total / args.steps, higher_is_better=True,
        scaling='weak', vs_baseline=None, dtype='f32 (bf16x2 split operands, fp32 accumulate)',
        data='synthetic',
        config=dict(workload=KITTI_WORKLOAD, pairs_per_step=world, planes=D, feature_hw=[H, W],
                    l2='per-step working set ~7 GB >> 126 MB L2; two input pairs alternate',
                    multi_gpu='replicas: one independent pair per rank, no data-path collective',
                    outputs='cost + stereo_feat + mono_feat + DepthHead(volume, softmax, preds)'),
        clocks=clocks,
        comm=dict(backend='nccl' if world > 1 else None, world_size=world,
                  collective='all_reduce(MAX) of the step time only'),
        e2e=dict(value=e2e_fps, unit='frames/s', h2d_bytes_per_step=h2d,
                 d2h_bytes_per_step=d2h, prefetch=use_prefetch[0],
                 ms_per_step=round(e2e_ms / args.steps, 4),
                 what='dfm_pipeline_submit_host / dfm_pipeline_wait (K frames submitted, K results '
                      'collected inside the timed region; the D2H copy of frame i overlaps the '
                      'compute of frame i+1): pinned host cur/prev stereo features + sem '
                      'features in -> DfMBackbone -> DepthHead reduction -> FrustumToVoxel -> '
                      'pinned host voxel features [1,32,5,304,288] + depth_preds [1,1,384,1248] '
                      'out (what DfM.simple_test hands to the BEV stage, detectors/dfm.py:'
                      '416-429); the next pair is prefetched on a side stream'),
        gpu_launches=launches, tc_launches=tc_launches,
        roofline=roof, hbm_kernels=hbm_rows,
        tensor=dict(achieved_tflops=round(FLOPS_PER_FRAME * fps / world / 1e12, 2),
                    frac_of_bf16_peak=round(FLOPS_PER_FRAME * fps / world / 1e12 / pk['bf16'], 4)),
        hbm=dict(compulsory_gbs=round(IO_BYTES_PER_FRAME * fps / world / 1e9, 1),
                 frac_of_peak=round(IO_BYTES_PER_FRAME * fps / world / 1e9 / pk['hbm'], 4)),
        conv_ms_per_step=round(conv_ms / args.steps, 3),
        tc_conv_ms_per_step=round(tc_ms / args.steps, 3),
        kernels=_kernel_table(prof, args.steps),
        cpu_baseline=cpu, gpu_eager_baseline=eager)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_waymo(args):
    """BASELINE.json configs[3] / [4]: per sample, MultiViewDfM.feature_transformation =
    multi-view lifting (multiview_dfm.py:119-209) + neck_3d (imvoxel_neck.py / dfm_neck.py)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    from depth_from_motion_b200 import capi, modules
    from depth_from_motion_b200 import synthetic as syn
    from depth_from_motion_b200.sharding import reduce_step_time

    rank, world, local = _setup_dist()
    capi.lib()
    spec = WAYMO[args.workload]
    t, nv = spec['T'], 5
    samples = []
    for i in range(2):
        feats, meta = syn.make_waymo_sample(200 + 2 * rank + i, t, nv)
        samples.append((feats.cuda(), meta, feats.pin_memory()))
    rng = np.random.RandomState(5)
    neck = (modules.DfMNeck(64, 256, num_frames=2) if spec['neck'] == 'DfMNeck'
            else modules.OutdoorImVoxelNeck(64, 256))
    neck.load_state_dict(syn.make_neck_params(rng, neck.state_dict()), strict=True)
    neck = neck.cuda().eval()

    class Host(modules.MultiViewDfMFeatureTransformation):
        n_voxels, voxel_range = syn.WAYMO_N_VOXELS, syn.WAYMO_RANGE
        temporal_aggregate, valid_sample, neck_3d = spec['agg'], True, neck
    host = Host()

    def step(i):
        feats, meta, _ = samples[i % 2]
        return host.feature_transformation(feats[None], [meta], nv, t)[0]

    ms_total, prof, clocks, launches, tc_launches, barrier, last = _timed_loop(
        step, args, world, rank, local, capi)
    sps = world * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(volume_feat=last))
    del last

    # ---- e2e: pinned host features in, pinned host BEV out --------------------------------
    # every step copies its sample H2D (166 / 83 MB) and its BEV map D2H (67.6 MB) inside the timed
    # region; the copy of sample i+1 and the read-back of result i-1 ride side streams underneath
    # step i (double-buffered on both sides), each result is waited for one step later
    cur_s = torch.cuda.current_stream()
    in_s, out_s = torch.cuda.Stream(), torch.cuda.Stream()
    d_in = [torch.empty_like(samples[0][0]) for _ in range(2)]
    h_bev = [torch.empty((1, 256, 300, 220)).pin_memory() for _ in range(2)]
    ev_in = [torch.cuda.Event() for _ in range(2)]       # sample staged
    ev_free = [torch.cuda.Event() for _ in range(2)]     # staging buffer consumed
    ev_out = [torch.cuda.Event() for _ in range(2)]      # result in host memory

    def stage(i):
        b = i % 2
        with torch.cuda.stream(in_s):
            in_s.wait_event(ev_free[b])
            d_in[b].copy_(samples[i % 2][2], non_blocking=True)
            ev_in[b].record(in_s)

    def e2e_step(i):
        b = i % 2
        stage(i + 1)
        cur_s.wait_event(ev_in[b])
        bev = host.feature_transformation(d_in[b][None], [samples[i % 2][1]], nv, t)[0]
        ev_free[b].record(cur_s)
        done = torch.cuda.Event()
        done.record(cur_s)
        bev.record_stream(out_s)
        with torch.cuda.stream(out_s):
            out_s.wait_event(done)
            h_bev[b].copy_(bev, non_blocking=True)
            ev_out[b].record(out_s)
        if i > 0:
            ev_out[(i - 1) % 2].synchronize()    # result of step i-1 is in host memory

    with torch.no_grad():
        for b in range(2):
            ev_free[b].record(cur_s)
        stage(0)
        for i in range(3):
            e2e_step(i)
        ev_out[2 % 2].synchronize()
        barrier()
        t0 = time.perf_counter()
        for i in range(3, 3 + args.steps):
            e2e_step(i)
        ev_out[(3 + args.steps - 1) % 2].synchronize()
        torch.cuda.synchronize()
        barrier()
        e2e_ms = reduce_step_time((time.perf_counter() - t0) * 1e3, 'cuda')
    e2e_sps = world * args.steps / (e2e_ms * 1e-3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    neck_ms = sum(v['ms'] for k, v in prof.items() if k.startswith('conv_')) / args.steps
    lift_ms = sum(v['ms'] for k, v in prof.items() if k.startswith('lift')) / args.steps
    in_bytes = samples[0][0].numel() * 4
    out_bytes = 64 * (t if spec['agg'] == 'concat' else 1) * 220 * 300 * 12 * 4
    ach = spec['flops'] / (neck_ms * 1e-3) / 1e12 if neck_ms else 0.0
    roof = dict(bound='tensor', kernel=f'conv_tc_neck (all 9/18 conv layers of {spec["neck"]})',
                achieved=round(ach, 2), peak=pk['bf16'], unit='TFLOP/s',
                frac=round(ach / pk['bf16'], 4), traffic=None,
                executed_bf16_tflops=round(3 * ach, 1),
                peak_source=pk['src'] + ' bf16 dense (sustained)',
                ms_per_step=round(neck_ms, 3), share_of_step=round(neck_ms * args.steps / ms_total, 4),
                note='algorithmic fp32 conv FLOPs of the neck (SURVEY.md 8d) / summed conv time')
    roof_lift = dict(bound='hbm', kernel='lift (NCHW->NHWC staging of the 2-D features + lift_cl_kernel, channels-last volume out)',
                     achieved=round((in_bytes + out_bytes) / (lift_ms * 1e-3) / 1e9, 1) if lift_ms else None,
                     peak=pk['hbm'], unit='GB/s',
                     frac=round((in_bytes + out_bytes) / (lift_ms * 1e-3) / 1e9 / pk['hbm'], 4) if lift_ms else None,
                     algorithmic_bytes=in_bytes + out_bytes, ms_per_step=round(lift_ms, 4))
    cores = os.cpu_count() or 1
    cpu = eager = None
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(cores)
        fn = _oracle_waymo_sample('cpu', args.workload)
        t0 = time.perf_counter()
        fn()
        t_cpu = time.perf_counter() - t0
        cpu = dict(value=1.0 / t_cpu, unit='frames/s', cores=cores, kind='port',
                   sample=f'one whole sample of this workload through the oracle, {t_cpu:.1f} s')
    if world == 1 and not args.no_gpu_eager:
        eager = gpu_eager_baseline(args.workload, nwarm=2, nrep=3)
    line = dict(
        metric='frames/sec', value=sps, unit='frames/s', n_gpus=world, steps=args.steps,
        warmup=args.warmup, ms_per_step=ms_total / args.steps, higher_is_better=True,
        scaling='weak', vs_baseline=None, dtype='f32 (bf16x2 split operands, fp32 accumulate)',
        data='synthetic',
        config=dict(workload=spec['name'], samples_per_step=world, frames=t, views=nv,
                    n_voxels=syn.WAYMO_N_VOXELS, frame_unit='one multi-view sample',
                    l2='volume 0.2-0.4 GB and 0.4-1.5 GB of activations per layer >> 126 MB L2; '
                       'two input samples alternate',
                    multi_gpu='replicas: one independent sample per rank'),
        clocks=clocks,
        comm=dict(backend='nccl' if world > 1 else None, world_size=world,
                  collective='all_reduce(MAX) of the step time only'),
        e2e=dict(value=e2e_sps, unit='frames/s', h2d_bytes_per_step=in_bytes,
                 d2h_bytes_per_step=h_bev[0].numel() * 4, ms_per_step=round(e2e_ms / args.steps, 3),
                 what='pinned host FPN features [T*5,64,208,312] -> H2D -> '
                      'MultiViewDfM.feature_transformation (lifting + neck_3d) -> BEV '
                      '[1,256,300,220] D2H to pinned host memory; the copy of sample i+1 and the '
                      'read-back of result i-1 run on side streams underneath step i, every step '
                      'waits for the previous result'),
        gpu_launches=launches, tc_launches=tc_launches, roofline=roof, roofline_lift=roof_lift,
        kernels=_kernel_table(prof, args.steps), cpu_baseline=cpu, gpu_eager_baseline=eager)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def _depths(cfg, ds):
    import torch
    nb = cfg['num_bins']
    interval = (cfg['depth_max'] - cfg['depth_min']) / nb
    d = torch.zeros(nb // ds, dtype=torch.float32)
    for i in range(nb // ds):
        d[i] = (i + 0.5) * ds * interval + cfg['depth_min']
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='kitti', choices=['kitti'] + sorted(WAYMO))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gpu-eager', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3)
    if args.impl == 'reference':
        run_reference(args)
    elif args.workload == 'kitti':
        run_kitti(args)
    else:
        run_waymo(args)


if __name__ == '__main__':
    main()
