#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native SHAPY hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 64] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

metric : bodies/sec, image -> SMPL-X vertices (+ betas, measurements), B = 64 per GPU (BASELINE configs[2],
         "Full SHAPY_A regressor (HRNet + iterative head + fused SMPL-X), batch=64, 1xB200, fp32 tol 1e-4";
         configs[4] shards 64 images per GPU, i.e. weak scaling).
value  : whole-job bodies/s with the images already resident in HBM (CUDA events, max over ranks).
e2e    : the same metric through the public serving loop with HOST buffers (shapy_b200.pipeline.HostPipeline around
         SMPLXRegressor.forward): every rank copies its own pinned host images H2D, runs the forward and copies
         vertices / betas / measurements D2H, the three stages overlapped across consecutive batches on three
         streams; all copies sit inside the timed region (one interval over the K batches, max over ranks).
roofline: the dominant kernel is the tcgen05 implicit-GEMM convolution (HRNet = ~99 % of the step);
         achieved = algorithmic conv FLOPs (36.93 GFLOP / image @224^2, SURVEY.md 8d) / HRNet device time.
         `roofline_lbs` / `roofline_shape` report the HBM rooflines of the fused SMPL-X kernels.
cpu_baseline / --impl reference: the CPU restatement of the reference path (oracle/, "port") timed on the
         box's host cores on a bounded sample of the same workload: one warm-up pass, then timed passes over the same
         sample (the in-line cpu_baseline and the --impl reference arm use the same procedure).  The in-line leg
         is also the bench's SELF-CHECK: the oracle's vertices / betas / measurements of the sampled images are
         compared with the GPU outputs of the same images before anything is timed ("selfcheck" in the line).
config2 : BASELINE configs[1] (HRNet-W48 only, plain fp16 operands, B = 32) timed in the same run.
dump    : --dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy, float32 or float64, at
         most 64 MB (a seeded sample of the batch rows beyond that): two builds can be compared output for output, the
         inputs being seeded.
config5 : (N > 1) BASELINE configs[4]: rank 0 holds the whole batch (N x 64 uint8 images) in HBM, NCCL scatter ->
         on-device crop / normalise -> forward -> NCCL gather of vertices / betas / measurements to rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'bodies/sec image->SMPL-X verts @ B=64 per GPU'
CONV_GFLOP_PER_IMAGE_224 = 36.93            # SURVEY.md 8d (2 x 18.4665 GMAC), conv-only
LBS_CONST_BYTES = 68.93e6                    # dense SMPL-X constants streamed by lbs() (SURVEY.md 8d)
LBS_BODY_BYTES = 254896                      # per-body compulsory I/O
SHAPE_CONST_BYTES = 1.38e6
SHAPE_BODY_BYTES = 40 + 125700
DUMP_LIMIT_BYTES = 64 << 20


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tf_burst=d['bf16_tflops'], tf_sustained=d.get('bf16_tflops_sustained', d['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.rows, self.stop, self.index = [], False, index
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop:
            try:
                o = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-i',
                                    str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([c.strip() for c in o.split(',')])
            except Exception:
                pass
            time.sleep(0.05)     # nvidia-smi itself takes ~0.1 s: 5-7 samples per second of timed region

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit())
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.rows[0][1]), 'reasons': reasons,
                'samples': len(sm)}


def conv_traffic(batch: int, mode: int):
    """DRAM bytes (read + write) of all conv launches of one HRNet forward, from the committed ncu capture
    profiles/r02_traffic.json (r01 if absent; taken at B=64, split mode); None for any other configuration."""
    path = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    if not os.path.exists(path):
        path = os.path.join(ROOT, 'profiles', 'r01_traffic.json')
    if batch != 64 or mode != 1 or not os.path.exists(path):
        return None
    with open(path) as f:
        return json.load(f).get('conv_dram_bytes_per_step')


def lbs_traffic(batch: int):
    """DRAM bytes of one SMPL-X forward (fused LBS + joints kernels) from the committed ncu capture; B=64 only."""
    path = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    if batch != 64 or not os.path.exists(path):
        return None
    with open(path) as f:
        return json.load(f).get('lbs_B64', {}).get('dram_bytes_per_call')


def usable_cores() -> int:
    """Host threads this process may really use: CPU affinity, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        pass
    return max(1, min(n, 64))


def output_arrays(out, prefix='', seen=None):
    """{dotted name: host array} of every tensor in a forward's output (`stage_02.vertices`, `measurements.chest`,
    `camera_parameters.scale`, ...).  float32 / float64 stay as they are, other dtypes become float64 (exact for the
    integer tables); an object met twice (the measurement dict, faces, proj_joints) is written once."""
    import numpy as np
    import torch
    seen = set() if seen is None else seen
    if id(out) in seen:
        return {}
    seen.add(id(out))
    if isinstance(out, dict):
        items = out.items()
    elif hasattr(out, 'KEYS'):                                              # CameraParams
        items = ((k, getattr(out, k, None)) for k in out.KEYS)
    else:
        a = getattr(out, '_t', out)                                         # KeypointTensor wraps its tensor
        if torch.is_tensor(a):
            a = a.detach().cpu().numpy()
        if not isinstance(a, np.ndarray):
            return {}
        return {prefix: a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)}
    arrays = {}
    for k, v in sorted(items, key=lambda kv: str(kv[0])):
        arrays.update(output_arrays(v, f'{prefix}.{k}' if prefix else str(k), seen))
    return arrays


def dump_outputs(arrays, batch, path):
    """Writes `arrays` as path/<name>.npy; above DUMP_LIMIT_BYTES only a seeded sample of the batch rows is written."""
    import numpy as np
    per_row = sum(a.nbytes // batch for a in arrays.values() if a.ndim and a.shape[0] == batch)
    fixed = sum(a.nbytes for a in arrays.values()) - per_row * batch
    n = min(batch, (DUMP_LIMIT_BYTES - fixed) // max(per_row, 1))
    if n < batch:
        rows = np.sort(np.random.default_rng(0).choice(batch, n, replace=False))
        arrays = {k: a[rows] if a.ndim and a.shape[0] == batch else a for k, a in arrays.items()}
        print(f'bench: --dump-outputs keeps {n} of {batch} rows', file=sys.stderr)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + '.npy'), a)


def cpu_reference_step(sd, smplx, lm, x):
    """One pass of the CPU restatement of the reference path (oracle/) over the images `x`."""
    import torch
    from oracle import measure_oracle, net_oracle, smplx_oracle
    with torch.no_grad():
        feats = net_oracle.hrnet_forward({k[9:]: v for k, v in sd.items() if k.startswith('backbone.')}, x)['concat']
        p = net_oracle.head_forward(sd, feats)[-1]
        body = smplx_oracle.smplx_forward(smplx, p[:, 132:142], smplx_oracle.decode_6d(p[:, :6]),
                                          smplx_oracle.decode_6d(p[:, 6:132]))
    faces = smplx['faces_tensor'].numpy()
    meas = [measure_oracle.measure(body['v_shaped'][b].numpy(), faces, lm) for b in range(x.shape[0])]
    return dict(measurements=meas, vertices=body['vertices'], betas=p[:, 132:142])


def run_reference(args):
    """--impl reference: the CPU port of the reference path on the host cores (rank 0 only)."""
    import torch
    if int(os.environ.get('RANK', '0')) != 0:
        return
    from shapy_b200 import synth
    cores = usable_cores()
    torch.set_num_threads(cores)
    model = synth.build_synthetic_regressor()
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    smplx, lm = synth.make_smplx(), synth.load_landmarks()
    # One warm-up pass over the sample, then K timed passes.  The sample is `--ref-sample` bodies (8, the same as the
    # in-line cpu_baseline leg of the GPU arm): the oneDNN / ATen convolutions of this port run at their best per-body
    # rate there (21-25 bodies/s on the 16 host cores; 64 bodies per pass: 9.7 bodies/s, profiles/
    # r02_bench_reference_arm_sample64.json), shrunk only if K passes would not fit in two minutes.
    x1 = torch.randn(1, 3, 224, 224, generator=torch.Generator().manual_seed(0))
    t0 = time.perf_counter()
    cpu_reference_step(sd, smplx, lm, x1)
    t1 = time.perf_counter() - t0
    sample = int(max(1, min(args.batch, args.ref_sample, 120.0 / max(args.steps, 1) / max(t1, 1e-3))))
    x = torch.randn(sample, 3, 224, 224, generator=torch.Generator().manual_seed(0))
    cpu_reference_step(sd, smplx, lm, x)                                     # warm-up pass at the timed sample size
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = cpu_reference_step(sd, smplx, lm, x)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        out['measurements'] = {k: torch.tensor([m[k] for m in out['measurements']]) for k in out['measurements'][0]}
        dump_outputs(output_arrays(out), sample, args.dump_outputs)
    v = sample / dt
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'bodies/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': 1, 'ms_per_step': dt * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'configs[2]: full SHAPY_A regressor, 224x224, CPU port of the reference path '
                                   '(oracle/: the same ATen / oneDNN kernels the reference modules call)',
                       'sample': f'{sample} bodies per step (per-body rate of the same workload; the GPU arm runs 64 per '
                                 f'step), 1 warm-up pass'},
            'cpu_baseline': {'value': v, 'unit': 'bodies/s', 'cores': cores, 'kind': 'port',
                             'sample': f'{sample} images per step x {args.steps} steps (HRNet+head+SMPL-X+measurements)'},
            'e2e': {'value': v, 'unit': 'bodies/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours')
    ap.add_argument('--batch', type=int, default=64, help='bodies per GPU')
    ap.add_argument('--mode', type=int, default=1, help='1 = split-fp16 parity mode (1e-4), 0 = plain fp16 (config 2)')
    ap.add_argument('--ref-sample', type=int, default=8)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from shapy_b200 import _lib, synth
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (there is no CPU fallback)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps
    B = args.batch

    model = synth.build_synthetic_regressor()
    model.backbone.precision_mode = args.mode
    sd_cpu = {k: v.clone() for k, v in model.state_dict().items()} if rank == 0 else None
    model = model.to(dev).eval()
    L = _lib.lib()
    g = torch.Generator().manual_seed(1000 + rank)
    x_host = torch.randn(B, 3, 224, 224, generator=g).pin_memory()
    x_dev = x_host.to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    last = {}

    def step_resident():
        with torch.no_grad():
            out = model(x_dev)
        if args.dump_outputs:
            last['out'] = out
        return out

    def timed(fn, k, pre=None):
        """Sum of per-step device times (CUDA events on the launching stream), L2 flushed before each step."""
        evs = []
        barrier()
        for _ in range(k):
            flush.zero_()
            if pre:
                pre()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            evs.append((a, b))
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(W):
        step_resident()
    torch.cuda.synchronize()
    n0 = L.shapy_launch_count()
    step_resident()
    torch.cuda.synchronize()
    launches_per_step = L.shapy_launch_count() - n0

    with ClockSampler(local_rank) as clk:
        total_ms = timed(step_resident, K)
    clocks = clk.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(output_arrays(last.pop('out')), B, args.dump_outputs)
    ms_per_step = total_ms / K
    value = world * B / (ms_per_step * 1e-3)

    # ---------------------------------------------------------------- end-to-end with host buffers
    # Every rank serves its own stream of batches from its own pinned host buffers through the public serving loop
    # (shapy_b200.pipeline.HostPipeline): H2D of batch i+1 and D2H of batch i-1 overlap the forward of batch i on
    # separate streams; the bodies are independent, so there is no data-path collective.  All K batches (copies,
    # forwards, the L2 flush before each forward) sit inside ONE timed interval per rank; max over ranks.
    from shapy_b200.pipeline import HostPipeline
    from shapy_b200.preprocess import InputStage
    per = B
    # the serving input: uint8 images in pinned host memory (what a decoder hands over) + the crop-descriptor table;
    # crop / resize / normalisation run on the GPU inside the timed region (shapy_preprocess_forward)
    stage = InputStage(dev, size=224)
    u8_host = torch.randint(0, 256, (per, 224, 224, 3), dtype=torch.uint8, generator=g).pin_memory()
    desc_host = stage.uniform_table(per, 224, 224)
    outs2 = [{'vertices': torch.empty(per, 10475, 3).pin_memory(), 'betas': torch.empty(per, 10).pin_memory(),
              'measurements': torch.empty(per, 5).pin_memory()} for _ in range(2)]

    # one pipeline for the whole run, as a serving loop has: building it inside the timed region put its staging-buffer
    # cudaMallocs there (new copy streams = new allocator pools), which with NCCL's peer mappings cost ~30 ms at N = 4
    pipe = HostPipeline(model, dev, input_stage=stage)

    def run_e2e(k):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(k):
            pipe.submit_u8(u8_host, desc_host, outs2[i % 2], between=flush.zero_)
        pipe.drain()
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    run_e2e(W)
    e2e_ms = run_e2e(K) / K
    e2e_mode = ('pipelined per rank: H2D of uint8 images + crop descriptors / on-GPU crop+normalise + forward / D2H on three '
                'streams, K batches in one timed interval (L2 flush included), max over ranks')
    e2e_value = world * B / (e2e_ms * 1e-3)
    h2d = world * (per * 224 * 224 * 3 + desc_host.numel())
    d2h = world * per * (10475 * 3 + 10 + 5) * 4

    # ---------------------------------------------------------------- configs[4]: rank-0 batch, NCCL scatter / gather
    cfg5 = None
    if world > 1:
        from shapy_b200 import dist as sdist
        full_u8 = torch.randint(0, 256, (world * per, 224, 224, 3), dtype=torch.uint8, generator=g).to(dev) if rank == 0 else None

        def step_cfg5():
            return sdist.sharded_forward_u8(model, stage, full_u8, per, 224, 224, device=dev)
        for _ in range(W):
            step_cfg5()
        c5_ms = timed(step_cfg5, K) / K
        cfg5 = {'value': world * per / (c5_ms * 1e-3), 'unit': 'bodies/s', 'ms_per_batch': c5_ms, 'batch': world * per,
                'scatter_bytes': (world - 1) * per * 224 * 224 * 3, 'gather_bytes': (world - 1) * per * (10475 * 3 + 10 + 5) * 4,
                'path': 'rank 0 holds the uint8 batch in HBM -> dist.scatter (NCCL) -> shapy_preprocess_forward -> forward -> '
                        'dist.gather of vertices / betas / measurements to rank 0; scatter, compute and gather run back to '
                        'back on one stream (no overlap), device-timed per batch, max over ranks',
                'limiter': 'the forward itself: rank-0 egress + ingress are < 3 % of the batch time at these sizes'}

    # ---------------------------------------------------------------- per-stage device times (rank 0, N = 1 view)
    line = None
    if True:
        pk = peaks()
        bb = model.backbone

        def hr():
            with torch.no_grad():
                return bb(x_dev)['concat']
        hr_ms = timed(hr, max(5, K // 2)) / max(5, K // 2)
        conv_tf = B * CONV_GFLOP_PER_IMAGE_224 * 1e9 / (hr_ms * 1e-3) / 1e12
        from shapy_b200 import ops
        packed = model.model.packed(dev)
        betas = torch.randn(B, 10, device=dev)
        rot = ops.decode_rot6d((torch.randn(B, 132, device=dev) * 0.3 + synth.mean_params()[:132].to(dev)))

        def lbs():
            return ops.smplx_forward(packed, betas, rot)
        for _ in range(3):
            lbs()
        lbs_ms = timed(lbs, 20) / 20
        lbs_gbs = (LBS_CONST_BYTES + B * LBS_BODY_BYTES) / (lbs_ms * 1e-3) / 1e9
        b4096 = torch.randn(4096, 10, device=dev).clamp(-3, 3)

        def shp():
            return ops.smplx_forward_shape(packed, b4096)
        for _ in range(3):
            shp()
        shp_ms = timed(shp, 20) / 20
        shp_gbs = (SHAPE_CONST_BYTES + 4096 * SHAPE_BODY_BYTES) / (shp_ms * 1e-3) / 1e9
        vs4096 = shp()
        faces = model.model.faces_i32
        lmk = model.body_measurements.landmarks()

        def meas():
            return ops.measure(lmk, v_shaped=vs4096, faces_i32=faces)
        for _ in range(2):
            meas()
        meas_ms = timed(meas, 5) / 5
        meas_gbs = (4096 * 125700 + faces.numel() * 4) / (meas_ms * 1e-3) / 1e9      # vertices once + the face table
        # BASELINE configs[1]: HRNet-W48 only, plain fp16 operands, B = 32 (a second plan of the same weights)
        import copy
        bb16 = copy.deepcopy(bb)
        bb16.precision_mode = 0
        bb16.invalidate()
        x32 = x_dev[:32].contiguous() if B >= 32 else torch.randn(32, 3, 224, 224, device=dev)

        def hr16():
            with torch.no_grad():
                return bb16(x32)['concat']
        for _ in range(3):
            hr16()
        hr16_ms = timed(hr16, 10) / 10
        c2_tf = 32 * CONV_GFLOP_PER_IMAGE_224 * 1e9 / (hr16_ms * 1e-3) / 1e12
        del bb16

    if rank == 0:
        cpu, selfcheck = None, None
        if world == 1 and not args.no_cpu_baseline:
            # One leg, two uses: (1) self-check -- the oracle's outputs for `n` of the step's images against the GPU outputs
            # of the same images (taken from the full B = 64 forward), (2) cpu_baseline -- the same oracle passes timed
            # with the procedure of the --impl reference arm: one warm-up pass, then `reps` timed passes.
            cores = usable_cores()
            torch.set_num_threads(cores)
            smplx, lm = synth.make_smplx(), synth.load_landmarks()
            n = min(args.ref_sample, B)
            rows = [int(round(i * (B - 1) / max(n - 1, 1))) for i in range(n)]
            xs = x_host[rows].clone()
            ref = cpu_reference_step(sd_cpu, smplx, lm, xs)                      # warm-up pass + self-check data
            with torch.no_grad():
                o = model(x_dev)
            st = o[o['stage_keys'][-1]]

            def rel(a, b):
                return float((a.double().cpu() - b.double()).abs().max() / b.double().abs().max())
            errs = {'vertices': rel(st['vertices'][rows], ref['vertices']), 'betas': rel(st['betas'][rows], ref['betas'])}
            for name in ('mass', 'height', 'chest', 'waist', 'hips'):
                r = torch.tensor([m[name] for m in ref['measurements']], dtype=torch.float64)
                errs[name] = float(((o['measurements'][name][rows].double().cpu() - r).abs() / r.abs()).max())
            selfcheck = {'bodies': n, 'rows': rows, 'max_rel_err': max(errs.values()), 'errors': errs, 'tolerance': 1e-4}
            assert selfcheck['max_rel_err'] < 1e-4, f'bench self-check failed: {errs}'
            reps = 3
            t0 = time.perf_counter()
            for _ in range(reps):
                cpu_reference_step(sd_cpu, smplx, lm, xs)
            dt = (time.perf_counter() - t0) / reps
            cpu = {'value': n / dt, 'unit': 'bodies/s', 'cores': cores, 'kind': 'port',
                   'sample': f'{n} of the {B} images of one step (HRNet+head+SMPL-X+measurements), 1 warm-up pass + {reps} timed '
                             f'passes, {dt:.2f} s per pass'}
        line = {
            'metric': METRIC, 'value': value, 'unit': 'bodies/s', 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32 (split-fp16 hi/lo tensor-core operands, fp32 accumulate)' if args.mode else 'f16',
            'data': 'synthetic',
            'config': {'workload': 'configs[2]: full SHAPY_A regressor (HRNet-W48 + iterative head + fused SMPL-X + '
                                   'measurements), 224x224, batch 64 per GPU', 'batch_per_gpu': B,
                       'l2': 'flushed (256 MB write) before every timed step', 'parallelism': f'dp{world}',
                       'precision_mode': args.mode},
            'e2e': {'value': e2e_value, 'unit': 'bodies/s', 'ms_per_step': e2e_ms, 'mode': e2e_mode, 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h},
            'gpu_launches': int(launches_per_step * K),
            'clocks': clocks,
            'roofline': {'bound': 'tensor', 'achieved': conv_tf, 'peak': pk['tf_sustained'], 'unit': 'TFLOP/s',
                         'frac': conv_tf / pk['tf_sustained'], 'traffic': conv_traffic(B, args.mode),
                         'kernel': 'conv_halo_kernel / conv_umma_kernel (HRNet forward: all 331 convs + fuse + pool, 4 lanes)',
                         'ms': hr_ms, 'mma_flops_factor': 3 if args.mode else 1, 'peak_source': pk['source']},
            'roofline_lbs': {'bound': 'hbm', 'achieved': lbs_gbs, 'peak': pk['hbm'], 'unit': 'GB/s',
                             'frac': lbs_gbs / pk['hbm'], 'ms': lbs_ms, 'traffic': lbs_traffic(B),
                             'kernel': 'smplx_lbs_kernel (fused tcgen05) + smplx_joints_kernel, B=%d posed; achieved counts the '
                                       'algorithmic bytes of SURVEY 8d (all 486 pose-basis rows), traffic is what ncu measured: the '
                                       'rows of identity joints are never read' % B},
            'roofline_shape': {'bound': 'hbm', 'achieved': shp_gbs, 'peak': pk['hbm'], 'unit': 'GB/s',
                               'frac': shp_gbs / pk['hbm'], 'ms': shp_ms, 'kernel': 'smplx_shape_kernel, 4096 bodies (config 4)'},
            'roofline_measure': {'bound': 'hbm', 'achieved': meas_gbs, 'peak': pk['hbm'], 'unit': 'GB/s',
                                 'frac': meas_gbs / pk['hbm'], 'ms': meas_ms, 'bodies_per_s': 4096 / (meas_ms * 1e-3),
                                 'kernel': 'measure_smem_kernel, 4096 bodies (config 4): 125 700 B of vertices per body read once'},
            'config2': {'workload': 'configs[1]: HRNet-W48 backbone only, 224x224, plain fp16 operands, batch 32',
                        'ms': hr16_ms, 'images_per_s': 32 / (hr16_ms * 1e-3),
                        'roofline': {'bound': 'tensor', 'achieved': c2_tf, 'peak': pk['tf_sustained'], 'unit': 'TFLOP/s',
                                     'frac': c2_tf / pk['tf_sustained'], 'mma_flops_factor': 1}},
        }
        if cfg5:
            line['config5'] = cfg5
        if cpu:
            line['cpu_baseline'] = cpu
        if selfcheck:
            line['selfcheck'] = selfcheck
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
