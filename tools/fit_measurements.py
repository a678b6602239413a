#!/usr/bin/env python
"""Fit SMPL-X shape coefficients to target measurements on the GPU: a headless port of the reference example
mesh-mesh-intersection/examples/fit_measurements.py, for a batch of bodies.

    python tools/fit_measurements.py --synthetic --height 1.80 --chest 1.00 --batch 64
    python tools/fit_measurements.py --model-folder <dir with SMPLX_NEUTRAL.npz> --height 1.80 --mass 80
    python tools/fit_measurements.py --synthetic --time --batches 64 4096 --out profiles/<name>.json

Same targets (a negative target is not fitted), loss weights (height 100, mass 1, chest 2000, waist 1000, hips 1000)
and `betas_weight` prior as the reference.  The reference steps a second-order TrustRegion optimizer
(torchtrustncg, which differentiates the gradient); the backward here is first-order only, so this uses
torch.optim.LBFGS.  Each body starts from its own seeded betas.

--time times, at each batch size, with the L2 cache overwritten before every timed call: the measurement forward,
its backward, the shape-blend backward and one full fitting step (shape blend + measurements + loss + backward), and
reports the backward's achieved HBM bandwidth from its algorithmic bytes (each body's vertices read once, its
gradient written once) against the B200's 7.7 TB/s, with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from shapy_b200 import ops, synth  # noqa: E402
from shapy_b200.body_measurements import BodyMeasurements  # noqa: E402
from shapy_b200.human_shape.models.body_models.body_models import SMPLX  # noqa: E402

NAMES = ('mass', 'height', 'chest', 'waist', 'hips')
WEIGHTS = dict(height=100.0, mass=1.0, chest=2000.0, waist=1000.0, hips=1000.0)
HBM_PEAK = 7.7e12


def build(args):
    if args.synthetic:
        model = SMPLX(data_struct=synth.make_smplx())
    else:
        model = SMPLX(model_folder=args.model_folder, gender=args.gender, betas={'num': args.num_betas})
    model = model.cuda()
    if args.meas_definition_path and args.meas_vertices_path:
        cfg = dict(meas_definition_path=args.meas_definition_path, meas_vertices_path=args.meas_vertices_path)
    else:
        cfg = dict(landmarks=synth.load_landmarks())
    return model, BodyMeasurements(cfg).cuda()


def fit(model, meas, args):
    dev = torch.device('cuda')
    nb = model.packed(dev).NB
    gen = torch.Generator().manual_seed(args.seed)
    betas = (torch.randn(args.batch, nb, generator=gen) * args.init_std).to(dev).requires_grad_(True)
    targets = {k: getattr(args, k) for k in NAMES}
    weights = {k: (WEIGHTS[k] if targets[k] > 0 else 0.0) for k in NAMES}
    f = model.faces_i32
    opt = torch.optim.LBFGS([betas], lr=1.0, max_iter=args.max_iter, history_size=20, line_search_fn='strong_wolfe')

    def losses():
        m = meas.forward_vertices(model.forward_shape(betas)['v_shaped'], f)['measurements']
        out = {k: weights[k] * (targets[k] - m[k]['tensor']).pow(2).sum() for k in NAMES if weights[k] > 1e-3}
        out['betas'] = args.betas_weight * betas.pow(2).sum()
        return out, m

    def closure():
        opt.zero_grad()
        loss = sum(losses()[0].values())
        loss.backward()
        return loss
    for n in range(args.num_iterations):
        opt.step(closure)
        if n % args.summary_steps == 0 or n == args.num_iterations - 1:
            with torch.no_grad():
                ls, m = losses()
            est = ', '.join(f'{k} {float(m[k]["tensor"].mean()):.4f}' for k in NAMES)
            print(f'[{n:04d}] loss {float(sum(ls.values())):.6f} | batch mean: {est} | targets '
                  + ', '.join(f'{k} {targets[k]}' for k in NAMES if weights[k] > 0))
    return betas.detach()


def _time(fn, flush, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        start.record()
        fn()
        end.record()
        end.synchronize()
        ts.append(start.elapsed_time(end) * 1e-3)
    ts.sort()
    return ts[len(ts) // 2]


def timing(model, meas, args):
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    card = dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip().splitlines()[:1])
    dev = torch.device('cuda')
    packed = model.packed(dev)
    lmk = meas.landmarks()
    f = model.faces_i32
    flush = torch.empty(512 * 2 ** 20, dtype=torch.uint8, device=dev)      # > the 126 MB L2
    rows = []
    for B in args.batches:
        betas = (torch.randn(B, packed.NB, generator=torch.Generator().manual_seed(B)) * args.init_std).to(dev)
        vs = ops.smplx_forward_shape(packed, betas)
        g = torch.ones(B, 5, device=dev)
        gv = torch.randn(B, packed.V, 3, device=dev)
        t_fwd = _time(lambda: ops.measure(lmk, v_shaped=vs, faces_i32=f), flush, args.reps)
        t_bwd = _time(lambda: ops.measure_backward(lmk, g, v_shaped=vs, faces_i32=f), flush, args.reps)
        t_shape_bwd = _time(lambda: ops.smplx_shape_backward(packed, gv), flush, args.reps)
        b = betas.clone().requires_grad_(True)
        w = torch.tensor([WEIGHTS[k] for k in NAMES], device=dev)
        target = ops.measure(lmk, v_shaped=vs, faces_i32=f) * 1.01

        def step():
            b.grad = None
            m = meas.forward_vertices(model.forward_shape(b)['v_shaped'], f)['measurements']
            est = torch.stack([m[k]['tensor'] for k in NAMES], 1)
            ((target - est).pow(2) * w).sum().backward()
        t_step = _time(step, flush, args.reps)
        nbytes = B * packed.V * 3 * 4 * 2
        rows.append(dict(B=B, measure_forward_s=t_fwd, measure_backward_s=t_bwd, shape_backward_s=t_shape_bwd,
                         fit_step_s=t_step, backward_over_forward=t_bwd / t_fwd,
                         backward_algorithmic_bytes=nbytes, backward_hbm_TBps=nbytes / t_bwd / 1e12,
                         backward_hbm_fraction=nbytes / t_bwd / HBM_PEAK))
        print(json.dumps(rows[-1]))
    return dict(card=card, l2_flushed_before_each_call=True, reps=args.reps, statistic='median', rows=rows)


def main():
    p = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    src = p.add_mutually_exclusive_group(required=True)
    src.add_argument('--synthetic', action='store_true', help='seeded synthetic SMPL-X of shapy_b200.synth')
    src.add_argument('--model-folder', help='folder with SMPLX_<GENDER>.npz')
    p.add_argument('--gender', default='neutral')
    p.add_argument('--num-betas', type=int, default=10)
    p.add_argument('--meas-definition-path', default='')
    p.add_argument('--meas-vertices-path', default='')
    for k, d in (('height', 1.80), ('mass', -1.0), ('chest', -1.0), ('waist', -1.0), ('hips', -1.0)):
        p.add_argument(f'--{k}', type=float, default=d, help='target (negative: not fitted)')
    p.add_argument('--betas-weight', type=float, default=0.0)
    p.add_argument('--batch', type=int, default=64)
    p.add_argument('--init-std', type=float, default=0.5)
    p.add_argument('--seed', type=int, default=0)
    p.add_argument('--num-iterations', type=int, default=50)
    p.add_argument('--max-iter', type=int, default=20, help='LBFGS iterations per step')
    p.add_argument('--summary-steps', type=int, default=10)
    p.add_argument('--time', action='store_true')
    p.add_argument('--batches', type=int, nargs='+', default=[64, 4096])
    p.add_argument('--reps', type=int, default=20)
    p.add_argument('--out', default='')
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('fit_measurements: needs a CUDA device')
    model, meas = build(args)
    if args.time:
        res = timing(model, meas, args)
        if args.out:
            with open(args.out, 'w') as fh:
                json.dump(res, fh, indent=1)
        return
    fit(model, meas, args)


if __name__ == '__main__':
    main()
