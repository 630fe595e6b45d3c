"""The fused step kernel with many short items per CTA: ring slots and mbarrier parities carry over from item to item, and
2-row items use fewer records than the ring holds.  RISP_FUSED_STEP_ROWS caps the rows per item; it is read once per
process, so the capped runs happen in a child process.  Against the default geometry: the output image bit for bit
(per-pixel work does not depend on the geometry), the loss and the gradients within the tolerances of
tests/test_fused_gpu.py (the summation order does), and every geometry bit-reproducible."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

IDENT = [0.0] * 30
IDENT[6] = IDENT[17] = IDENT[28] = 1.0
SIGS = {'A': (['gain', 'poly10', 'gamma', ('gtm', 4)], [1.1, 0.9, 1.2] + IDENT + [0.55, 0.2, 0.5, 0.8]),
        'D': (['gamma', ('gtm', 4)], [0.55, 0.2, 0.5, 0.8])}
# 2 frames x 8 strips (the last one partial) x 2400 rows: 4-row items are several per CTA at any occupancy
N, H, W = 2, 2400, 1000


def run_steps(out):
    """Two steps per signature on seeded inputs -> npz with y, loss and gradients of each."""
    import torch
    from reconfigisp_b200 import ops
    g = torch.Generator().manual_seed(5)
    raw = torch.rand(N, 1, H, W, generator=g).cuda()
    gt = torch.rand(N, 3, H, W, generator=g).cuda()
    res = {}
    for sig, (st, vals) in SIGS.items():
        chain = ops.Chain(st)
        p = (torch.tensor([vals]) + 0.02 * torch.randn(1, len(vals), generator=g)).cuda()
        step = ops.PipelineStep(N, H, W, 'bilinear', chain, 'cuda')
        for rep in range(2):
            y = torch.empty(N, 3, H, W, device='cuda')
            loss, dp = step(raw, gt, p, y)
            res['%s_y%d' % (sig, rep)] = y.cpu().numpy()
            res['%s_loss%d' % (sig, rep)] = loss.cpu().numpy()
            res['%s_grad%d' % (sig, rep)] = dp.cpu().numpy()
    np.savez(out, **res)


def child(rows, out):
    env = dict(os.environ)
    env.pop('RISP_FUSED_STEP_ROWS', None)
    if rows:
        env['RISP_FUSED_STEP_ROWS'] = str(rows)
    cmd = [sys.executable] + (['-s'] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    return np.load(out)


@pytest.mark.parametrize('rows', [2, 4])
def test_step_many_items_per_cta(tmp_path, rows):
    ref = child(0, tmp_path / 'default.npz')
    cap = child(rows, tmp_path / ('rows%d.npz' % rows))
    for sig in SIGS:
        for r in (ref, cap):      # fixed summation order: bit-reproducible
            assert np.array_equal(r['%s_loss0' % sig], r['%s_loss1' % sig])
            assert np.array_equal(r['%s_grad0' % sig], r['%s_grad1' % sig])
            assert np.array_equal(r['%s_y0' % sig], r['%s_y1' % sig])
        assert np.array_equal(cap['%s_y0' % sig], ref['%s_y0' % sig])
        la, lb = float(cap['%s_loss0' % sig][0]), float(ref['%s_loss0' % sig][0])
        assert abs(la - lb) <= 1e-5 * max(1.0, abs(lb)), (sig, la, lb)
        ga, gb = cap['%s_grad0' % sig].astype(np.float64), ref['%s_grad0' % sig].astype(np.float64)
        assert np.abs(ga - gb).max() <= 1e-6 + 1e-3 * np.abs(gb).max(), (sig, ga, gb)


if __name__ == '__main__':
    sys.path.insert(0, ROOT)
    run_steps(sys.argv[1])
