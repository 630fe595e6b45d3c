"""The tuning step (`risp_pipeline_mse_step`) and its upstream-gradient backward (`risp_pipeline_bwd`) on every kernel route
the dispatch can pick, against the float64 oracle (`oracle.isp_oracle.pixel_chain`):

* the packed kernel (`fused_kernel`): signatures A-D with a shared row or at most 8 per-image rows;
* the interpreter kernel (`pipeline_kernel`): generic chains without (BIG = false) and with (BIG = true) a poly10 / ccm
  stage, and the A-D instantiations when more than 8 frames carry their own rows;
* the finalisers: `finalize_rows_kernel` (at most 64 frames) and `finalize_kernel` (more than 64 frames, or a
  demosaic-only step with no parameters).

`test_every_route_runs_the_kernel_it_claims` profiles one call per route, so a change of the dispatch cannot move a case
off the route it is meant to cover without a failure here.

Tolerances against the oracle are those of tests/test_fused_gpu.py: outputs max-abs 1e-4, loss 1e-5 relative, gradients
2e-3 of the largest entry -- taken per parameter row (one row per frame with per-image rows), so that one wrong row of a
table cannot hide behind a larger one.  Near-black pixels need no mask: the oracle runs in float64, where x^gamma of a
near-black input is exact to far below the tolerance, and the kernels' own fp32 error there stays within it."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
pytestmark = pytest.mark.gpu

from oracle import isp_oracle as O   # noqa: E402  (the checker)

IDENT = [0.0] * 30
IDENT[6] = IDENT[17] = IDENT[28] = 1.0
KINDS = ['nearest', 'bilinear', 'malvar']
DM = {'nearest': O.demosaic_nearest, 'bilinear': O.demosaic_bilinear, 'malvar': lambda r: O.demosaic_laplacian(r, 1.0)}
SIGS = {
    'A': ['gain', 'poly10', 'gamma', ('gtm', 4)],
    'B': ['gamma', 'poly10', 'gain'],
    'C': ['gamma', 'poly10'],
    'D': ['gamma', ('gtm', 4)],
}
GENERIC = {                                        # no packed signature, no poly10 / ccm: pipeline_kernel<.., 0, false>
    'gtm5_clip': ['gamma', ('gtm', 5), 'gain_clip'],
    'gain_gtm3': ['gain', ('gtm', 3)],
    'six': ['gamma', 'gain', 'gain_clip', ('gtm', 2), 'gamma', 'gain'],
}
GENERIC_BIG = {                                    # one poly10 / ccm stage: pipeline_kernel<.., 0, true>
    'classical': ['gain', 'poly10', 'gamma'],      # the sRGB tail 11_13_01
    'ccm': ['gain', 'ccm', 'gamma'],
    'six_poly': ['gain', 'gamma', 'poly10', ('gtm', 3), 'gain_clip', 'gamma'],
}
CHAINS = dict(GENERIC, **GENERIC_BIG)
# a partial last strip (remnant 4 columns), the smallest frame, several strips (remnant 8), a remnant of 36 columns
SHAPES = [(2, 12, 132), (1, 6, 8), (2, 50, 520), (2, 10, 164)]

TOL_Y, TOL_LOSS, TOL_GRAD = 1e-4, 1e-5, 2e-3
# Two fp32 routes on the same inputs (packed kernel against interpreter kernel, a shared row against the same row repeated):
# both evaluate the same per-pixel formulas in fp32, so each pixel's gradient term differs by a few ulp (approximate
# lg2 / ex2, FMA contraction, the packed kernel's folded gain and hinge-sum tone-curve gradient), and the sums differ in
# order.  Each route accumulates at most ~2^10 terms in one register before a tree reduction, so the reordering error of a
# sum is at most ~2^10 * 2^-24 ~ 6e-5 of the sum of the terms' magnitudes; the terms' signs are random, so in practice it
# is the square root of that count, ~2e-6.  1e-4 of the row's largest gradient (20x tighter than the oracle bound) leaves
# headroom for the hinge-sum cancellation while still failing on a wrong slot, scale or mask.  The loss is one sum of
# squares of like sign: 1e-6 relative.
TIGHT_GRAD, TIGHT_LOSS = 1e-4, 1e-6
# dy = 2 (y - gt) / numel fed to the backward must reproduce the step's own gradients: the same kernel, the same summation
# order, only the place where the 2 / numel scale is applied differs (one rounding per term)
SELF_GRAD = 1e-5


@pytest.fixture(scope='module')
def ops():
    import reconfigisp_b200.ops as ops
    return ops


# ---- inputs, parameters, oracle -------------------------------------------------------------------------------------
def inputs(N, H, W, seed):
    """raw in [0, 1.05] with 5 % exact 0 / 1 samples and a near-black corner (1e-4 of the signal); gt uniform in [0, 1]."""
    g = torch.Generator().manual_seed(seed)
    raw = torch.rand(N, 1, H, W, generator=g) * 1.05
    pick = torch.rand(N, 1, H, W, generator=g)
    raw = torch.where(pick < 0.05, (pick < 0.025).float(), raw)
    raw[:, :, :4, :16] *= 1e-4
    raw.view(-1)[:3] = torch.tensor([0., 1., 0.5])
    gt = torch.rand(N, 3, H, W, generator=g)
    return raw, gt, g


def param_row(st, g, knots=None):
    """One kernel-level parameter row.  gain_clip's first gain is exactly 1, so tone-curve outputs of exactly 1 reach its
    inclusive clamp bound; the other gains push bright pixels past it."""
    vals, second_gamma = [], False
    for s in st:
        name, iarg = (s, 0) if isinstance(s, str) else s
        if name == 'gain':
            vals += [1.1, 0.9, 1.2]
        elif name == 'gain_clip':
            vals += [1.0, 0.9, 1.6]
        elif name == 'poly10':
            vals += (torch.tensor(IDENT) + torch.randn(30, generator=g) * 0.03).tolist()
        elif name == 'gamma':
            vals += [0.8 if second_gamma else 0.55]
            second_gamma = True
        elif name == 'gtm':
            vals += list(knots) if knots is not None else torch.linspace(0.15, 0.85, iarg - 1).tolist()
        elif name == 'ccm':
            vals += [0.9, 0.05, 0.05, 0.1, 0.8, 0.1, 0.0, 0.1, 1.3]
    return torch.tensor([vals])


def per_image(row, N):
    return row.repeat(N, 1) * (1 + 0.01 * (torch.arange(N).view(N, 1) % 16))


def oracle_step(raw, gt, kind, st, rows):
    po = rows.double().requires_grad_()
    yo = O.pixel_chain(DM[kind](raw.double()), st, po)
    lo = O.mse(yo, gt.double())
    dpo, = torch.autograd.grad(lo, po)
    return yo.detach(), float(lo.detach()), dpo


def oracle_bwd(raw, dys, kind, st, rows):
    """-> [(d y / d params)^T dy for dy in dys]"""
    po = rows.double().requires_grad_()
    yo = O.pixel_chain(DM[kind](raw.double()), st, po)
    return [torch.autograd.grad(yo, po, dy.double(), retain_graph=True)[0] for dy in dys]


def rowclose(a, b, rtol=TOL_GRAD, atol=1e-6):
    """max |a - b| <= atol + rtol * max |b| in every parameter row."""
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    assert a.shape == b.shape, (a.shape, b.shape)
    for r in range(b.shape[0]):
        err, lim = float((a[r] - b[r]).abs().max()), atol + rtol * float(b[r].abs().max())
        assert err <= lim, ('row', r, err, lim)


def lossclose(a, b, rtol=TOL_LOSS):
    assert abs(float(a) - float(b)) <= rtol * abs(float(b)), (float(a), float(b))


# ---- the entry points ---------------------------------------------------------------------------------------------
def step(ops, raw, gt, kind, chain, rows):
    """-> y, loss, dparams of one MSE tuning step (y written by the step kernel)."""
    N, _, H, W = raw.shape
    y = torch.empty(N, 3, H, W, device='cuda')
    shared = rows is None or rows.shape[0] == 1
    loss, dp = ops.PipelineStep(N, H, W, kind, chain, 'cuda', shared_row=shared)(raw, gt, rows, y)
    return y, loss.clone(), dp.clone()


def bwd(ops, raw, dy, kind, chain, rows):
    """dparams = (d y / d params)^T dy through `risp_pipeline_bwd`, as `_FusedHeadFn.backward` calls it."""
    from reconfigisp_b200 import _lib as L
    N, _, H, W = raw.shape
    tab, stride = ops._param_table(rows, N, chain.P)
    dpar = torch.empty((1 if stride == 0 else N, chain.P), device='cuda')
    ws = L.workspace(L.size('risp_pipeline_step_workspace', N, H, W, chain.P), 'cuda')
    L.call('risp_pipeline_bwd', L.ptr(raw), L.ptr(dy.contiguous()), L.ptr(dpar), N, H, W, ops.DM[kind], 1.0, *chain.desc(),
           L.ptr(tab), stride, chain.P, L.ptr(ws), ws.numel() * 4, L.stream())
    return dpar


def check_step(ops, raw, gt, kind, st, rows):
    """The step against the oracle; returns the device results."""
    yo, lo, dpo = oracle_step(raw, gt, kind, st, rows)
    y, loss, dp = step(ops, raw.cuda(), gt.cuda(), kind, ops.Chain(st), rows.cuda())
    assert float((y.cpu().double() - yo).abs().max()) <= TOL_Y
    lossclose(loss, lo)
    rowclose(dp, dpo)
    return y, loss, dp


def last_strip_only(dy):
    W = dy.shape[-1]
    out = torch.zeros_like(dy)
    c = (W - 1) // 128 * 128
    out[..., c:] = dy[..., c:]
    return out


def check_bwd(ops, raw, gt, kind, st, rows):
    """risp_pipeline_bwd against autograd of the oracle for a random dy and a dy that is zero outside the last 128-column
    strip, and the self-check dy = 2 (y - gt) / numel == the step's own gradients."""
    N, _, H, W = raw.shape
    g = torch.Generator().manual_seed(N * H * W + len(st))
    chain = ops.Chain(st)
    dy = torch.randn(N, 3, H, W, generator=g)
    dys = (dy, last_strip_only(dy))
    for d, ref in zip(dys, oracle_bwd(raw, dys, kind, st, rows)):
        rowclose(bwd(ops, raw.cuda(), d.cuda(), kind, chain, rows.cuda()), ref)
    y, _, dp = step(ops, raw.cuda(), gt.cuda(), kind, chain, rows.cuda())
    dself = bwd(ops, raw.cuda(), 2 * (y - gt.cuda()) / y.numel(), kind, chain, rows.cuda())
    rowclose(dself, dp, rtol=SELF_GRAD, atol=0)


# ---- the step ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('shape', SHAPES)
@pytest.mark.parametrize('name', sorted(CHAINS))
@pytest.mark.parametrize('kind', KINDS)
def test_generic_step_vs_oracle(ops, kind, name, shape):
    N, H, W = shape
    st = CHAINS[name]
    assert not ops.fused_chain_supported(ops.Chain(st))
    raw, gt, g = inputs(N, H, W, sum(map(ord, kind + name)) + H * W)
    row = param_row(st, g)
    check_step(ops, raw, gt, kind, st, row)
    if N > 1:
        check_step(ops, raw, gt, kind, st, per_image(row, N))


@pytest.mark.parametrize('shape', [(9, 10, 164), (12, 8, 132)])
@pytest.mark.parametrize('sig', sorted(SIGS))
@pytest.mark.parametrize('kind', KINDS)
def test_signature_step_many_rows_vs_oracle(ops, kind, sig, shape):
    """More per-image rows than the packed kernel's constant slot holds (8): the A-D instantiations of pipeline_kernel."""
    N, H, W = shape
    st = SIGS[sig]
    raw, gt, g = inputs(N, H, W, sum(map(ord, kind + sig)) + N)
    check_step(ops, raw, gt, kind, st, per_image(param_row(st, g), N))


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('st, knots', [(['gain', ('gtm', 3)], (-0.15, 1.2)),
                                       (['gamma', ('gtm', 5), 'gain_clip'], (-0.2, 0.3, 0.9, 1.3))],
                         ids=['gtm3', 'gtm5'])
def test_generic_step_out_of_range_knots(ops, kind, st, knots):
    """Tone-curve knots outside [0,1] (the final clamp is active: the CHECK_RANGE branch of gtm_bwd_px), in a table whose
    first row is in range and whose second row is not: the branch is taken per frame."""
    N, H, W = 2, 20, 136
    raw, gt, g = inputs(N, H, W, 7 + len(knots))
    bad = param_row(st, g, knots)
    good = param_row(st, g)
    check_step(ops, raw, gt, kind, st, bad)
    check_step(ops, raw, gt, kind, st, torch.cat([good, bad]))


@pytest.mark.parametrize('name', ['classical', 'six_poly', 'gtm5_clip', 'six'])
def test_generic_step_saturated_frames(ops, name):
    """Frames of exact 0 / 1 samples, unit gains and the identity polynomial: stage outputs land exactly on the clamp bounds,
    where every mask is inclusive, and the tone curves see x == 1 (the pass-through pixel)."""
    st = CHAINS[name]
    N, H, W = 2, 16, 136
    g = torch.Generator().manual_seed(9)
    raw = (torch.rand(N, 1, H, W, generator=g) > 0.5).float()
    gt = torch.rand(N, 3, H, W, generator=g)
    row = param_row(st, g)
    chain = ops.Chain(st)
    for s, o in zip(chain.names, chain.offsets):
        if s in ('gain', 'gain_clip'):
            row[0, o:o + 3] = 1.0
        elif s == 'poly10':
            row[0, o:o + 30] = torch.tensor(IDENT)
    check_step(ops, raw, gt, 'nearest', st, row)


# ---- the backward with an upstream gradient --------------------------------------------------------------------------
PACKED_SHAPES = [(2, 12, 256), (2, 12, 132), (2, 10, 164)]    # whole strips; narrow remnants of 4 and 36 columns


@pytest.mark.parametrize('shape', PACKED_SHAPES)
@pytest.mark.parametrize('sig', sorted(SIGS))
@pytest.mark.parametrize('kind', KINDS)
def test_packed_bwd_vs_oracle(ops, kind, sig, shape):
    N, H, W = shape
    st = SIGS[sig]
    assert ops.fused_chain_supported(ops.Chain(st))
    raw, gt, g = inputs(N, H, W, sum(map(ord, kind + sig)) + W)
    row = param_row(st, g)
    check_bwd(ops, raw, gt, kind, st, row)
    check_bwd(ops, raw, gt, kind, st, per_image(row, N))


@pytest.mark.parametrize('shape', [(2, 12, 132), (2, 50, 520)])
@pytest.mark.parametrize('name', sorted(CHAINS))
@pytest.mark.parametrize('kind', KINDS)
def test_generic_bwd_vs_oracle(ops, kind, name, shape):
    N, H, W = shape
    st = CHAINS[name]
    raw, gt, g = inputs(N, H, W, sum(map(ord, kind + name)) + W)
    row = param_row(st, g)
    check_bwd(ops, raw, gt, kind, st, row)
    check_bwd(ops, raw, gt, kind, st, per_image(row, N))


# ---- the finalisers ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['A', 'classical', 'gtm5_clip'])
def test_finalisers_at_64_and_65_frames(ops, name):
    """65 frames: `finalize_kernel` for the loss and the gradients, shared row (summed over frames) and per-image rows (one
    output row per frame).  64 frames with per-image rows: the R <= 64 edge of `finalize_rows_kernel`."""
    st = SIGS.get(name) or CHAINS[name]
    for N, shared in ((65, True), (65, False), (64, False)):
        raw, gt, g = inputs(N, 6, 8, N + len(name))
        row = param_row(st, g)
        check_step(ops, raw, gt, 'bilinear', st, row if shared else per_image(row, N))
        if not shared:
            check_bwd(ops, raw, gt, 'malvar', st, per_image(row, N))


@pytest.mark.parametrize('N', [3, 65])
@pytest.mark.parametrize('kind', KINDS)
def test_demosaic_only_step(ops, kind, N):
    """No parameters (P == 0): the step is the loss of the demosaic alone, reduced by `finalize_kernel`."""
    raw, gt, _ = inputs(N, 10, 132, N)
    y, loss, _ = step(ops, raw.cuda(), gt.cuda(), kind, ops.Chain([]), None)
    yo = DM[kind](raw.double())
    assert float((y.cpu().double() - yo).abs().max()) <= TOL_Y
    lossclose(loss, O.mse(yo, gt.double()))


# ---- agreement between routes ------------------------------------------------------------------------------------------
CROSS_SHAPE = (3, 20, 164)


def cross_cases(ops):
    """-> {key: array} of every signature x demosaic: step (loss, dparams) with a shared and with per-image rows, and the
    backward of a fixed dy.  Every result is computed twice and must be bit-identical."""
    N, H, W = CROSS_SHAPE
    res = {}
    for sig, st in sorted(SIGS.items()):
        chain = ops.Chain(st)
        for kind in KINDS:
            raw, gt, g = inputs(N, H, W, sum(map(ord, kind + sig)))
            raw, gt = raw.cuda(), gt.cuda()
            row = param_row(st, g)
            dy = torch.randn(N, 3, H, W, generator=g).cuda()
            for mode, rows in (('shared', row), ('rows', per_image(row, N))):
                rows = rows.cuda()
                for rep in range(2):
                    _, loss, dp = step(ops, raw, gt, kind, chain, rows)
                    db = bwd(ops, raw, dy, kind, chain, rows)
                    out = {'loss': loss, 'dp': dp, 'bwd': db}
                    for k, v in out.items():
                        key = '%s_%s_%s_%s' % (sig, kind, mode, k)
                        v = v.cpu().numpy()
                        if rep == 0:
                            res[key] = v
                        else:
                            assert np.array_equal(v, res[key]), ('not bit-reproducible', key)
    return res


def child_main(out):
    """Child process with RISP_FUSED=0 (read once per process): every chain on pipeline_kernel."""
    import reconfigisp_b200.ops as ops
    raw, gt, g = inputs(2, 12, 132, 1)
    st = SIGS['A']
    fams = families(kernels_of(lambda: step(ops, raw.cuda(), gt.cuda(), 'bilinear', ops.Chain(st), param_row(st, g).cuda())))
    assert 'pipeline_kernel' in fams and 'fused_kernel' not in fams, fams
    np.savez(out, **cross_cases(ops))


def run_child(env_update, out):
    env = dict(os.environ)
    env.pop('RISP_FUSED', None)
    env.update(env_update)
    cmd = [sys.executable] + (['-s'] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    return np.load(out)


def test_packed_kernel_equals_interpreter_kernel(ops, tmp_path):
    """Signatures A-D: the packed kernel (this process) against pipeline_kernel (a child with RISP_FUSED=0), step and
    backward, shared and per-image rows, within the bound derived at TIGHT_GRAD; both routes bit-reproducible."""
    packed = cross_cases(ops)
    interp = run_child({'RISP_FUSED': '0'}, tmp_path / 'interp.npz')
    assert sorted(interp.files) == sorted(packed)
    for k, v in packed.items():
        if k.endswith('_loss'):
            lossclose(v[0], interp[k][0], TIGHT_LOSS)
        else:
            rowclose(torch.from_numpy(v), torch.from_numpy(interp[k]), TIGHT_GRAD, atol=0)


@pytest.mark.parametrize('N', [4, 9])
@pytest.mark.parametrize('name', sorted(SIGS) + ['classical', 'six'])
def test_shared_row_equals_repeated_rows(ops, name, N):
    """One shared row against the same row repeated N times: the same loss, and the per-image gradients sum to the shared
    one.  With signatures A-D and N = 9 the two run on different kernels (packed / pipeline_kernel)."""
    st = SIGS.get(name) or CHAINS[name]
    chain = ops.Chain(st)
    raw, gt, g = inputs(N, 14, 164, N + len(name))
    raw, gt = raw.cuda(), gt.cuda()
    row = param_row(st, g).cuda()
    _, l1, d1 = step(ops, raw, gt, 'bilinear', chain, row)
    _, l2, d2 = step(ops, raw, gt, 'bilinear', chain, row.repeat(N, 1))
    _, l3, d3 = step(ops, raw, gt, 'bilinear', chain, row.repeat(N, 1))
    assert torch.equal(l2, l3) and torch.equal(d2, d3)
    lossclose(l2, l1, TIGHT_LOSS)
    rowclose(d2.double().sum(0, keepdim=True), d1, TIGHT_GRAD, atol=0)


# ---- the route of every case ----------------------------------------------------------------------------------------
FAMILIES = ('fused_kernel', 'pipeline_kernel', 'finalize_kernel', 'finalize_rows_kernel')


def kernels_of(fn):
    """Names of the CUDA kernels one call of fn launches."""
    from torch.profiler import ProfilerActivity, profile
    fn()                                   # warm (module load, attributes), then profile a second call
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def families(names):
    return {f for f in FAMILIES for n in names if f in n}


def pipeline_instances(names):
    """(MODE, SIG, BIG) of every pipeline_kernel instantiation in the list (demangled or mangled names)."""
    out = set()
    for n in names:
        m = re.search(r'pipeline_kernel<\s*(\d+),\s*(\d+),\s*(\d+)u?,\s*(true|false)\s*>', n) or \
            re.search(r'pipeline_kernelILi(\d+)ELi(\d+)ELj(\d+)ELb([01])E', n)
        if m:
            out.add((int(m.group(2)), int(m.group(3)) != 0, m.group(4) in ('true', '1')))
        else:
            assert 'pipeline_kernel' not in n, ('cannot parse', n)
    return out


def test_every_route_runs_the_kernel_it_claims(ops):
    N, H, W = 2, 12, 132
    raw, gt, g = inputs(9, H, W, 3)
    raw, gt = raw.cuda(), gt.cuda()
    dy = torch.randn(9, 3, H, W, generator=g).cuda()
    A, big, small = SIGS['A'], CHAINS['classical'], CHAINS['gtm5_clip']
    rA, rbig, rsmall = param_row(A, g).cuda(), param_row(big, g).cuda(), param_row(small, g).cuda()
    r2, r9 = raw[:N], raw
    cases = [
        # label, call, kernel families that must run, families that must not, pipeline_kernel instantiations
        # (MODE, SIG != 0, BIG template flag; the A-D instantiations derive BIG from the signature and pass false)
        ('packed step', lambda: step(ops, r2, gt[:N], 'bilinear', ops.Chain(A), rA),
         {'fused_kernel', 'finalize_rows_kernel'}, {'pipeline_kernel', 'finalize_kernel'}, set()),
        ('packed step, per-image rows', lambda: step(ops, r2, gt[:N], 'bilinear', ops.Chain(A), rA.repeat(N, 1)),
         {'fused_kernel', 'finalize_rows_kernel'}, {'pipeline_kernel'}, set()),
        ('packed bwd', lambda: bwd(ops, r2, dy[:N], 'malvar', ops.Chain(A), rA),
         {'fused_kernel', 'finalize_rows_kernel'}, {'pipeline_kernel', 'finalize_kernel'}, set()),
        ('generic step', lambda: step(ops, r2, gt[:N], 'bilinear', ops.Chain(small), rsmall),
         {'pipeline_kernel', 'finalize_rows_kernel'}, {'fused_kernel'}, {(1, False, False)}),
        ('generic BIG step', lambda: step(ops, r2, gt[:N], 'nearest', ops.Chain(big), rbig),
         {'pipeline_kernel', 'finalize_rows_kernel'}, {'fused_kernel'}, {(1, False, True)}),
        ('generic bwd', lambda: bwd(ops, r2, dy[:N], 'bilinear', ops.Chain(small), rsmall.repeat(N, 1)),
         {'pipeline_kernel', 'finalize_rows_kernel'}, {'fused_kernel', 'finalize_kernel'}, {(1, False, False)}),
        ('generic BIG bwd', lambda: bwd(ops, r2, dy[:N], 'malvar', ops.Chain(big), rbig),
         {'pipeline_kernel', 'finalize_rows_kernel'}, {'fused_kernel'}, {(1, False, True)}),
        ('signature on pipeline_kernel', lambda: step(ops, r9, gt, 'bilinear', ops.Chain(A), rA.repeat(9, 1)),
         {'pipeline_kernel', 'finalize_rows_kernel'}, {'fused_kernel'}, {(1, True, False)}),
        ('signature bwd on pipeline_kernel', lambda: bwd(ops, r9, dy, 'bilinear', ops.Chain(SIGS['D']),
                                                         param_row(SIGS['D'], g).cuda().repeat(9, 1)),
         {'pipeline_kernel', 'finalize_rows_kernel'}, {'fused_kernel'}, {(1, True, False)}),
    ]
    raw65, gt65, _ = inputs(65, 6, 8, 65)
    raw65, gt65 = raw65.cuda(), gt65.cuda()
    raw64, gt64 = raw65[:64].contiguous(), gt65[:64].contiguous()
    cases += [
        ('65 frames, shared row', lambda: step(ops, raw65, gt65, 'bilinear', ops.Chain(A), rA),
         {'fused_kernel', 'finalize_kernel'}, {'finalize_rows_kernel'}, set()),
        ('65 frames, per-image rows', lambda: step(ops, raw65, gt65, 'bilinear', ops.Chain(big), rbig.repeat(65, 1)),
         {'pipeline_kernel', 'finalize_kernel'}, {'finalize_rows_kernel', 'fused_kernel'}, {(1, False, True)}),
        ('64 frames, per-image rows', lambda: step(ops, raw64, gt64, 'bilinear', ops.Chain(A), rA.repeat(64, 1)),
         {'pipeline_kernel', 'finalize_rows_kernel'}, {'fused_kernel'}, {(1, True, False)}),
        ('demosaic only', lambda: step(ops, r2, gt[:N], 'bilinear', ops.Chain([]), None),
         {'finalize_kernel'}, {'finalize_rows_kernel', 'fused_kernel'}, {(1, False, False)}),
    ]
    for label, fn, must, must_not, inst in cases:
        names = kernels_of(fn)
        fams = families(names)
        assert must <= fams and not (must_not & fams), (label, names)
        assert pipeline_instances(names) == inst, (label, names)


# ---- containers ---------------------------------------------------------------------------------------------------
def _first_step(arch, loss, fuse, raw, gt):
    """One IspModel step -> (loss, [logit gradients])."""
    from reconfigisp_b200.tuning import IspModel
    opt = {'model': 'isp', 'is_train': True, 'cuda_graph': False,
           'network_G': {'which_model_G': 'OriginUniversal', 'architecture': arch, 'weight_seed': 10},
           'train': {'lr_G': 1e-2, 'beta1': 0.9, 'beta2': 0.99, 'pixel_criterion': loss, 'lr_scheme': 'MultiStepLR',
                     'lr_steps': [100], 'lr_gamma': 0.5}}
    m = IspModel(opt)
    m.netG.fuse = fuse
    m.feed_data((raw, gt))
    m.optimize_parameters()
    return float(m.l_pix), [p.grad.detach().clone() for p in m.netG.trainable_parameters if p.numel()], m


@pytest.mark.parametrize('arch, loss', [('Bayer_02_Demosaic_02_sRGB_11_13_01', 'l2'),
                                        ('Bayer_02_Demosaic_02_sRGB_11_13_01_05', 'l2'),
                                        ('Bayer_02_Demosaic_02_sRGB_11_13_01', 'l1')])
def test_container_generic_chain_fused_equals_unfused(ops, arch, loss):
    """IspModel on the classical tail 11_13_01 (a generic chain): the fused step (MSE), the fused head followed by grayworld
    (05: the head's gradient comes from `risp_pipeline_bwd` on pipeline_kernel) and the L1 criterion (no fused L1 step for
    a generic chain: the model steps through its unfused fallback) give the first step's logit gradients of the unfused
    stage-by-stage model."""
    from reconfigisp_b200.synthetic import synthetic_frames
    raw, gt = synthetic_frames(2, 48, 136, seed=3)
    raw, gt = raw.cuda(), gt.cuda()
    lf, gf, m = _first_step(arch, loss, True, raw, gt)
    lu, gu, _ = _first_step(arch, loss, False, raw, gt)
    plan = m.netG.fused_mse_step_plan()
    if arch.endswith('_05'):
        assert plan is None
    else:
        dm_kind, chain, keep = plan
        assert chain.names == ['gain', 'poly10', 'gamma'] and not ops.fused_chain_supported(chain)
        if loss == 'l1':
            table = m.netG._segment_table(keep, 2)
            with pytest.raises(NotImplementedError):
                ops.pipeline_l1(table, raw, gt, dm_kind, chain)
    fams = families(kernels_of(lambda: m.optimize_parameters()))
    assert 'pipeline_kernel' in fams and 'fused_kernel' not in fams, fams
    assert abs(lf - lu) <= TOL_LOSS * lu, (lf, lu)
    assert len(gf) == len(gu) >= 3
    for a, b in zip(gf, gu):
        rowclose(a.view(1, -1), b.view(1, -1))


if __name__ == '__main__':
    child_main(sys.argv[1])
