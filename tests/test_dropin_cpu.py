"""Boundary 1 drop-in (SURVEY.md §8b, INTEGRATION.md §1): the reference's `codes/models/modules/tools_origin.py` calls this
repository's plugin directory `reconfigisp_b200/isp_kernels/` (the five module names it resolves through sys.path,
tools_origin.py:8-17).  Without a GPU: `reconfigisp_b200.ops` -- what the plugins call -- is patched to the CPU oracle, so what is
exercised is the contract between the reference wrappers and the plugins: option names, NHWC / NCHW layouts, 0-255 scaling,
numpy vs tensor parameters, integer window tensors, dict descriptors.  Every wrapper class of the file is called once and its
result is compared with the oracle applied to the wrapper's documented parameter mapping.

Two ways in: the calls recorded from the wrappers in tests/golden/tools_origin_calls.json are replayed against the plugins
(always), and the reference's UNMODIFIED file is imported over the plugins when its tree is present (RISP_REFERENCE_ROOT)."""
import importlib
import json
import os
import sys

import numpy as np
import pytest
import torch

from oracle import isp_oracle as O
from oracle import ref_loader as RL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PLUGINS = ('whitebalance', 'gamma', 'demosaic', 'globaltonemapping', 'spatialnoisereduction')

# wrapper -> (input, parameter tensor) it is called with, and the oracle applied to its documented parameter mapping
ARGS = {'Gamma': ('x', 'p1'), 'Grayworld': ('x', None), 'WbManual': ('x', 'p3'), 'DemosaicNearest': ('raw', None),
        'OriginDemosBilinear': ('raw', None), 'OriginDemosLaplacian': ('raw', None), 'OriginToneReinhard': ('x', 'p2'),
        'OriginToneCrysis': ('x', 'p1'), 'OriginToneFilmic': ('x', 'p2'), 'OriginWbWhiteworld': ('x', 'p1'),
        'OriginNoiseBilateral': ('x', 'pb'), 'OriginNoiseMedian': ('x', 'pm'), 'OriginNoiseFastnlm': ('x', 'pn')}
EXPECTED = {
    # differentiable wrappers, image in [0,1]
    'Gamma': (lambda t: O.gamma_manual(t['x'], t['p1']), 1e-5),
    'Grayworld': (lambda t: O.wb_grayworld(t['x']), 1e-5),
    'WbManual': (lambda t: O.wb_manual(t['x'], t['p3'] * 5), 1e-5),                                          # gain = p*5 (:214)
    'DemosaicNearest': (lambda t: O.demosaic_nearest(t['raw']), 0),
    # Origin* wrappers: x255, numpy parameters, /255 (:462-473, :535-546, :655-662, :696-710, :742-751, :785-797)
    'OriginDemosBilinear': (lambda t: O.demosaic_bilinear(t['raw'] * 255) / 255, 1e-5),
    'OriginDemosLaplacian': (lambda t: O.demosaic_laplacian(t['raw'] * 255, 255.) / 255, 1e-5),
    'OriginToneReinhard': (lambda t: O.tone_reinhard(t['x'] * 255, t['p2'][:, 0], t['p2'][:, 1]) / 255, 1e-5),
    'OriginToneCrysis': (lambda t: O.tone_crysis(t['x'] * 255, t['p1'][:, 0]) / 255, 1e-5),
    'OriginToneFilmic': (lambda t: O.tone_filmic(t['x'] * 255, t['p2'][:, 0], t['p2'][:, 1] * 9 + 1) / 255, 1e-5),  # p*9+1 (:613)
    'OriginWbWhiteworld': (lambda t: O.wb_whiteworld(t['x'] * 255, t['p1'][:, 0]) / 255, 1e-5),
    'OriginNoiseBilateral': (lambda t: O.denoise_bilateral(t['x'] * 255, O.bilateral_window_from_param(t['pb'][:, 0]),   # .int()*7 (:698)
                                                           t['pb'][:, 1] * 99 + 1, t['pb'][:, 2] * 99 + 1) / 255, 1e-5),
    'OriginNoiseMedian': (lambda t: O.denoise_median(t['x'] * 255, O.median_size_from_param(0.45)) / 255, 0),       # batch row 0 (:744)
    'OriginNoiseFastnlm': (lambda t: O.denoise_fastnlm(t['x'] * 255, O.bilateral_window_from_param(t['pn'][:, 0]),
                                                       O.bilateral_window_from_param(t['pn'][:, 1]), t['pn'][:, 2] * 99 + 1) / 255, 1e-5),
}
FAMILIES = {'gamma', 'gain', 'grayworld', 'whiteworld', 'demosaic', 'reinhard', 'crysis', 'filmic', 'bilateral', 'median', 'fastnlm'}


def inputs():
    g = torch.Generator().manual_seed(2)
    N, H, W = 2, 12, 16
    t = {'x': torch.rand(N, 3, H, W, generator=g), 'raw': torch.rand(N, 1, H, W, generator=g)}
    for name, P in (('p1', 1), ('p3', 3), ('p2', 2), ('pb', 3), ('pn', 3)):
        t[name] = torch.rand(N, P, generator=g)
    t['pm'] = torch.tensor([[0.45], [0.9]])
    return t


@pytest.fixture
def plugin_calls(request):
    """Patch the ops the plugins call to the oracle, put the plugin directory on sys.path; -> the list of ops reached."""
    import reconfigisp_b200.ops as ops
    from reconfigisp_b200 import isp_kernels
    saved = {k: getattr(ops, k) for k in ('gamma', 'gain', 'grayworld', 'whiteworld', 'demosaic', 'tone_reinhard', 'tone_crysis',
                                          'tone_filmic', 'bilateral', 'median', 'fastnlm')}
    calls = []

    def log(name, fn):
        def w(*a, **k):
            calls.append(name)
            return fn(*a, **k)
        return w
    ops.gamma = log('gamma', lambda x, g: O.gamma_manual(x, g))
    ops.gain = log('gain', lambda x, g: O.wb_manual(x, g))
    ops.grayworld = log('grayworld', lambda x: O.wb_grayworld(x))
    ops.whiteworld = log('whiteworld', lambda x, r, s=1.0: O.wb_whiteworld(x, r))
    ops.demosaic = log('demosaic', lambda raw, kind, clip_hi=1.0: {'nearest': O.demosaic_nearest, 'bilinear': O.demosaic_bilinear,
                                                                  'malvar': lambda r: O.demosaic_laplacian(r, clip_hi)}[kind](raw))
    ops.tone_reinhard = log('reinhard', lambda x, wp, mg, s=1.0: O.tone_reinhard(x, wp, mg))
    ops.tone_crysis = log('crysis', lambda x, la, s=1.0: O.tone_crysis(x, la))
    ops.tone_filmic = log('filmic', lambda x, wp, eb, s=1.0: O.tone_filmic(x, wp, eb))
    ops.bilateral = log('bilateral', lambda x, win, sc, ss, max_window=None: O.denoise_bilateral(x, win, sc, ss))
    ops.median = log('median', lambda x, k: O.denoise_median(x, k))
    ops.fastnlm = log('fastnlm', lambda x, b, s, h, max_halo=None: O.denoise_fastnlm(x, b, s, h))
    here = isp_kernels.install()                      # what a deployment does: put the plugin directory on sys.path
    for name in PLUGINS:
        sys.modules.pop(name, None)

    def restore():
        for k, v in saved.items():
            setattr(ops, k, v)
        for name in PLUGINS:
            sys.modules.pop(name, None)
    request.addfinalizer(restore)
    return calls, here


@pytest.fixture
def tools_origin(request, plugin_calls):
    if not RL.reference_available():
        pytest.skip('reference tree not present (set RISP_REFERENCE_ROOT)')
    calls, here = plugin_calls
    codes = os.path.join(RL.REFERENCE_ROOT, 'codes')
    sys.path.insert(0, codes)
    sys.modules.pop('models.modules.tools_origin', None)
    with RL.cpu_only():
        T = importlib.import_module('models.modules.tools_origin')
    assert os.path.dirname(sys.modules['whitebalance'].__file__) == here      # OUR plugins were resolved
    assert T.__file__.startswith(RL.REFERENCE_ROOT)                           # the reference's own, unmodified file

    def restore():
        sys.modules.pop('models.modules.tools_origin', None)
        sys.path.remove(codes)
    request.addfinalizer(restore)
    T._calls = calls
    return T


def close(a, b, tol=1e-5):
    assert a.shape == b.shape, (a.shape, b.shape)
    assert float((a.detach() - b.detach()).abs().max()) <= tol, float((a.detach() - b.detach()).abs().max())


def test_reference_wrappers_run_on_our_plugins(tools_origin):
    T = tools_origin
    t = inputs()
    with RL.cpu_only():
        for name, (inp, par) in ARGS.items():
            fn, tol = EXPECTED[name]
            close(getattr(T, name)()(t[inp], None if par is None else t[par]), fn(t), tol)
    # every plugin family was reached through the reference's own call sites
    assert set(T._calls) >= FAMILIES


def _param(spec, t):
    src, col, mul, add, kind = spec
    p = t[src] if col is None else t[src][:, col]
    if kind == 'window':
        return (p.int() * 7) * 2 + 3
    if kind == 'median_size':
        return 2 * int(p[0] * 7) + 3
    v = p * mul + add
    return v.detach().cpu().numpy() if kind == 'numpy' else v


def test_recorded_wrapper_calls_run_on_our_plugins(plugin_calls):
    """The wrappers' calls into the plugins, as recorded in tests/golden/tools_origin_calls.json, replayed against this
    repository's plugins: each result, mapped back the way the wrapper does, equals the oracle on the wrapper's parameter mapping."""
    calls, here = plugin_calls
    with open(os.path.join(ROOT, 'tests', 'golden', 'tools_origin_calls.json')) as fh:
        recorded = json.load(fh)['calls']
    assert [c['wrapper'] for c in recorded] == list(EXPECTED)               # one recorded call per wrapper class
    t = inputs()
    for c in recorded:
        mod = importlib.import_module(c['module'])                          # bare name, resolved through sys.path
        assert os.path.dirname(mod.__file__) == here
        img = t[c['input']] * c['scale']
        if c['layout'] == 'nhwc':
            img = img.permute(0, 2, 3, 1)
        params = {k: _param(spec, t) for k, spec in c['params'].items()}
        if c['desc']:
            fi, bi, fo, bo = c['desc']
            H, W = t[c['input']].shape[2:]
            params.update(input={'width': W, 'height': H, 'format': fi, 'bitdepth': bi},
                          output={'width': W, 'height': H, 'format': fo, 'bitdepth': bo})
        out = getattr(mod, c['cls'])().run(img, c['option'], params)
        if c['layout'] == 'nhwc':
            out = out.permute(0, 3, 1, 2)
        fn, tol = EXPECTED[c['wrapper']]
        close(out.float() / c['scale'], fn(t), tol)
    assert set(calls) >= FAMILIES
