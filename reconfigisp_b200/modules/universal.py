"""Fixed-pipeline containers: `IspUniversal` (proxy ISP, isp_universal.py:12-236) and `OriginUniversal`
(original algorithms, origin_universal.py:9-165).  Same constructor signatures, attributes
(`all_modules`, `all_params`, `is_conditional`, `trainable_parameters`, `intermediate_results`) and
state-dict keys (`param_step{n}_{name}`), so a checkpoint tuned with IspUniversal loads `strict` into
OriginUniversal exactly as in the reference (options/test/S7ISP_test.yml:29-30).

B200-first difference: the reference runs one full-image pass per stage.  Here `forward` PLANS the
pipeline into segments -- [CNN stage] | [demosaic head + run of per-pixel stages] | [statistics stage] --
and each classical segment is ONE kernel launch (`ops.pipeline_fwd` / `ops.chain_apply`), with the
per-stage outputs the reference keeps in `intermediate_results` materialised lazily on first access.
`fuse=False` restores the stage-by-stage evaluation (used by the parity tests).
"""
import numpy as np
import torch
import torch.nn as nn

from .. import ops
from . import registry as R
from . import tools_origin as T


class _LazyIntermediates:
    """List-like view of the per-stage outputs (isp_universal.py:230): computed stage by stage on demand."""

    def __init__(self, net, x):
        self._net, self._x, self._cache = net, x, None

    def _materialise(self):
        if self._cache is None:
            with torch.no_grad():
                self._cache = self._net._run_sequential(self._x)[1]
        return self._cache

    def __len__(self):
        return len(self._net.all_modules)

    def __getitem__(self, i):
        return self._materialise()[i]

    def __iter__(self):
        return iter(self._materialise())


class _FusedHeadFn(torch.autograd.Function):
    """demosaic head + per-pixel chain as one kernel; backward recomputes from raw (16 B/px each way)."""

    @staticmethod
    def forward(ctx, raw, table, dm_kind, chain):
        y = ops.pipeline_fwd(raw, dm_kind, chain, table)
        ctx.dm_kind, ctx.chain = dm_kind, chain
        ctx.save_for_backward(raw.detach(), table.detach() if table is not None else None)
        ctx.tshape = None if table is None else table.shape
        return y

    @staticmethod
    def backward(ctx, dy):
        raw, table = ctx.saved_tensors
        chain = ctx.chain
        if not chain.differentiable:
            raise NotImplementedError('the fused segment holds a forward-only (Origin*) stage')
        if ctx.needs_input_grad[0]:
            raise NotImplementedError('no gradient w.r.t. the raw frame through a fused demosaic head')
        if chain.P == 0:
            return None, None, None, None
        from .. import _lib as L
        N, _, H, W = raw.shape
        tab, stride = ops._param_table(table, N, chain.P)
        dpar = torch.empty((1 if stride == 0 else N, chain.P), device=raw.device, dtype=torch.float32)
        ws = L.workspace(L.size('risp_pipeline_step_workspace', N, H, W, chain.P), raw.device)
        L.call('risp_pipeline_bwd', L.ptr(raw), L.ptr(dy.contiguous()), L.ptr(dpar), N, H, W, ops.DM[ctx.dm_kind], 1.0,
               *chain.desc(), L.ptr(tab), stride, chain.P, L.ptr(ws), ws.numel() * 4, L.stream())
        return None, dpar.view(ctx.tshape), None, None


class _Universal(nn.Module):
    ORIGIN = False

    def __init__(self, module_path, architecture, indiv_module_paths=None, weight_seed=None, fuse=True, **kwargs):
        super().__init__()
        self.architecture = architecture
        self.fuse = fuse
        self.all_modules, self.all_params, self.is_conditional, self.stage_names = [], [], [], []
        n_srgb = R.N_SRGB_ORIGIN if self.ORIGIN else len(R.NAMES['sRGB'])
        n_nets = 0
        for st in R.parse_architecture(architecture, n_srgb):
            name, cond = st.name, False
            logits = list(R.DEFAULT_LOGITS.get(name, []))
            use_net = name in ('path_bayer', 'path_bgr', 'bm3d') or (not self.ORIGIN and name in R.PROXY_CKPT)
            if use_net:
                path = None
                if weight_seed is None:
                    indiv = None if indiv_module_paths is None else indiv_module_paths[st.step - 1]
                    path = (module_path + R.PROXY_CKPT[name][1]) if indiv is None else indiv
                mod = R.build_net(name, path, None if weight_seed is None else weight_seed + n_nets)
                n_nets += 1
            elif name == 'gtmmanual':
                mod = T.GtmManual(4)                      # hard-coded 4 segments (isp_universal.py:176-178)
            elif name in R.CONDITIONAL:
                cls, key = R.CONDITIONAL[name]
                in_channels = kwargs.get(key)
                assert in_channels is not None
                mod = cls(in_channels=in_channels)
                logits = R.conditional_init(mod.total_params, logits)
                cond = True
            elif name in R.CLASSICAL:
                mod = R.CLASSICAL[name]()
            elif name in R.ORIGIN:
                mod = R.ORIGIN[name]()
            else:
                raise NotImplementedError('module %r (sRGB 19-21) is not defined by the reference either '
                                          '(isp_universal.py:92-94)' % name)
            self.all_modules.append(mod)
            self.is_conditional.append(cond)
            self.stage_names.append(name)
            if len(logits) == 0:
                self.all_params.append(nn.Parameter(torch.Tensor([])))
            else:
                key = 'param_step{}_{}'.format(st.step, name)
                setattr(self, key, nn.Parameter(torch.Tensor(logits)))
                self.all_params.append(getattr(self, key))
        self._plan = None
        self.intermediate_results = []

    def _apply(self, fn, *a, **k):
        # like the reference, candidate modules live in a plain list (their weights stay out of
        # state_dict / DDP); unlike it, `.to(device)` still has to reach them
        super()._apply(fn, *a, **k)
        for m in self.all_modules:
            m._apply(fn, *a, **k)
        registered = {id(p) for p in self.parameters()}
        for p in self.all_params:                      # the empty placeholders of parameter-free stages follow the module
            if id(p) not in registered:
                p.data = fn(p.data)
        return self

    # -- reference semantics, stage by stage (isp_universal.py:210-232) --------------------------------------
    def _stage_params(self, idx, N):
        par, cond = self.all_params[idx], self.is_conditional[idx]
        if par.nelement() == 0:
            return None
        if cond:
            return par                                    # raw vector, no sigmoid / repeat (:224-226)
        return torch.sigmoid(par).repeat(N, 1)

    def _run_sequential(self, x):
        N = x.size(0)
        inter = []
        for i, mod in enumerate(self.all_modules):
            x = mod(x, self._stage_params(i, N))
            inter.append(x)
        return x, inter

    # -- fusion plan -----------------------------------------------------------------------------------------
    def _make_plan(self):
        """Segments: ('module', i) | ('chain', [i...]) | ('head', dm_index, [i...])."""
        plan, i, n = [], 0, len(self.all_modules)
        chainable = lambda k: hasattr(self.all_modules[k], 'chain_op') and not self.is_conditional[k]
        while i < n:
            mod = self.all_modules[i]
            if hasattr(mod, 'demosaic_kind') or chainable(i):
                head = i if hasattr(mod, 'demosaic_kind') else None
                j = i + 1 if head is not None else i
                run, big = [], 0
                while j < n and chainable(j) and len(run) < ops.MAX_STAGES:
                    isbig = self.all_modules[j].chain_op[0] in ops.BIG
                    if isbig and big:
                        break
                    big += isbig
                    run.append(j)
                    j += 1
                run_ops = [self.all_modules[k].chain_op for k in run if self.all_modules[k].chain_op[0] != 'skip']
                chain = ops.Chain(run_ops)
                keep = [k for k in run if self.all_modules[k].chain_op[0] != 'skip']
                if head is not None:
                    plan.append(('head', head, keep, chain))
                elif run:
                    plan.append(('chain', None, keep, chain))
                i = j
            else:
                plan.append(('module', i, None, None))
                i += 1
        return plan

    def _segment_table(self, keep, N):
        cols = []
        for k in keep:
            kp = self.all_modules[k].kernel_params(torch.sigmoid(self.all_params[k]).view(1, -1))
            if kp is not None:
                cols.append(kp.reshape(1, -1))
        return torch.cat(cols, dim=1) if cols else None

    def _run_fused(self, x, stop=None):
        """The planned segments [0, stop) (all of them by default)."""
        if self._plan is None:
            self._plan = self._make_plan()
        N = x.size(0)
        for kind, idx, keep, chain in self._plan[:stop]:
            if kind == 'module':
                x = self.all_modules[idx](x, self._stage_params(idx, N))
            elif kind == 'chain':
                x = ops.chain_apply(x, chain, self._segment_table(keep, N))
            else:
                dm_kind = self.all_modules[idx].demosaic_kind
                if x.requires_grad or not (x.shape[2] % 2 == 0 and x.shape[3] % 4 == 0):
                    x = self.all_modules[idx](x, None)              # needs d/d raw, or odd geometry: unfused head
                    if keep:
                        x = ops.chain_apply(x, chain, self._segment_table(keep, N))
                else:
                    x = _FusedHeadFn.apply(x, self._segment_table(keep, N), dm_kind, chain)
        return x

    def forward(self, x):
        """x: (N,1,H,W) RGGB in [0,1] -> (N,3,H,W) BGR."""
        if self.fuse:
            y = self._run_fused(x)
            self.intermediate_results = _LazyIntermediates(self, x.detach())
            return y
        y, self.intermediate_results = self._run_sequential(x)
        return y

    @property
    def trainable_parameters(self):
        return self.all_params

    # -- evaluation (test.py: tensor2bgr -> psnr per image; get_ssim) ------------------------------------------
    def evaluate(self, x, gt, u8=False, ssim=False):
        """Score the pipeline's output on x against gt the way the reference's test scripts do -> (sse, u8_or_None):
        sse = int64 (N,) sums of squared 8-bit code differences on the device (`metrics.psnr_from_sse(sse, 3*H*W)` gives
        the per-image PSNR), u8 = the (N,H,W,3) 8-bit output images when asked for.  When the last segment of the plan is a
        fused head on a frame with even H and W % 4 == 0, that segment runs in the pipeline kernels' evaluation mode and
        its image is never written; otherwise the forward runs and `ops.sse_u8` scores it.  Runs under no_grad; parameters
        and `intermediate_results` are left as they are.
        With ssim=True -> (sse, u8_or_None, ssim_sums): ssim_sums = `ops.ssim_u8` of the output and gt, int64 (N,)
        (`metrics.ssim_from_sums(ssim_sums, 3, H, W)` gives the per-image SSIM).  On the fused-head path SSIM is computed
        from the evaluation mode's 8-bit image, which is dropped afterwards unless u8 was asked for."""
        with torch.no_grad():
            if self.fuse:
                if self._plan is None:
                    self._plan = self._make_plan()
                last = len(self._plan)
                while last > 0 and self._plan[last - 1][0] == 'chain' and not self._plan[last - 1][2]:
                    last -= 1                                   # trailing skip-only segments change nothing
                if last > 0 and self._plan[last - 1][0] == 'head':
                    _, idx, keep, chain = self._plan[last - 1]
                    h = self._run_fused(x, last - 1)
                    if h.shape[2] % 2 == 0 and h.shape[3] % 4 == 0:
                        sse, img = ops.pipeline_eval(h, gt, self.all_modules[idx].demosaic_kind, chain,
                                                     self._segment_table(keep, x.size(0)), u8=u8 or ssim)
                        if not ssim:
                            return sse, img
                        return sse, (img if u8 else None), ops.ssim_u8(img, gt)
                y = self._run_fused(x)
            else:
                y = self._run_sequential(x)[0]
            sse = ops.sse_u8(y, gt)
            img = torch.stack([ops.to_u8_hwc(y[n]) for n in range(y.shape[0])]) if u8 else None
            return (sse, img, ops.ssim_u8(y, gt)) if ssim else (sse, img)

    def store_eval_plan(self):
        """If the fused pipeline is [skip*] + one fused head (demosaic + per-pixel stages), returns (dm_kind, chain, params
        table) for `ops.pipeline_eval_store` (what `DeviceDataset.evaluate` runs on the frame store); else None."""
        if not self.fuse:
            return None
        if self._plan is None:
            self._plan = self._make_plan()
        segs = [s for s in self._plan if not (s[0] == 'chain' and not s[2])]
        if len(segs) == 1 and segs[0][0] == 'head':
            _, idx, keep, chain = segs[0]
            return self.all_modules[idx].demosaic_kind, chain, self._segment_table(keep, 1)
        return None

    # -- the whole proxy-tuning step in one pass (isp_model.py:128-142) ----------------------------------------
    def fused_mse_step_plan(self):
        """If the pipeline is [skip*] + classical demosaic + differentiable per-pixel stages, returns
        (dm_kind, chain, keep) for `ops.pipeline_mse`; else None."""
        if self._plan is None:
            self._plan = self._make_plan()
        segs = [s for s in self._plan if not (s[0] == 'chain' and not s[2])]
        if len(segs) == 1 and segs[0][0] == 'head' and segs[0][3].differentiable:
            return self.all_modules[segs[0][1]].demosaic_kind, segs[0][3], segs[0][2]
        return None


class IspUniversal(_Universal):
    """isp_universal.py:12 -- IspUniversal(module_path, indiv_module_paths, architecture, **cond_kwargs).
    `weight_seed` (extension) builds the proxy nets with seeded stand-in weights instead of loading the
    un-shipped checkpoints."""
    ORIGIN = False

    def __init__(self, module_path, indiv_module_paths, architecture, weight_seed=None, fuse=True, **kwargs):
        super().__init__(module_path, architecture, indiv_module_paths, weight_seed, fuse, **kwargs)


class OriginUniversal(_Universal):
    """origin_universal.py:9 -- OriginUniversal(module_path, architecture)."""
    ORIGIN = True

    def __init__(self, module_path, architecture, weight_seed=None, fuse=True):
        super().__init__(module_path, architecture, None, weight_seed, fuse)
