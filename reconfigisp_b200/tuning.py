"""`IspModel` -- proxy tuning / inference driver of a fixed pipeline (codes/models/isp_model.py:15-151):
same public methods (`feed_data`, `optimize_parameters`, `test`, `get_current_log`, `save`, `load`) and
option keys.  When the pipeline is a classical demosaic followed by differentiable per-pixel stages,
`optimize_parameters` runs the WHOLE step -- forward, MSE, gradients of every stage parameter -- as one
pass over the frame (`ops.pipeline_mse`, 16 B/px); otherwise it runs the planned segments with autograd.

B200 additions: `feed_data` copies into persistent device buffers (and decodes integer sensor codes on the device),
and the fused step -- parameter table, the pipeline kernel, the gradient all-reduce, Adam -- is captured once into
a CUDA graph and replayed (`opt['cuda_graph']`, default on): the ~25 tiny launches around the one big kernel are
launch-latency-bound and cost ~10 % of a 48 MP step when issued one by one."""
from collections import OrderedDict

import torch
import torch.nn as nn

from . import dist as D
from . import ops
from .networks import define_G


class IspModel:
    def __init__(self, opt):
        self.opt = opt
        self.device = torch.device('cuda')
        if not torch.cuda.is_available():
            raise RuntimeError('IspModel needs a CUDA device (no CPU fallback)')
        self.is_train = opt.get('is_train', True)
        self.netG = define_G(opt).to(self.device)
        self.netG_attr = self.netG
        self._records = None
        self.img = self.gt = self.val_img = self.val_gt = self.meta = None
        self._output = None
        self.log_dict = OrderedDict()
        self.optimizers, self.schedulers = [], []
        if self.is_train:
            t = opt['train']
            self.loss_type = t['pixel_criterion']
            if self.loss_type not in ('l1', 'l2'):
                raise NotImplementedError('pixel_criterion %r' % self.loss_type)
            self.use_graph = bool(opt.get('cuda_graph', True))
            # capturable: the step counter lives on the device, so the update can be replayed from a CUDA graph;
            # fused: one multi-tensor kernel for the whole update instead of ~7 foreach launches
            self.optimizer_G = torch.optim.Adam([p for p in self.netG.trainable_parameters], t['lr_G'], (t['beta1'], t['beta2']),
                                                capturable=self.use_graph, fused=self.use_graph)
            self._graph, self._graph_key, self._eager_steps = None, None, 0
            # all trainable gradients are views of ONE flat buffer: zeroing is one kernel and the data-parallel exchange is
            # one in-place all-reduce (no cat / div / per-tensor copies; codes/models/darts_model.py:31,173 use a DDP bucket)
            ps = [p for p in self.netG.trainable_parameters if p.numel() > 0]
            self._flat_grad = torch.zeros(sum(p.numel() for p in ps), device=self.device, dtype=torch.float32)
            o = 0
            for p in ps:
                p.grad = self._flat_grad[o:o + p.numel()].view_as(p)
                o += p.numel()
            self.optimizers.append(self.optimizer_G)
            if t.get('lr_scheme', 'MultiStepLR') == 'MultiStepLR':
                self.schedulers.append(torch.optim.lr_scheduler.MultiStepLR(self.optimizer_G, t['lr_steps'], t['lr_gamma']))
            else:
                raise NotImplementedError('MultiStepLR learning rate scheme is enough.')
        self.load()

    # -- data ------------------------------------------------------------------------------------------------
    @property
    def img(self):
        """The fed batch's raw (N,1,H,W) fp32; after a records feed, decoded from the stores on first use."""
        if self._img is None and self._records is not None:
            self._img, self._gt = self._records.decode()
        return self._img

    @img.setter
    def img(self, v):
        self._img = v

    @property
    def gt(self):
        """The fed batch's target (N,3,H,W) fp32, decoded on first use like `img`."""
        if self._gt is None and self._records is not None:
            self._img, self._gt = self._records.decode()
        return self._gt

    @gt.setter
    def gt(self, v):
        self._gt = v

    def feed_data(self, data):
        """(img, gt[, val_img, val_gt]) host or device tensors, or a `data.StoreBatch` (`DeviceDataset.records`).

        A StoreBatch is kept as its records: when the fused step applies (`_fast_plan`, frames with W % 16 == 0, crops with
        w % 4 == 0 and h even) `optimize_parameters` reads the crops' codes straight from the stores; `img` / `gt` are
        decoded only when something needs them (`output`, `test`, `evaluate`, the step of any other pipeline).

        Host tensors are copied on a side stream into one of TWO persistent device buffer sets (alternating), and integer
        sensor / display codes are decoded there as well, so the copy of batch k+1 overlaps the step of batch k when the
        caller feeds the next batch before reading the loss:  optimize_parameters(); feed_data(next); loss.item().
        The step waits for its own batch's copy (event), and a buffer set is not overwritten before the step that read it
        has finished -- the plain feed_data(); optimize_parameters() order of the reference keeps working unchanged."""
        from .data import StoreBatch
        if isinstance(data, StoreBatch):
            self._records, self._pending, self._output = data, None, None
            self.img = self.gt = None
            return
        self._records = None
        if len(data) == 2:
            img, gt = data
        elif len(data) == 4:
            img, gt, val_img, val_gt = data
            self.val_img = val_img.to(self.device, non_blocking=True)
            self.val_gt = val_gt.to(self.device, non_blocking=True)
        else:
            raise ValueError('Invalid data format.')
        st = self.__dict__.setdefault('_feed', {'parity': 0, 'stream': torch.cuda.Stream(), 'copied': [None, None],
                                                'used': [None, None]})
        on_host = not (img.is_cuda and gt.is_cuda)
        if on_host:
            b = st['parity'] = 1 - st['parity']
            cur = torch.cuda.current_stream()
            if st['used'][b] is not None:
                st['stream'].wait_event(st['used'][b])        # the step that last read this buffer set is done
            st['stream'].wait_stream(cur) if st['copied'][b] is None else None
            with torch.cuda.stream(st['stream']):
                self.img = self._to_device('img%d' % b, img, self.opt.get('raw_white_level', 1023.))
                self.gt = self._to_device('gt%d' % b, gt, 255.)
                ev = torch.cuda.Event()
                ev.record(st['stream'])
            st['copied'][b] = ev
            self._pending = (b, ev)
        else:
            self.img = self._to_device('img', img, self.opt.get('raw_white_level', 1023.))
            self.gt = self._to_device('gt', gt, 255.)
            self._pending = None
        self._output = None

    def _sync_feed(self):
        """Make the current stream wait for the copy of the batch it is about to read."""
        pend = getattr(self, '_pending', None)
        if pend is not None:
            torch.cuda.current_stream().wait_event(pend[1])

    def _mark_used(self):
        pend = getattr(self, '_pending', None)
        if pend is not None:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            self._feed['used'][pend[0]] = ev

    def _to_device(self, slot, t, denom):
        """fp32 tensors are copied as they are (the reference's contract); integer sensor / display codes
        (uint8, uint16/int16) are copied as codes and normalised on the device (`ops.decode_codes`).  The device
        buffers persist across calls of the same shape (stable addresses: the captured step reads them)."""
        bufs = self.__dict__.setdefault('_bufs', {})
        if t.is_cuda and t.dtype == torch.float32:
            return t                                        # caller-owned device tensor: used in place
        dst = bufs.get(slot)
        if dst is None or dst.shape != t.shape:
            dst = bufs[slot] = torch.empty(t.shape, device=self.device, dtype=torch.float32)
        if t.dtype.is_floating_point:
            dst.copy_(t, non_blocking=True)
            return dst
        key = slot + '_codes'
        codes = bufs.get(key)
        if codes is None or codes.shape != t.shape or codes.dtype != t.dtype:
            codes = bufs[key] = torch.empty(t.shape, device=self.device, dtype=t.dtype)
        codes.copy_(t, non_blocking=True)
        return ops.decode_codes(codes, denom, out=dst)

    # -- training step ---------------------------------------------------------------------------------------
    def _fast_plan(self):
        """The whole step without an autograd graph: [logits -> table] -> single-pass fused step -> [d table -> d logits]
        written straight into the flat gradient buffer.  Possible when the pipeline fuses into one head (classical demosaic
        + per-pixel stages the packed kernels are instantiated for) and every stage maps sigmoid(logit) affinely into its
        range.  Built once; returns None when the pipeline does not qualify."""
        if hasattr(self, '_fast'):
            return self._fast
        self._fast = None
        plan = self.netG.fused_mse_step_plan() if self.netG.fuse else None
        if plan is None or not ops.fused_chain_supported(plan[1]):
            return None
        dm_kind, chain, keep = plan
        a, b, params = [], [], []
        for k in keep:
            p, mod = self.netG.all_params[k], self.netG.all_modules[k]
            n = p.numel()
            if n == 0:
                continue
            with torch.no_grad():
                k0 = mod.kernel_params(torch.zeros(1, n, device=self.device))
                k1 = mod.kernel_params(torch.ones(1, n, device=self.device))
                kh = mod.kernel_params(torch.full((1, n), 0.5, device=self.device))
            if k0 is None or k0.numel() != n or not torch.allclose(kh, 0.5 * (k0 + k1), atol=1e-6):
                return None                                   # not an element-wise affine mapping
            a.append((k1 - k0).reshape(-1)); b.append(k0.reshape(-1)); params.append(p)
        covered = {id(p) for p in params}
        if any(p.numel() > 0 and id(p) not in covered for p in self.netG.trainable_parameters) or not params:
            return None
        # the covered logits become views of ONE flat buffer, in table order (state-dict keys and Parameter objects unchanged)
        flat = torch.cat([p.detach().reshape(-1) for p in params]).contiguous()
        grad = torch.zeros_like(flat)
        o = 0
        for p in params:
            n = p.numel()
            p.data = flat[o:o + n].view_as(p)
            p.grad = grad[o:o + n].view_as(p)
            o += n
        self._flat_grad = grad
        P = flat.numel()
        assert P == chain.P
        self._fast = dict(dm=dm_kind, chain=chain, logits=flat, grad=grad, a=torch.cat(a).contiguous(), b=torch.cat(b).contiguous(),
                          table=torch.empty((1, P), device=self.device), steps={})
        return self._fast

    def _store_step(self):
        """The fed StoreBatch when the fused step can read its crops from the stores, else None."""
        rec = self._records
        if rec is None or not self.opt.get('fast_step', True) or self._fast_plan() is None:
            return None
        if rec.h % 2 or rec.w % 4 or rec.ds.W % 16 or self.loss_type not in ('l1', 'l2'):
            return None
        return rec

    def _fast_loss_and_grads(self):
        f = self._fast_plan()
        rec = self._store_step()
        if f is None:
            return False
        N, H, W = (rec.B, rec.h, rec.w) if rec is not None else (self.img.shape[0],) + tuple(self.img.shape[2:])
        if H % 2 or W % 4 or self.loss_type not in ('l1', 'l2'):
            return False
        from . import _lib as L
        key = (N, H, W)
        step = f['steps'].get(key)
        if step is None:
            step = f['steps'][key] = ops.PipelineStep(N, H, W, f['dm'], f['chain'], self.device, l1=(self.loss_type == 'l1'))
        P = f['logits'].numel()
        L.call('risp_param_table_fwd', L.ptr(f['logits']), L.ptr(f['a']), L.ptr(f['b']), L.ptr(f['table']), P, L.stream())
        if rec is not None:
            ds = rec.ds
            loss, dtable = step.store(ds.raw_store, ds.gt_store, rec.pos, ds.white_level, ds.status, f['table'])
        else:
            loss, dtable = step(self.img, self.gt, f['table'])
        L.call('risp_param_table_bwd', L.ptr(f['logits']), L.ptr(f['a']), L.ptr(dtable), L.ptr(f['grad']), P, L.stream())
        self.l_pix = loss.view(())
        # device scalar living in the step's persistent buffer: the NEXT step overwrites it, so read (`.item()`) or clone it
        # before stepping again -- the reference stores `l_pix.item()` (isp_model.py:141)
        self.log_dict['loss'] = self.l_pix
        return True

    def _fused_loss(self):
        plan = self.netG.fused_mse_step_plan() if self.netG.fuse else None
        H, W = self.img.shape[2:]
        if plan is None or H % 2 or W % 4:
            return None
        dm_kind, chain, keep = plan
        table = self.netG._segment_table(keep, self.img.shape[0])
        if self.loss_type == 'l1':
            if not ops.fused_chain_supported(chain):
                return None                                   # generic chains: unfused path with ops.l1_loss
            return ops.pipeline_l1(table, self.img, self.gt, dm_kind, chain)
        return ops.pipeline_mse(table, self.img, self.gt, dm_kind, chain)

    def optimize_parameters(self):
        """isp_model.py:132-141.  Eager for the first two calls (allocator / optimizer-state warm-up), then the fused
        step is captured into a CUDA graph and replayed for as long as buffers, shapes and learning rates stay put."""
        self._sync_feed()
        if not (self.use_graph and self._graph_replay()):
            self._step_eager()
        self._mark_used()

    def _graph_signature(self):
        lrs = tuple(float(g['lr']) for g in self.optimizer_G.param_groups)
        rec = self._store_step()
        if rec is not None:          # the captured store step reads the record buffer and the stores
            return ('records', rec.pos.data_ptr(), rec.ds.raw_store.data_ptr(), rec.ds.gt_store.data_ptr(),
                    (rec.B, rec.h, rec.w), lrs)
        return (self.img.data_ptr(), self.gt.data_ptr(), tuple(self.img.shape), tuple(self.gt.shape), lrs)

    def _graph_replay(self):
        key = self._graph_signature()
        graphs = self.__dict__.setdefault('_graphs', {})   # one captured step per buffer set (double-buffered feed)
        if key in graphs:
            g_loss, g_update, l_pix = graphs[key]
            g_loss.replay()
            if g_update is not None:                       # data parallel: the collective stays outside the graphs
                self._allreduce_grads()
                g_update.replay()
            self.l_pix = l_pix
            self.log_dict['loss'] = l_pix
            return True
        seen = self.__dict__.setdefault('_seen_keys', {})
        seen[key] = seen.get(key, 0) + 1
        if len(seen) > 8:                                   # a loop that feeds fresh device tensors every step: stay eager
            seen.clear(); graphs.clear()
        # capture only once the same buffers / shapes / learning rates have been seen before (a loop that feeds fresh
        # device tensors every step would otherwise re-capture every step)
        if seen.get(key, 0) < 2 or self._eager_steps < 2 or not self.netG.fuse or \
                self.netG.fused_mse_step_plan() is None:
            return False
        try:
            torch.cuda.synchronize()
            g_loss, g_update = torch.cuda.CUDAGraph(), None
            if not D.is_dist() or self.__dict__.get('_p2p') is not None:
                # single GPU, or data parallel with the peer-memory exchange (a plain kernel): the whole step is ONE graph
                with torch.cuda.graph(g_loss):
                    self._step_eager(count=False)
            else:
                # NCCL kernels are kept out of the graphs: [table, pipeline kernel, finaliser, backward] | all-reduce | [Adam].
                # Capturing the collective as well was measured at 2 GPUs (round 2): no gain (0.410 vs 0.406 ms per step) and the
                # captured communicator stalls process teardown -- not worth it for one 37-float all-reduce.
                with torch.cuda.graph(g_loss):
                    self._loss_and_grads()
                g_update = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g_update, pool=g_loss.pool()):
                    self.optimizer_G.step()
            graphs[key] = (g_loss, g_update, self.l_pix)
            self._graph = graphs                           # (kept for callers that drop the graphs before teardown)
            return self._graph_replay()                    # capturing does not execute: run the step now
        except Exception as e:                             # capture is an optimisation: fall back to eager launches
            import logging
            logging.getLogger('base').warning('CUDA-graph capture of the tuning step failed (%s); running eagerly', e)
            self.use_graph, self._graph = False, None
            graphs.clear()
            torch.cuda.synchronize()
            return False

    def _loss_and_grads(self):
        if self.opt.get('fast_step', True) and self._fast_loss_and_grads():
            return
        l_pix = self._fused_loss()
        if l_pix is None:
            self._output = self.netG(self.img)
            l_pix = (ops.l1_loss if self.loss_type == 'l1' else ops.mse_loss)(self._output, self.gt)
        self._flat_grad.zero_()                        # p.grad are views of it; backward accumulates in place
        l_pix.backward()
        self.l_pix = l_pix.detach()
        self.log_dict['loss'] = self.l_pix             # device scalar; `.item()` it when logging

    def _allreduce_grads(self):
        if not D.is_dist():
            return
        if '_p2p' not in self.__dict__:                    # first exchange: try to set up the NVLink peer-memory path (all ranks or none)
            self._p2p = D.P2PAllReduce.create(cap=max(1024, self._flat_grad.numel())) if self.opt.get('p2p_allreduce', True) else None
        if self._p2p is not None:
            self._p2p(self._flat_grad)                     # one single-CTA kernel: peer stores + flags + rank-ordered sum
        else:
            D.allreduce_mean_(self._flat_grad)

    def _step_eager(self, count=True):
        if count:
            self._eager_steps += 1
        self._loss_and_grads()
        self._allreduce_grads()
        self.optimizer_G.step()

    @property
    def output(self):
        """The output image of the last step (computed on demand when the fused step skipped it)."""
        if self._output is None and self.img is not None:
            with torch.no_grad():
                self._output = self.netG(self.img)
        return self._output

    def test(self):
        self._output = self.netG(self.img)
        return self._output, self.netG.intermediate_results

    def evaluate(self, u8=False, ssim=False):
        """Score the fed batch like the reference's test script (tensor2bgr -> psnr per image) -> (sse, u8_or_None), or with
        ssim=True (sse, u8_or_None, ssim_sums), see `_Universal.evaluate`; `metrics.psnr_from_sse(sse, 3*H*W)` gives the
        PSNR and `metrics.ssim_from_sums(ssim_sums, 3, H, W)` the SSIM.  Reads the batch like a step does (waits for its
        copy, marks it used for the double-buffered feed) and leaves the optimizer, the gradients and the captured step
        graphs alone."""
        self._sync_feed()
        res = self.netG.evaluate(self.img, self.gt, u8=u8, ssim=ssim)
        self._mark_used()
        return res

    def get_current_log(self):
        return self.log_dict

    # -- checkpoints (base_model.py:77-97): {iter}_G.pth = CPU state_dict, 'module.' prefixes stripped on load --
    def save_network(self, path):
        torch.save(OrderedDict((k, v.cpu()) for k, v in self.netG.state_dict().items()), path)

    def load_network(self, path, strict=True):
        state = torch.load(path, map_location='cpu')
        clean = OrderedDict((k[7:] if k.startswith('module.') else k, v) for k, v in state.items())
        self.netG.load_state_dict(clean, strict=strict)

    def load(self):
        path = (self.opt.get('path') or {}).get('pretrain_model_G')
        if path is not None:
            self.load_network(path, (self.opt.get('path') or {}).get('strict_load', True))

    def save(self, path):
        self.save_network(path)
