"""Binds a Plan to device buffers and executes it through the C ABI (libcunet_b200.so).

One Engine = one model replica on one GPU for one (batch, dtype).  All kernel parameter structs are built
once (buffers never move), so a step is a fixed sequence of C-ABI launches on the current stream: safe to
capture in a CUDA graph.  No PyTorch compute ops are on the step path (torch is used for allocation, zero
fills and the NCCL process group only).

HBM layout (all pixel-row / NHWC):
  params   fp32 flat  : every conv weight [Cout][Cin][k][k] and BN weight/bias, reference order
  grads    fp32 flat  : same layout (one contiguous allreduce bucket)
  sq_avg   fp32 flat  : RMSprop state
  bnbuf    fp32 flat  : BN running_mean / running_var
  wpack    bytes      : tensor-core operand images of every conv (fwd + dgrad), rebuilt each step
  acts     dtype      : one buffer per plan tensor [N*res*res][C]; heads fp32 [rows][head_pad]
  G        dtype      : gradient accumulator per tensor (training)
  zbuf     fp64       : per-tensor (sum, sumsq) and (sum G, sum G*T), loss, decode keys -- zeroed once per step
"""
import ctypes as C

import torch

from . import lib as L
from .plan import Plan

BN_EPS = 1e-5
BN_MOMENTUM = 0.1


def _struct_array_to_device(structs, device):
    raw = b"".join(bytes(s) for s in structs)
    return torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(device)


class BnUpdateDesc(C.Structure):
    _fields_ = [("stats", C.c_void_p * L.MAX_SEG), ("inv_count", C.c_double * L.MAX_SEG),
                ("C", C.c_int * L.MAX_SEG), ("nseg", C.c_int), ("reps", C.c_int),
                ("rmean", C.c_void_p), ("rvar", C.c_void_p), ("n_elems", C.c_double),
                ("momentum", C.c_float), ("reserved", C.c_int)]


class Engine(object):
    def __init__(self, plan, batch, dtype="bf16", device=None, double_bn_update=True, share=None):
        """share: another Engine of the same plan / dtype whose parameter storage (params, grads, optimizer
        state, BN buffers) this engine reuses -- one model, several batch sizes."""
        assert isinstance(plan, Plan)
        L.load()
        if not torch.cuda.is_available():
            raise L.CunetError("cunet_b200 needs a CUDA device: there is no CPU fallback")
        self.plan, self.N = plan, int(batch)
        self.device = torch.device(device if device is not None else "cuda")
        self.dtype = L.BF16 if dtype in ("bf16", torch.bfloat16) else L.F32
        self.tdtype = torch.bfloat16 if self.dtype == L.BF16 else torch.float32
        self.double_bn_update = double_bn_update
        self.grad_scale = 1.0          # 1 / world_size under data parallelism
        # pixel rows from which a 1x1 conv's backward runs as ONE fused dgrad+wgrad launch (CUNET_BWD1X1_MIN_ROWS).
        # Default: always -- since the fused kernel's tail was fixed (channel sums through shared memory, full-line dW
        # reductions) it beats dgrad || wgrad on two streams at every size (16x16 batch 24: 17.7 us against ~21 us;
        # whole CU-Net-8 step 12.32 ms with the old 12288-row threshold, 12.00 ms with 0)
        import os
        self.fuse1x1_min_rows = int(os.environ.get("CUNET_BWD1X1_MIN_ROWS", "0"))
        if os.environ.get("CUNET_BWD1X1_OFF"):
            self.fuse1x1_min_rows = 1 << 62
        self.wgrad_serial = os.environ.get("CUNET_WGRAD_SIDE", "1") == "0"   # debug: no side stream
        dev = self.device
        p = plan

        # ---- parameters
        off = 0
        boff = 0
        self.p_off, self.b_off, self.cnt_idx = {}, {}, {}
        for s in p.params:
            if s.kind in ("conv", "bn_weight", "bn_bias"):
                self.p_off[s.name] = (off, s.numel, s.shape)
                off += (s.numel + 3) // 4 * 4                      # keep every tensor 16-byte aligned
            elif s.kind in ("bn_mean", "bn_var"):
                self.b_off[s.name] = (boff, s.numel, s.shape)
                boff += (s.numel + 3) // 4 * 4
            else:
                self.cnt_idx[s.name] = len(self.cnt_idx)
        self.n_params = off
        # flat buffers are padded to a multiple of 64 elements so that they split evenly over 1/2/4/8/16 ranks into
        # 16-byte-aligned shards (reduce-scatter -> shard RMSprop -> all-gather variant of the optimizer step)
        off = (off + 63) // 64 * 64
        self.n_params_padded = off
        if share is not None:
            assert share.n_params_padded == off and share.dtype == self.dtype
            self.params, self.grads, self.sq_avg = share.params, share.grads, share.sq_avg
            self.bnbuf, self.counters, self.lr = share.bnbuf, share.counters, share.lr
        else:
            self.params = torch.zeros(off, device=dev)
            self.grads = torch.zeros(off, device=dev)
            self.sq_avg = torch.zeros(off, device=dev)
            self.bnbuf = torch.zeros(boff, device=dev)
            self.counters = torch.zeros(len(self.cnt_idx), dtype=torch.long, device=dev)
            for name, (o, n, _) in self.b_off.items():
                if name.endswith("running_var"):
                    self.bnbuf[o:o + n] = 1.0
            self.lr = torch.zeros(1, device=dev)

        # ---- activations, gradient accumulators, statistics
        N = self.N
        self.act, self.G, self.pidx = {}, {}, {}
        zoff = 0
        self.stat_off, self.gstat_off = {}, {}
        for t in p.tensors.values():
            rows = N * t.res * t.res
            self.act[t.name] = torch.empty(rows, t.C, device=dev, dtype=torch.float32 if t.fp32 else self.tdtype)
            self.stat_off[t.name] = zoff
            zoff += 2 * t.C
            self.gstat_off[t.name] = zoff
            zoff += 2 * t.C
            if t.fp32:
                self.G[t.name] = torch.zeros(rows, t.C, device=dev, dtype=self.tdtype)   # dLoss/dhead
            elif t.name != "stem.y":
                self.G[t.name] = torch.empty(rows, t.C, device=dev, dtype=self.tdtype)
        for op in p.ops:
            if op.pool:
                self.pidx[op.out.name] = torch.empty(N * (op.res // 2) ** 2, op.cout, device=dev, dtype=torch.uint8)
        self.nheads = len(p.heads)
        self.loss_off = zoff
        zoff += 1 + self.nheads
        self.keys_off = zoff
        zoff += N * p.class_num
        self.zbuf = torch.zeros(zoff, dtype=torch.float64, device=dev)
        self.preds = torch.zeros(N, p.class_num, 2, device=dev)
        self.target = torch.zeros(N, p.class_num, p.out_res, p.out_res, device=dev)
        self.img = torch.zeros(N, 3, p.in_res, p.in_res, device=dev)
        self.cols = torch.empty(N * p.stem_res ** 2, 160, device=dev, dtype=self.tdtype)
        self.dy0 = torch.empty(N * p.stem_res ** 2, p.C0, device=dev, dtype=self.tdtype)

        # ---- packed weights
        descs, woff = [], 0
        self.wfwd, self.wdg = {}, {}
        plist = [("features.conv0", 147, 1, p.C0, p.C0, False)]
        for op in p.ops:
            plist.append((op.conv, op.cin, op.taps, op.cout, op.cout_pad, True))
        sizes = []
        for name, cin, taps, cout, cpad, need_dg in plist:
            nf = L.pack_fwd_bytes(cin, taps, cpad, self.dtype)
            nd = L.pack_dgrad_bytes(cin, taps, cpad, self.dtype) if need_dg else 0
            sizes.append((woff, nf, nd))
            woff += nf + nd
        self.wpack = torch.zeros(woff, dtype=torch.uint8, device=dev)
        base = self.wpack.data_ptr()
        for (name, cin, taps, cout, cpad, need_dg), (o, nf, nd) in zip(plist, sizes):
            self.wfwd[name] = base + o
            self.wdg[name] = base + o + nf if need_dg else None
            wptr = self.params.data_ptr() + 4 * self.p_off[name + ".weight"][0]
            descs.append(L.PackDesc(wptr, base + o, (base + o + nf) if need_dg else None, cout, cin, taps, cpad))
        self.pack_descs = _struct_array_to_device(descs, dev)
        self.n_pack = len(descs)

        self._build_calls()

    # ------------------------------------------------------------------------------------------ pointers
    def _pp(self, name):
        return self.params.data_ptr() + 4 * self.p_off[name][0]

    def _gp(self, name):
        return self.grads.data_ptr() + 4 * self.p_off[name][0]

    def _bp(self, name):
        return self.bnbuf.data_ptr() + 4 * self.b_off[name][0]

    def _stats(self, tname):
        return self.zbuf.data_ptr() + 8 * self.stat_off[tname]

    def _gstats(self, tname):
        return self.zbuf.data_ptr() + 8 * self.gstat_off[tname]

    def is_fused_1x1(self, op):
        """True when the backward of this op is the single fused dgrad+wgrad launch of csrc/conv_bwd1x1.cu."""
        return op.taps == 1 and self.dtype == L.BF16 and self.N * op.res * op.res >= self.fuse1x1_min_rows

    def _concat(self, cc, op, mode):
        """mode: 1 train, 0 eval."""
        cc.nseg = len(op.srcs)
        for i, (t, up) in enumerate(op.srcs):
            s = cc.seg[i]
            s.ptr = self.act[t.name].data_ptr()
            s.stats = self._stats(t.name)
            s.inv_count = 1.0 / (self.N * t.res * t.res)
            s.C, s.ld, s.up = t.C, t.C, int(up)
        cc.bn_train = mode
        cc.gamma, cc.beta = self._pp(op.norm + ".weight"), self._pp(op.norm + ".bias")
        cc.rmean, cc.rvar = self._bp(op.norm + ".running_mean"), self._bp(op.norm + ".running_var")
        cc.eps = BN_EPS
        cc.act_bits = self.plan.quan_input_bits if op.quan_input else 0

    def _grad_src(self, gs, t, op):
        """Gradient of tensor t = output of op."""
        gs.g = self.G[t.name].data_ptr()
        gs.C, gs.ld = t.C, t.C
        gs.eps = BN_EPS
        if t.fp32:                       # head: plain dLoss/dhead
            gs.mode, gs.pooled = 0, 0
            gs.t = gs.stats = gs.gstats = gs.pool_idx = None
            gs.inv_count = 1.0
        else:
            gs.mode = 1
            gs.t = self.act[t.name].data_ptr()
            gs.stats, gs.gstats = self._stats(t.name), self._gstats(t.name)
            gs.inv_count = 1.0 / (self.N * t.res * t.res)
            gs.pooled = int(op.pool)
            gs.pool_idx = self.pidx[t.name].data_ptr() if op.pool else None

    # ------------------------------------------------------------------------------------------ launch lists
    def _build_calls(self):
        p, N, lib = self.plan, self.N, L.load()
        self.call_index = {}      # (op name, "fwd" | "dgrad" | "wgrad") -> parameter struct (bench probes)

        def fwd_list(mode):
            calls = []
            # stem
            sp = L.ConvFwdParams()
            self._stem_cols(sp.inp)
            sp.N, sp.H, sp.W, sp.taps = self._stem_geom()
            sp.wpack, sp.Cout, sp.CoutPad = self.wfwd["features.conv0"], p.C0, p.C0
            sp.out, sp.out_ld, sp.out_fp32 = self.act["stem.y"].data_ptr(), p.C0, 0
            sp.out_stats = self._stats("stem.y") if mode else None
            sp.pool, sp.pool_idx, sp.dtype = 0, None, self.dtype
            calls.append((lib.cunet_conv_fwd, sp))
            pp = L.StemPoolParams()
            pp.y, pp.y_stats = self.act["stem.y"].data_ptr(), self._stats("stem.y")
            pp.gamma, pp.beta = self._pp("features.norm0.weight"), self._pp("features.norm0.bias")
            pp.rmean, pp.rvar = self._bp("features.norm0.running_mean"), self._bp("features.norm0.running_var")
            pp.x = self.act["stem.x"].data_ptr()
            pp.x_stats = self._stats("stem.x") if mode else None
            pp.N, pp.H, pp.W = N, p.stem_res, p.stem_res
            pp.bn_train, pp.eps, pp.dtype = mode, BN_EPS, self.dtype
            calls.append((lib.cunet_stem_pool_fwd, pp))
            for op in p.ops:
                cp = L.ConvFwdParams()
                self._concat(cp.inp, op, mode)
                cp.N, cp.H, cp.W, cp.taps = N, op.res, op.res, op.taps
                cp.wpack, cp.Cout, cp.CoutPad = self.wfwd[op.conv], op.cout, op.cout_pad
                cp.out, cp.out_ld = self.act[op.out.name].data_ptr(), op.out.C
                cp.out_fp32 = int(op.kind == "head")
                cp.out_stats = self._stats(op.out.name) if (mode and op.kind != "head") else None
                cp.pool = int(op.pool)
                cp.pool_idx = self.pidx[op.out.name].data_ptr() if op.pool else None
                cp.dtype = self.dtype
                calls.append((lib.cunet_conv_fwd, cp))
                if mode:
                    self.call_index[(op.name, "fwd")] = cp
            return calls

        self.fwd_train, self.fwd_eval = fwd_list(1), fwd_list(0)

        # BN running statistics (one launch)
        upd = []
        d = BnUpdateDesc()
        d.stats[0], d.inv_count[0], d.C[0], d.nseg = self._stats("stem.y"), 1.0 / (N * p.stem_res ** 2), p.C0, 1
        d.reps, d.n_elems, d.momentum = 1, float(N * p.stem_res ** 2), BN_MOMENTUM
        d.rmean, d.rvar = self._bp("features.norm0.running_mean"), self._bp("features.norm0.running_var")
        upd.append(d)
        incr = torch.zeros(len(self.cnt_idx), dtype=torch.long)
        incr[self.cnt_idx["features.norm0.num_batches_tracked"]] = 1
        for op in p.ops:
            d = BnUpdateDesc()
            d.nseg = len(op.srcs)
            for i, (t, up) in enumerate(op.srcs):
                d.stats[i], d.inv_count[i], d.C[i] = self._stats(t.name), 1.0 / (N * t.res * t.res), t.C
            d.reps = 2 if (op.checkpointed and self.double_bn_update) else 1
            d.n_elems, d.momentum = float(N * op.res * op.res), BN_MOMENTUM
            d.rmean, d.rvar = self._bp(op.norm + ".running_mean"), self._bp(op.norm + ".running_var")
            upd.append(d)
            incr[self.cnt_idx[op.norm + ".num_batches_tracked"]] = d.reps
        self.bn_descs = _struct_array_to_device(upd, self.device)
        self.n_bn = len(upd)
        self.counter_incr = incr.to(self.device)

        # loss
        def mse_params(with_grad):
            mp = L.MseParams()
            for k, h in enumerate(p.heads):
                mp.heads[k] = self.act[h.name].data_ptr()
                mp.dheads[k] = self.G[h.name].data_ptr() if with_grad else None
            mp.nheads = self.nheads
            mp.target = self.target.data_ptr()
            mp.N, mp.C, mp.H, mp.W, mp.ld = N, p.class_num, p.out_res, p.out_res, p.head_pad
            mp.loss = self.zbuf.data_ptr() + 8 * self.loss_off
            mp.keys = self.zbuf.data_ptr() + 8 * self.keys_off
            mp.grad_scale, mp.dtype = 1.0, self.dtype
            return mp
        self.mse_train, self.mse_eval = mse_params(True), mse_params(False)

        # backward: the dgrad chain is the critical path; every wgrad only feeds the optimizer, so the wgrads run
        # on a side stream (a parallel branch of the captured graph) and fill the SMs the small low-resolution
        # dgrads leave idle
        calls, wcalls = [], []
        for op, flags in p.backward_schedule():
            dp = L.ConvDgradParams()
            self._concat(dp.inp, op, 1)
            for i, ((t, up), (acc, last)) in enumerate(zip(op.srcs, flags)):
                dp.gacc[i].G = self.G[t.name].data_ptr()
                dp.gacc[i].gstats = self._gstats(t.name)   # every consumer adds its share gamma*(dbeta, dgamma)
                dp.gacc[i].ld, dp.gacc[i].accumulate = t.C, int(acc)
            self._grad_src(dp.dy, op.out, op)
            dp.N, dp.H, dp.W, dp.taps = N, op.res, op.res, op.taps
            dp.wpack_dgrad, dp.Cout, dp.CoutPad = self.wdg[op.conv], op.cout, op.cout_pad
            dp.dgamma, dp.dbeta = self._gp(op.norm + ".weight"), self._gp(op.norm + ".bias")
            dp.dtype = self.dtype
            self.call_index[(op.name, "dgrad")] = dp
            wp = L.ConvWgradParams()
            self._concat(wp.inp, op, 1)
            self._grad_src(wp.dy, op.out, op)
            wp.N, wp.H, wp.W, wp.taps, wp.Cout = N, op.res, op.res, op.taps, op.cout
            wp.dw, wp.nsplit, wp.dtype, wp.dw_cin = self._gp(op.conv + ".weight"), 0, self.dtype, 0
            self.call_index[(op.name, "wgrad")] = wp
            if op.taps == 9 and self.dtype == L.BF16:
                # dense-layer 3x3: backward-data and backward-filter share the im2col of the output gradient ->
                # one fused launch on the main stream (csrc/conv_bwd3x3.cu)
                calls.append((lib.cunet_conv_bwd3x3, (dp, wp)))
            elif self.is_fused_1x1(op):
                # 1x1: backward-data and backward-filter share the gradient operand and the landed sources ->
                # one fused launch (csrc/conv_bwd1x1.cu); the split form below remains for fp32 and for shapes the
                # fused kernel does not take (it falls back by itself) and for A/B runs (CUNET_BWD1X1_MIN_ROWS)
                calls.append((lib.cunet_conv_bwd1x1, (dp, wp)))
            else:
                calls.append((lib.cunet_conv_dgrad, dp))
                wcalls.append((len(calls) - 1, lib.cunet_conv_wgrad, wp))  # may start once dgrad #k may start
        # stem backward: parameter-gradient reduction, dy, conv0 wgrad
        for phase in (0, 1):
            sb = L.StemBwdParams()
            sb.y, sb.y_stats = self.act["stem.y"].data_ptr(), self._stats("stem.y")
            sb.gamma, sb.beta = self._pp("features.norm0.weight"), self._pp("features.norm0.bias")
            sx = p.stem_x
            sb.dx.g, sb.dx.t = self.G["stem.x"].data_ptr(), self.act["stem.x"].data_ptr()
            sb.dx.stats, sb.dx.gstats = self._stats("stem.x"), self._gstats("stem.x")
            sb.dx.pool_idx, sb.dx.inv_count = None, 1.0 / (N * sx.res * sx.res)
            sb.dx.C, sb.dx.ld, sb.dx.mode, sb.dx.pooled, sb.dx.eps = sx.C, sx.C, 1, 0, BN_EPS
            sb.dgamma, sb.dbeta = self._gp("features.norm0.weight"), self._gp("features.norm0.bias")
            sb.dy = self.dy0.data_ptr()
            sb.N, sb.H, sb.W, sb.eps, sb.dtype, sb.phase = N, p.stem_res, p.stem_res, BN_EPS, self.dtype, phase
            calls.append((lib.cunet_stem_bwd, sb))
        wp = L.ConvWgradParams()
        self._stem_cols(wp.inp)
        wp.dy.g, wp.dy.C, wp.dy.ld, wp.dy.mode, wp.dy.pooled = self.dy0.data_ptr(), p.C0, p.C0, 0, 0
        wp.dy.inv_count = 1.0
        (wp.N, wp.H, wp.W, wp.taps), wp.Cout = self._stem_geom(), p.C0
        wp.dw, wp.nsplit, wp.dtype, wp.dw_cin = self._gp("features.conv0.weight"), 0, self.dtype, 147
        calls.append((lib.cunet_conv_wgrad, wp))
        self.bwd_calls = calls
        self.bwd_wgrad_calls = wcalls
        self.side_stream = torch.cuda.Stream(device=self.device)
        self._evpool = [torch.cuda.Event() for _ in range(len(wcalls) + 1)]

    def _stem_cols(self, cc):
        """The im2col matrix as an identity-input concat of its two column blocks (cunet_stem_im2col's layout)."""
        rows = self.N * self.plan.stem_res ** 2
        esz = self.cols.element_size()
        cc.nseg = 2
        for i, (off, c) in enumerate(((0, 128), (rows * 128 * esz, 32))):
            cc.seg[i].ptr = self.cols.data_ptr() + off
            cc.seg[i].C, cc.seg[i].ld, cc.seg[i].up = c, c, 0
            cc.seg[i].inv_count = 1.0
        cc.bn_train = 2

    def _stem_geom(self):
        """(N, H, W, taps) of conv0 as a 1x1 conv over the im2col rows.  Only the row count matters to a 1x1 conv without
        pooling or upsampling; maps wider than 64 are presented as more images of 64x64 so that the persistent kernels
        (csrc/conv_fwd_v3.cu, csrc/conv_wgrad_v2.cu: W <= 64) take them."""
        r = self.plan.stem_res
        if r > 64 and r % 64 == 0:
            return self.N * (r // 64) ** 2, 64, 64, 1
        return self.N, r, r, 1

    # ------------------------------------------------------------------------------------------ execution
    def _run(self, calls):
        st = L.stream_ptr()
        probes = getattr(self, "probes", None)
        for fn, prm in calls:
            ev = probes.get(id(prm[0] if isinstance(prm, tuple) else prm)) if probes else None
            if ev is not None:
                ev[0].record()
            rc = self._launch(fn, prm, st)
            if ev is not None:
                ev[1].record()
            if rc != 0:
                L.check(rc, fn.__name__)

    @staticmethod
    def _launch(fn, prm, st):
        if isinstance(prm, tuple):
            return fn(*[C.byref(q) for q in prm], st)
        return fn(C.byref(prm), st)

    def pack_weights(self):
        L.pack_weights(self.pack_descs.data_ptr(), self.n_pack, self.dtype)

    def forward(self, train):
        """img must already be in self.img.  Leaves the head outputs in self.act[head]."""
        lib = L.load()
        self.pack_weights()
        L.check(lib.cunet_stem_im2col(C.c_void_p(self.img.data_ptr()), C.c_void_p(self.cols.data_ptr()), self.N,
                                      self.plan.in_res, self.plan.in_res, self.dtype, L.stream_ptr()), "stem_im2col")
        if train:
            self.zbuf.zero_()
        self._run(self.fwd_train if train else self.fwd_eval)
        if train:
            L.check(lib.cunet_bn_running_update(C.c_void_p(self.bn_descs.data_ptr()), self.n_bn, L.stream_ptr()),
                    "bn_running_update")
            self.counters.add_(self.counter_incr)

    def loss_and_decode(self, with_grad):
        """target must already be in self.target. loss -> zbuf[loss_off], preds -> self.preds."""
        lib = L.load()
        mp = self.mse_train if with_grad else self.mse_eval
        mp.grad_scale = self.grad_scale
        if not with_grad:
            self.zbuf[self.loss_off:].zero_()
        L.check(lib.cunet_mse_decode(C.byref(mp), L.stream_ptr()), "mse_decode")
        L.check(lib.cunet_decode_finalize(C.c_void_p(self.zbuf.data_ptr() + 8 * self.keys_off),
                                          C.c_void_p(self.preds.data_ptr()), self.N * self.plan.class_num,
                                          self.plan.out_res, L.stream_ptr()), "decode_finalize")

    def backward(self):
        """dLoss/dhead must be in self.G[head] (written by loss_and_decode or by the autograd bridge)."""
        self.grads.zero_()
        main = torch.cuda.current_stream()
        side = self.side_stream
        probes = getattr(self, "probes", None)
        if probes or self.wgrad_serial:  # instrumentation mode (bench probes) / CUNET_WGRAD_SIDE=0: plain serial order
            k = 0
            for i, (fn, prm) in enumerate(self.bwd_calls):
                self._run([(fn, prm)])
                while k < len(self.bwd_wgrad_calls) and self.bwd_wgrad_calls[k][0] == i:
                    self._run([self.bwd_wgrad_calls[k][1:]])
                    k += 1
            return
        st_main = C.c_void_p(main.cuda_stream)
        st_side = C.c_void_p(side.cuda_stream)
        k = 0
        for i, (fn, prm) in enumerate(self.bwd_calls):
            # wgrad of this op needs exactly what its dgrad needs: everything launched so far on the main stream
            if k < len(self.bwd_wgrad_calls) and self.bwd_wgrad_calls[k][0] == i:
                ev = self._evpool[k]
                ev.record(main)
                side.wait_event(ev)
                _, wfn, wprm = self.bwd_wgrad_calls[k]
                rc = wfn(C.byref(wprm), st_side)
                if rc != 0:
                    L.check(rc, wfn.__name__)
                k += 1
            rc = self._launch(fn, prm, st_main)
            if rc != 0:
                L.check(rc, fn.__name__)
        if k:   # join the side branch (nothing to join when every backward-filter is fused into its backward-data)
            ev = self._evpool[-1]
            ev.record(side)
            main.wait_event(ev)

    def optimizer_step(self, alpha=0.99, eps=1e-8, start=0, end=None, grads=None):
        """RMSprop on elements [start, end) of the flat buffers; ``grads`` (default: the same slice of the gradient
        bucket) may be a separate buffer of end - start elements (the reduce-scattered shard)."""
        lib = L.load()
        end = self.n_params if end is None else end
        gptr = (self.grads.data_ptr() + 4 * start) if grads is None else grads.data_ptr()
        L.check(lib.cunet_rmsprop_step(C.c_void_p(self.params.data_ptr() + 4 * start), C.c_void_p(gptr),
                                       C.c_void_p(self.sq_avg.data_ptr() + 4 * start), C.c_long(end - start),
                                       C.c_void_p(self.lr.data_ptr()), C.c_float(alpha), C.c_float(eps),
                                       L.stream_ptr()), "rmsprop_step")

    def _state(self):
        return (self.params, self.sq_avg, self.bnbuf, self.counters)

    def save_state(self):
        """Copy of the model state a training step reads and updates: parameters, optimizer state, BatchNorm running
        statistics and counters."""
        return [t.clone() for t in self._state()]

    def restore_state(self, saved):
        """Put back a save_state() copy (in place, on the current stream: captured graphs keep their buffers)."""
        for t, k in zip(self._state(), saved):
            t.copy_(k)

    def loss_value(self):
        return self.zbuf[self.loss_off].clone()

    def head_outputs(self):
        """loss_num views shaped like the reference's outputs: [N, class_num, H, W] (NCHW view of NHWC)."""
        p = self.plan
        outs = []
        for h in p.heads:
            a = self.act[h.name].view(self.N, p.out_res, p.out_res, p.head_pad)[..., :p.class_num]
            outs.append(a.permute(0, 3, 1, 2))
        return outs

    # kernels launched per call, for bench.py's gpu_launches
    def launches_per_train_step(self):
        return 2 + len(self.fwd_train) + 1 + 2 + len(self.bwd_calls) + len(self.bwd_wgrad_calls) + 1


class Trainer(object):
    """Fused training / evaluation steps on one GPU (one process per GPU under data parallelism).

    train_step = [H2D(img, heatmap)] -> forward -> multi-loss MSE + decode -> backward -> [NCCL allreduce of the
    flat gradient bucket] -> RMSprop -> (weights re-packed at the start of the next step).
    Mirrors train() of the reference (cu-net.py:147-206) with the per-iteration .cpu() metric loops replaced by
    the fused on-device decode.  With use_graph=True the two launch sequences (forward+loss+backward, optimizer)
    are captured once into CUDA graphs and replayed; the allreduce runs between them on the same stream.
    """

    def __init__(self, net, batch, lr=2.5e-4, alpha=0.99, eps=1e-8, device=None, process_group=None,
                 world_size=1, use_graph=False, quant=None, shard_optimizer=False, rank=0):
        """quant: optional BinOp / QuanOp built on ``net`` -- the step then follows the reference's quantized
        protocol (cu-net-prev-version-bin.py:163-191): quantize -> fwd/bwd -> restore -> fix grads -> step."""
        self.net = net
        self.quant = quant
        self.eng = net.engine(batch, device)
        net.bind_grads()
        self.alpha, self.eps = alpha, eps
        self.set_lr(lr)
        self.pg, self.world = process_group, world_size
        self.eng.grad_scale = 1.0 / world_size
        self.use_graph = use_graph
        # SURVEY.md section 8(f)1: reduce-scatter -> RMSprop on this rank's 1/world slice -> all-gather of the updated
        # parameters, instead of allreduce -> replicated RMSprop (same bytes on the wire, 1/world of the optimizer
        # work and state traffic per GPU).  The quantized protocol needs the full reduced gradient of every target
        # tensor before the update, so it keeps the allreduce form.
        self.shard_optimizer = bool(shard_optimizer) and world_size > 1 and quant is None
        self.rank = rank
        if self.shard_optimizer:
            from .parallel import shard_range
            self._sh0, self._sh1 = shard_range(self.eng.n_params_padded, rank, world_size)
            self._gshard = torch.zeros(self._sh1 - self._sh0, device=self.eng.device)
        self._g_fb = self._g_opt = None
        self._stage = self._staged = self._copy_stream = None     # prefetch() staging (double-buffered H2D)
        self.probe = None            # optional (name -> [start_event, end_event]) instrumentation, see bench.py

    def set_lr(self, lr):
        self.eng.lr.fill_(lr)

    def load_batch(self, img, heatmap):
        """Copy one batch into the engine's static input buffers (pinned host or device tensors)."""
        self.eng.img.copy_(img, non_blocking=True)
        self.eng.target.copy_(heatmap, non_blocking=True)

    def prefetch(self, img, heatmap):
        """Start the host -> device copy of the NEXT step's batch on a copy stream, into the staging buffers the next
        train_step() / eval_step() will consume (call it right after launching the current step: the copy then
        overlaps the step's kernels instead of preceding them).  Two staging sets alternate, so a prefetch never
        overwrites a batch that a launched step has not consumed yet."""
        e = self.eng
        if self._stage is None:
            self._copy_stream = torch.cuda.Stream(device=e.device)
            self._stage = [(torch.empty_like(e.img), torch.empty_like(e.target), torch.cuda.Event(), torch.cuda.Event())
                           for _ in range(2)]
            self._stage_next = 0
        simg, stgt, ready, consumed = self._stage[self._stage_next]
        cs = self._copy_stream
        cs.wait_event(consumed)              # the step that used this staging set two prefetches ago has read it
        with torch.cuda.stream(cs):
            simg.copy_(img, non_blocking=True)
            stgt.copy_(heatmap, non_blocking=True)
            ready.record(cs)
        self._staged = self._stage_next
        self._stage_next ^= 1

    def _consume_staged(self):
        if self._staged is None:
            return
        simg, stgt, ready, consumed = self._stage[self._staged]
        main = torch.cuda.current_stream()
        main.wait_event(ready)
        self.eng.img.copy_(simg, non_blocking=True)          # device -> device, ~20 us
        self.eng.target.copy_(stgt, non_blocking=True)
        consumed.record(main)
        self._staged = None

    def _quant_fwd(self):
        q = self.quant
        if q is not None:
            (q.binarization if hasattr(q, "binarization") else q.quantization)()

    def _quant_bwd(self):
        """restore + gradient fix-up of the quantized protocol (cu-net-prev-version-bin.py:189-190).  Runs AFTER the
        gradient allreduce, like the reference (DataParallel reduces the replica gradients inside backward(), then
        updateQuanGradWeight sees the reduced gradient): QuanOp's clip + round is not linear in the gradient."""
        q = self.quant
        if q is not None:
            q.restore()
            (q.updateBinaryGradWeight if hasattr(q, "updateBinaryGradWeight") else q.updateQuanGradWeight)()

    def _fwd_bwd(self):
        e = self.eng
        self._quant_fwd()
        e.forward(train=True)
        e.loss_and_decode(with_grad=True)
        e.backward()

    def _opt(self):
        self._quant_bwd()
        if self.shard_optimizer:
            self.eng.optimizer_step(self.alpha, self.eps, self._sh0, self._sh1, grads=self._gshard)
        else:
            self.eng.optimizer_step(self.alpha, self.eps)

    def _capture(self):
        # warm-up on a side stream (sets kernel attributes, allocates nothing afterwards), then capture.  The warm-up
        # is a real step on whatever sits in the input buffers: the model state it touches (parameters, optimizer
        # state, BatchNorm running statistics and counters) is put back, so capturing is invisible to training
        e = self.eng
        keep = e.save_state()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._fwd_bwd()
            self._opt()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        e.restore_state(keep)
        del keep
        self._g_fb = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._g_fb):
            self._fwd_bwd()
        self._g_opt = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._g_opt):
            self._opt()

    def _reduce_and_step(self):
        """Gradient exchange + optimizer: allreduce -> replicated RMSprop, or (shard_optimizer) reduce-scatter ->
        RMSprop on this rank's slice -> all-gather of the updated parameters."""
        e = self.eng
        if self.shard_optimizer:
            from .parallel import reduce_scatter_mean, all_gather_params
            reduce_scatter_mean(e.grads, self._gshard, self.world, self.pg)
        elif self.world > 1:
            from .parallel import allreduce_mean
            allreduce_mean(e.grads, self.world, self.pg)  # gradients were pre-scaled by 1/world (sum == mean)
        if self.use_graph:
            if self._g_opt is None:
                self._capture()
            self._g_opt.replay()
        else:
            self._opt()
        if self.shard_optimizer:
            all_gather_params(e.params, e.params[self._sh0:self._sh1], self.world, self.pg)

    def train_step(self, img=None, heatmap=None):
        """One training step.  Inputs: ``img`` / ``heatmap`` given (copied now, on the current stream), or staged
        earlier by prefetch(), or already resident in the engine's input buffers."""
        e = self.eng
        if img is not None:
            self._staged = None
            self.load_batch(img, heatmap)
        else:
            self._consume_staged()
        if self.use_graph:
            if self._g_fb is None:
                self._capture()
            self._g_fb.replay()
        else:
            self._fwd_bwd()
        self._reduce_and_step()
        return e.loss_value()

    def eval_step_flip(self, img=None, heatmap=None, flip_index=None):
        """validate() of the reference with its flip test-time augmentation (cu-net.py:225-249), without leaving the
        GPU: forward, multi-loss MSE of the un-flipped pass (:235-238), forward of the width-flipped image (:240-245),
        flip the last head back + swap the left/right channels (:246-247), average (:248), decode.
        Returns (loss, preds [N,C,2] of the averaged map, averaged map [N,C,H,W])."""
        from .pylib import Evaluation, HumanAug
        e = self.eng
        if img is not None:
            self.load_batch(img, heatmap)
        if flip_index is None:
            if e.plan.class_num != 16:
                raise ValueError("flip_index is required unless class_num == 16 (MPII pairs, cu-net.py:32-33)")
            flip_index = HumanAug.MPII_FLIP_INDEX
        e.forward(train=False)
        e.loss_and_decode(with_grad=False)
        loss = e.loss_value()
        out1 = e.head_outputs()[-1].float().clone()
        orig = e.img.clone()
        e.img.copy_(torch.flip(orig, dims=[3]))
        e.forward(train=False)
        out2 = HumanAug.shuffle_channels_for_horizontal_flipping(HumanAug.flip_channels(e.head_outputs()[-1]),
                                                                 flip_index)
        e.img.copy_(orig)
        avg = ((out1 + out2) / 2).contiguous()
        return loss, Evaluation.get_preds(avg), avg

    def eval_step(self, img=None, heatmap=None):
        e = self.eng
        if img is not None:
            self._staged = None
            self.load_batch(img, heatmap)
        else:
            self._consume_staged()
        e.forward(train=False)
        e.loss_and_decode(with_grad=False)
        return e.loss_value(), e.preds
