"""Execution plan for `recurrent_inference` in eval mode: the same function as
HanabiMuZeroNet.recurrent_inference_device (dynamics + reward/value/policy heads;
/root/reference/core/model.py:74-84, config/hanabi_control/model.py:199-216, 301-318), laid out for
a latency-bound batch.  A simulation is bounded by launch count, not FLOPs (SURVEY.md §7.4-9):
PyTorch's module needs ~70 kernels per call; this plan needs 7 (Hanabi-Full) / 5 (Hanabi-Small)
cuBLASLt GEMMs with fused epilogues (hz_gemm_plan, include/hzb200.h) and nothing else:

  * eval-mode BatchNorm folded into the preceding Linear;
  * the one-hot action concat of `dynamics` is literal: the batch handed over by the tree kernel is
    [hidden ‖ one-hot(action) ‖ 0-pad], so fc1 is one GEMM with K = 512 + 32;
  * bias, ReLU and the residual adds run in the GEMM epilogues (beta = 1 with C = the skip input);
  * the first layers of the three heads are one GEMM (shared input), their second layers one
    strided-batched GEMM, the three output layers one strided-batched GEMM (policy rows zero-padded);
  * value / reward logits are consumed raw by the tree kernel (hz_trees_search_step decodes them).

Weights live in fixed buffers that `refresh()` rewrites in place whenever the module's parameters
change, so chains and CUDA graphs built over a plan stay valid across training updates.
"""
import ctypes as C
import weakref

import torch

from . import _lib
from ._lib import GemmStep, check, ptr


def _fold(linear, bn):
    """Linear followed by eval-mode BatchNorm1d -> (W', b') in float32."""
    w, b = linear.weight.detach().float(), linear.bias.detach().float()
    if bn is None:
        return w, b
    scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    return w * scale[:, None], (b - bn.running_mean.detach().float()) * scale + bn.bias.detach().float()


def _pad_rows(w, b, rows):
    pad = rows - w.shape[0]
    if pad > 0:
        w = torch.cat((w, w.new_zeros(pad, w.shape[1])))
        b = torch.cat((b, b.new_zeros(pad)))
    return w, b


def _round_up(x, m):
    return (x + m - 1) // m * m


class BoundChain:
    """The plan instantiated for a fixed batch size: static activation buffers + the cuBLASLt chain."""

    def __init__(self, plan, n):
        self.plan, self.n = plan, n
        dev, dt = plan.device, plan.dtype
        F, H, KP, P3 = plan.F, plan.H, plan.KP, plan.P3
        z = lambda *shape: torch.zeros(*shape, dtype=dt, device=dev)
        self.x0 = z(n, KP)            # [hidden ‖ one-hot(action) ‖ 0]  <- written by the tree kernel
        self.y1, self.y2 = z(n, F), z(n, F)
        self.state = z(n, F)          # next hidden state (copied into the pool by the tree kernel)
        self.h1 = z(n, 3 * H)
        self.xb = z(4, n, H) if plan.full else None   # [a1, v2, r2, a2]
        self.out = z(3, n, P3)        # value logits | reward logits | policy logits (first A columns)
        w = plan._w
        steps = []

        def step(a, wt, bias, d, m, nn, k, c=None, relu=True, batch=1, sa=0, sw=0, sb=0, sc=0, sd=0, lda=None,
                 ldc=None):
            s = GemmStep()
            s.a, s.lda, s.stride_a = a.data_ptr(), (a.stride(-2) if lda is None else lda), sa
            s.w, s.ldw, s.stride_w = wt.data_ptr(), wt.stride(-2), sw
            s.bias, s.stride_bias = bias.data_ptr(), sb
            s.c, s.ldc, s.stride_c = (0 if c is None else c.data_ptr()), (0 if c is None else (c.stride(-2) if ldc is None else ldc)), sc
            s.d, s.ldd, s.stride_d = d.data_ptr(), d.stride(-2), sd
            s.m, s.n, s.k, s.batch, s.relu = m, nn, k, batch, 1 if relu else 0
            steps.append(s)

        if plan.full:
            # dynamics: relu(bn1 fc1 [s‖a]) -> relu(bn2 fc2) -> relu(bn3 fc3 + s)
            step(self.x0, w["W1"], w["b1"], self.y1, n, F, KP)
            step(self.y1, w["W2"], w["b2"], self.y2, n, F, F)
            step(self.y2, w["W3"], w["b3"], self.state, n, F, F, c=self.x0)
            # heads: [actor | value | reward] first layers, then [a1 | v2 | r2], a2 (+skip), outputs
            step(self.state, w["Wh1"], w["bh1"], self.h1, n, 3 * H, F)
            step(self.h1, w["WB2"], w["bB2"], self.xb, n, H, H, batch=3, sa=H, sw=H * H, sb=H, sd=n * H,
                 lda=3 * H)
            step(self.xb[0], w["Wa2"], w["ba2"], self.xb[3], n, H, H, c=self.h1)
            step(self.xb[1], w["WB3"], w["bB3"], self.out, n, P3, H, relu=False, batch=3, sa=n * H, sw=P3 * H,
                 sb=P3, sd=n * P3)
        else:
            # dynamics: relu(bn1 fc1 [s‖a] + s) -> relu(bn2 fc2) -> relu(bn3 fc3)
            step(self.x0, w["W1"], w["b1"], self.y1, n, F, KP, c=self.x0)
            step(self.y1, w["W2"], w["b2"], self.y2, n, F, F)
            step(self.y2, w["W3"], w["b3"], self.state, n, F, F)
            step(self.state, w["Wh1"], w["bh1"], self.h1, n, 3 * H, F)   # [value | reward | actor]
            step(self.h1, w["WB3"], w["bB3"], self.out, n, P3, H, relu=False, batch=3, sa=H, sw=P3 * H, sb=P3,
                 sd=n * P3, lda=3 * H)
        self.n_steps = len(steps)
        arr = (GemmStep * self.n_steps)(*steps)
        self._h = C.c_void_p()
        check(plan.lib.hz_gemm_plan_create(C.byref(self._h), dev.index, self.x0.element_size(), arr, self.n_steps))
        self._state_ptr = self.state.data_ptr()   # where step 2 writes / step 3 reads the new hidden state
        self._rows, self._use_rows = C.c_void_p(), False

    def rows_supported(self):
        """The row-block resident executor (hz_rowchain, include/hzb200.h) covers the fp16 plans of both networks:
        Hanabi-Full (F 512, H 256, one-hot 32) and Hanabi-Small (F 512, H 128, one-hot 16, 64 logit columns)."""
        p = self.plan
        if p.dtype != torch.float16 or p.F != 512:
            return False
        if p.full:
            return bool(p.H == 256 and p.OH == 32 and p.P3 <= 256)
        return bool(p.H == 128 and p.OH == 16 and p.P3 == 64)

    def set_executor(self, name):
        """"library": seven (Hanabi-Full) / five (Hanabi-Small) cuBLASLt launches (lowest latency for one search on an
        idle GPU).  "rows": ONE launch in which each CTA carries 128 rows through the whole chain (hz_rowchain): 1/4 of
        the SMs at 4096 rows, for searches in flight.  Same function; roundings differ in the last fp16 bits."""
        if name not in ("library", "rows"):
            raise ValueError("executor must be 'library' or 'rows'")
        if name == "rows":
            if not self.rows_supported():
                raise RuntimeError("the row-block executor needs an fp16 plan of Hanabi-Full (F=512, H=256) or "
                                   "Hanabi-Small (F=512, H=128)")
            if not self._rows:
                p, w = self.plan, self.plan._w
                ws = _lib.RowChainWeights()
                ws.w1, ws.ld_w1, ws.w1a_t, ws.b1 = w["W1"].data_ptr(), w["W1"].stride(0), w["W1aT"].data_ptr(), w["b1"].data_ptr()
                ws.w2, ws.b2, ws.w3, ws.b3 = w["W2"].data_ptr(), w["b2"].data_ptr(), w["W3"].data_ptr(), w["b3"].data_ptr()
                ws.wh1, ws.bh1 = w["Wh1"].data_ptr(), w["bh1"].data_ptr()
                if p.full:   # Hanabi-Small's heads have no second layers: those pointers stay NULL
                    ws.wb2, ws.bb2 = w["WB2"].data_ptr(), w["bB2"].data_ptr()
                    ws.wa2, ws.ba2 = w["Wa2"].data_ptr(), w["ba2"].data_ptr()
                ws.wb3, ws.bb3 = w["WB3"].data_ptr(), w["bB3"].data_ptr()
                ws.state_cols, ws.head_cols, ws.onehot_cols, ws.logit_cols = p.F, p.H, p.OH, p.P3
                create = p.lib.hz_rowchain_create if p.full else p.lib.hz_rowchain_create_small
                check(create(C.byref(self._rows), p.device.index, C.byref(ws), self.n, self.x0.data_ptr(),
                             self.x0.stride(0), self._state_ptr, self.out.data_ptr()))
        self._use_rows = name == "rows"

    def set_sm_target(self, sm_count):
        """Size the chain's library kernels for `sm_count` SMs (0 = the whole device): see hz_gemm_plan_set_sm_target."""
        check(self.plan.lib.hz_gemm_plan_set_sm_target(self._h, int(sm_count)))

    def bind_state(self, state):
        """Make the dynamics network write its output (and the heads read it) at `state` ([n, F], plan dtype,
        contiguous) instead of the chain's own buffer: the search loop passes pool[x], so no copy is needed."""
        p = state.data_ptr()
        if p != self._state_ptr:
            if state.shape != self.state.shape or state.dtype != self.state.dtype or not state.is_contiguous():
                raise ValueError("bind_state: shape/dtype/layout must match the chain's state buffer")
            check(self.plan.lib.hz_gemm_plan_set_operand(self._h, 2, 2, p))   # fc3: D
            check(self.plan.lib.hz_gemm_plan_set_operand(self._h, 3, 0, p))   # heads' first layer: A
            if self._rows:
                check(self.plan.lib.hz_rowchain_set_state(self._rows, p))
            self._state_ptr = p

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            try:
                self.plan.lib.hz_gemm_plan_destroy(h)
            except Exception:
                pass
            self._h = None
        r = getattr(self, "_rows", None)
        if r:
            try:
                self.plan.lib.hz_rowchain_destroy(r)
            except Exception:
                pass
            self._rows = C.c_void_p()

    def run(self, stream):
        if self._use_rows:
            check(self.plan.lib.hz_rowchain_run(self._rows, stream))
        else:
            check(self.plan.lib.hz_gemm_plan_run(self._h, stream, 0, self.n_steps))

    @property
    def value_logits(self):
        return self.out[0]

    @property
    def reward_logits(self):
        return self.out[1]

    @property
    def policy_logits(self):
        return self.out[2]


class RecurrentPlan:
    def __init__(self, net, dtype):
        if dtype not in (torch.float16, torch.float32):
            raise ValueError("plan dtype must be float16 or float32")
        self.net, self.dtype = net, dtype
        self.device = next(net.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("RecurrentPlan needs the module on a CUDA device (no CPU fallback)")
        self.lib = _lib.load()
        self.F, self.A, self.H, self.full = net.feature_size, net.action_space_n, net.hidden_size, net.full
        self.OH = _round_up(self.A, 16)            # one-hot columns handed over by the tree kernel
        self.KP = self.F + self.OH
        self.n_support = net._value_support.numel()
        if net._reward_support.numel() != self.n_support:
            raise ValueError("value and reward supports must have the same size")
        # 32-byte aligned logit rows (vector loads in the decode), wide enough for the policy's A logits too
        self.P3 = _round_up(max(self.n_support, self.A), 16)
        self.support = net._value_support.detach().float().contiguous()
        self._sig, self._w, self._chains = None, {}, {}
        self.refresh(force=True)

    # -- weights ---------------------------------------------------------------------------------------
    def _signature(self):
        """Identity (data_ptr) and version counter of every parameter / buffer: in-place updates (optimizer steps,
        load_state_dict, BN statistics) bump tensor._version, re-assignment (.half(), .to(), a new Parameter) changes
        the tensor object.  The modules of a network are fixed after construction, so the list of modules is cached
        and only their _parameters / _buffers dicts (where a re-assigned tensor shows up) are read per call."""
        if getattr(self, "_modules_cache", None) is None:
            self._modules_cache = list(self.net.modules())
        sig = []
        for m in self._modules_cache:
            for t in m._parameters.values():
                if t is not None:
                    sig.append((t.data_ptr(), t._version))
            for t in m._buffers.values():
                if t is not None:
                    sig.append((t.data_ptr(), t._version))
        return tuple(sig)

    def _set(self, name, value):
        value = value.to(self.dtype).contiguous()
        cur = self._w.get(name)
        if cur is None:
            self._w[name] = value.clone()
        else:
            cur.copy_(value)

    @torch.no_grad()
    def refresh(self, force=False):
        """Re-fold the module's current parameters into the plan's fixed buffers (in place)."""
        sig = self._signature()
        if not force and sig == self._sig:
            return False
        net, F, A = self.net, self.F, self.A
        d = net._dynamics_state
        w1, b1 = _fold(d.fc1, d.bn1)
        w1c = w1.new_zeros(F, self.KP)
        w1c[:, :F + A] = w1
        self._set("W1", w1c)
        self._set("W1aT", w1c[:, F:].t())          # [OH, F]: the action columns of fc1, one row per action (hz_rowchain)
        self._set("b1", b1)
        for i, (fc, bn) in ((2, (d.fc2, d.bn2)), (3, (d.fc3, d.bn3))):
            w, b = _fold(fc, bn)
            self._set(f"W{i}", w)
            self._set(f"b{i}", b)
        v, r, p = net._prediction_value, net._dynamics_reward, net._prediction_actor
        fv, fr, fp = (v[6], r[6], p[4]) if self.full else (v[3], r[3], p[3])
        order = (p, v, r) if self.full else (v, r, p)
        heads1 = [_fold(h[0], h[1]) for h in order]
        self._set("Wh1", torch.cat([w for w, _ in heads1]))
        self._set("bh1", torch.cat([b for _, b in heads1]))
        if self.full:
            second = [_fold(p[3].fc1, p[3].bn1), _fold(v[3], v[4]), _fold(r[3], r[4])]   # a1 | v2 | r2
            self._set("WB2", torch.stack([w for w, _ in second]))
            self._set("bB2", torch.stack([b for _, b in second]))
            wa2, ba2 = _fold(p[3].fc2, p[3].bn2)
            self._set("Wa2", wa2)
            self._set("ba2", ba2)
        outs = [_pad_rows(*_fold(fc, None), self.P3) for fc in (fv, fr, fp)]                # value | reward | policy
        self._set("WB3", torch.stack([w for w, _ in outs]))
        self._set("bB3", torch.stack([b for _, b in outs]))
        self._sig = sig
        return True

    # -- execution -------------------------------------------------------------------------------------
    def chain(self, n):
        """Static buffers + GEMM chain for batch size n (cached)."""
        c = self._chains.get(n)
        if c is None:
            if len(self._chains) >= 4:
                self._chains.pop(next(iter(self._chains)))
            c = self._chains[n] = BoundChain(self, n)
        return c

    @torch.no_grad()
    def run(self, hidden, action, out_state):
        """Standalone call with the module's signature: hidden [N, F], action int64 [N] or [N, 1],
        out_state [N, F] (plan dtype).  Returns (value [N], reward [N], policy_logits [N, A]) fp32.
        (The search loop does not use this: the tree kernel writes/reads the chain's buffers directly.)"""
        n = hidden.shape[0]
        ch = self.chain(n)
        st = torch.cuda.current_stream(self.device).cuda_stream
        ch.x0[:, :self.F].copy_(hidden)
        ch.x0[:, self.F:].zero_()
        ch.x0[:, self.F:].scatter_(1, action.reshape(-1, 1), 1.0)
        ch.bind_state(ch.state)
        ch.run(st)
        out_state.copy_(ch.state)
        dec = torch.empty(2 * n, dtype=torch.float32, device=self.device)
        vr = ch.out[:2].reshape(2 * n, self.P3)
        check(self.lib.hz_support_decode(st, ptr(vr), vr.element_size(), ptr(self.support), ptr(dec), 2 * n,
                                         self.n_support, self.P3, self.net.support_delta))
        return dec[:n], dec[n:], ch.policy_logits[:, :self.A].float().contiguous()


class BoundInitial:
    """InitialPlan's static buffers and GEMM chain for one (n, owner).  It owns its hz_gemm_plan (a cuBLASLt handle and
    a 32 MB device workspace), released with the object."""

    def __init__(self, lib, owner):
        self.lib, self.handle = lib, C.c_void_p()
        self._owner = None if owner is None else weakref.ref(owner)

    def owner_collected(self):
        return self._owner is not None and self._owner() is None

    def __del__(self):
        h = getattr(self, "handle", None)
        if h:
            try:
                self.lib.hz_gemm_plan_destroy(h)
            except Exception:
                pass
            self.handle = None


class InitialPlan:
    """Execution plan for `initial_inference` in eval mode (representation + policy / value heads;
    /root/reference/core/model.py:61-72, config/hanabi_control/model.py:127-335) — the per-move counterpart of
    RecurrentPlan: eval-mode BatchNorm folded, bias / ReLU / residual in the GEMM epilogues, the two heads' first layers
    one GEMM, their later layers strided batches: 10 (Hanabi-Full) / 5 (Hanabi-Small) cuBLASLt launches instead of the
    module's ~70 kernels.

    Input layout: the frame stack as [n, stack * frame_stride] with every frame padded to `frame_stride` (a multiple of
    16) values — what hz_ring_gather writes; the first layer's weight columns are spread out to the same stride (zero
    columns over the padding), so no repacking of the observation is ever needed."""

    def __init__(self, net, dtype, frame_dim, stack):
        if dtype not in (torch.float16, torch.float32):
            raise ValueError("plan dtype must be float16 or float32")
        self.net, self.dtype = net, dtype
        self.device = next(net.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("InitialPlan needs the module on a CUDA device (no CPU fallback)")
        self.lib = _lib.load()
        self.F, self.A, self.H, self.full = net.feature_size, net.action_space_n, net.hidden_size, net.full
        self.frame_dim, self.stack = int(frame_dim), int(stack)
        self.frame_stride = _round_up(self.frame_dim, 16)
        self.K0 = self.stack * self.frame_stride
        first = net._representation[0]
        if first.in_features != self.frame_dim * self.stack:
            raise ValueError(f"the network takes {first.in_features} inputs, not {self.stack} frames of {self.frame_dim}")
        self.n_support = net._value_support.numel()
        self.P3 = _round_up(max(self.n_support, self.A), 16)
        self.support = net._value_support.detach().float().contiguous()
        self._sig, self._w, self._bound = None, {}, {}
        self._modules_cache = None
        self.refresh(force=True)

    _signature = RecurrentPlan._signature
    _set = RecurrentPlan._set

    @torch.no_grad()
    def refresh(self, force=False):
        sig = self._signature()
        if not force and sig == self._sig:
            return False
        net, rep = self.net, self.net._representation
        w0, b0 = _fold(rep[0], rep[1])
        w0p = w0.new_zeros(w0.shape[0], self.K0)       # frame j's columns start at j * frame_stride
        for j in range(self.stack):
            w0p[:, j * self.frame_stride:j * self.frame_stride + self.frame_dim] = w0[:, j * self.frame_dim:(j + 1) * self.frame_dim]
        self._set("W0", w0p)
        self._set("b0", b0)
        blocks = [rep[3]] + ([rep[7]] if self.full else [])
        for i, blk in enumerate(blocks):
            for nm, (fc, bn) in (("a", (blk.fc1, blk.bn1)), ("b", (blk.fc2, blk.bn2))):
                w, b = _fold(fc, bn)
                self._set(f"Wr{i}{nm}", w)
                self._set(f"br{i}{nm}", b)
        if self.full:
            w, b = _fold(rep[4], rep[5])
            self._set("Wmid", w)
            self._set("bmid", b)
        v, p = net._prediction_value, net._prediction_actor
        order = (p, v) if self.full else (v, p)
        heads1 = [_fold(h[0], h[1]) for h in order]
        self._set("Wh1", torch.cat([w for w, _ in heads1]))
        self._set("bh1", torch.cat([b for _, b in heads1]))
        if self.full:
            second = [_fold(p[3].fc1, p[3].bn1), _fold(v[3], v[4])]      # a1 | v2
            self._set("WB2", torch.stack([w for w, _ in second]))
            self._set("bB2", torch.stack([b for _, b in second]))
            wa2, ba2 = _fold(p[3].fc2, p[3].bn2)
            self._set("Wa2", wa2)
            self._set("ba2", ba2)
            fv, fp = v[6], p[4]
        else:
            fv, fp = v[3], p[3]
        outs = [_pad_rows(*_fold(fc, None), self.P3) for fc in (fv, fp)]  # value | policy
        self._set("WB3", torch.stack([w for w, _ in outs]))
        self._set("bB3", torch.stack([b for _, b in outs]))
        self._sig = sig
        return True

    def bound(self, n, owner=None):
        """Static buffers + GEMM chain for batch size n (cached per (n, owner); `x` is the input buffer hz_ring_gather
        fills).  Callers that may run at the same time on different streams (the engines of a SelfPlayPool) pass
        themselves as `owner` and get buffers of their own.  Every call first drops the entries of owners that have been
        collected (a dead engine's buffers and GEMM plan go now, not when the cache evicts them); a remaining entry
        under id(owner) therefore belongs to `owner`, since live objects have distinct ids."""
        for k in [k for k, v in self._bound.items() if v.owner_collected()]:
            del self._bound[k]
        key = (n, None if owner is None else id(owner))
        b = self._bound.get(key)
        if b is not None:
            return b
        dev, dt, w = self.device, self.dtype, self._w
        F, H, P3 = self.F, self.H, self.P3
        z = lambda *shape: torch.zeros(*shape, dtype=dt, device=dev)
        steps = []

        def step(a, wt, bias, d, m, nn, k, c=None, relu=True, batch=1, sa=0, sw=0, sb=0, sd=0, lda=None, ldc=None):
            s = GemmStep()
            s.a, s.lda, s.stride_a = a.data_ptr(), (a.stride(-2) if lda is None else lda), sa
            s.w, s.ldw, s.stride_w = wt.data_ptr(), wt.stride(-2), sw
            s.bias, s.stride_bias = bias.data_ptr(), sb
            s.c, s.ldc, s.stride_c = (0 if c is None else c.data_ptr()), (0 if c is None else (c.stride(-2) if ldc is None else ldc)), 0
            s.d, s.ldd, s.stride_d = d.data_ptr(), d.stride(-2), sd
            s.m, s.n, s.k, s.batch, s.relu = m, nn, k, batch, 1 if relu else 0
            steps.append(s)

        b = BoundInitial(self.lib, owner)
        b.x = z(n, self.K0)
        b.state = z(n, F)
        b.h1 = z(n, 2 * H)
        b.out = z(2, n, P3)
        if self.full:
            I = self.net.init_size
            b.r1, b.t1, b.r2, b.r3, b.t2 = z(n, I), z(n, I), z(n, I), z(n, F), z(n, F)
            b.xb = z(3, n, H)                                   # [a1, v2, a2]
            step(b.x, w["W0"], w["b0"], b.r1, n, I, self.K0)
            step(b.r1, w["Wr0a"], w["br0a"], b.t1, n, I, I)
            step(b.t1, w["Wr0b"], w["br0b"], b.r2, n, I, I, c=b.r1)
            step(b.r2, w["Wmid"], w["bmid"], b.r3, n, F, I)
            step(b.r3, w["Wr1a"], w["br1a"], b.t2, n, F, F)
            step(b.t2, w["Wr1b"], w["br1b"], b.state, n, F, F, c=b.r3)
            step(b.state, w["Wh1"], w["bh1"], b.h1, n, 2 * H, F)                     # [actor | value]
            step(b.h1, w["WB2"], w["bB2"], b.xb, n, H, H, batch=2, sa=H, sw=H * H, sb=H, sd=n * H, lda=2 * H)
            step(b.xb[0], w["Wa2"], w["ba2"], b.xb[2], n, H, H, c=b.h1)
            # value logits from v2 (xb[1]), policy logits from a2 (xb[2]): consecutive batches of one strided GEMM
            step(b.xb[1], w["WB3"], w["bB3"], b.out, n, P3, H, relu=False, batch=2, sa=n * H, sw=P3 * H, sb=P3, sd=n * P3)
        else:
            b.r1, b.t1 = z(n, F), z(n, F)
            step(b.x, w["W0"], w["b0"], b.r1, n, F, self.K0)
            step(b.r1, w["Wr0a"], w["br0a"], b.t1, n, F, F, c=b.r1)                 # relu(bn1 fc1 x + x)
            step(b.t1, w["Wr0b"], w["br0b"], b.state, n, F, F)                      # relu(bn2 fc2 .)
            step(b.state, w["Wh1"], w["bh1"], b.h1, n, 2 * H, F)                     # [value | actor]
            step(b.h1, w["WB3"], w["bB3"], b.out, n, P3, H, relu=False, batch=2, sa=H, sw=P3 * H, sb=P3, sd=n * P3, lda=2 * H)
        b.n_steps = len(steps)
        arr = (GemmStep * b.n_steps)(*steps)
        check(self.lib.hz_gemm_plan_create(C.byref(b.handle), dev.index, b.x.element_size(), arr, b.n_steps))
        if len(self._bound) >= 16:
            self._bound.pop(next(iter(self._bound)))   # buffers stay alive while a caller holds the object
        self._bound[key] = b
        return b

    @torch.no_grad()
    def run(self, n, decode_value=False, owner=None):
        """Runs the chain on bound(n, owner).x (already filled).  Returns (value [n] or None, policy_logits [n, A]
        float32, hidden_state [n, F] plan dtype) — views of the plan's buffers, valid until the next run."""
        b = self.bound(n, owner)
        st = torch.cuda.current_stream(self.device).cuda_stream
        check(self.lib.hz_gemm_plan_run(b.handle, st, 0, b.n_steps))
        value = None
        if decode_value:
            value = torch.empty(n, dtype=torch.float32, device=self.device)
            check(self.lib.hz_support_decode(st, ptr(b.out[0]), b.out.element_size(), ptr(self.support), ptr(value), n,
                                             self.n_support, self.P3, self.net.support_delta))
        return value, b.out[1][:, :self.A].float(), b.state

    @torch.no_grad()
    def run_bound(self, b, logits):
        """Runs the chain of `b` (an entry of bound() the caller keeps, its x already filled) on the current stream and
        converts the policy logits into `logits` (float32 [n, A]) in place, so that a caller whose later kernels point
        at `logits` (a search slot's prepare input, wave after wave) keeps one buffer.  Returns b.state, the hidden
        states [n, F] in the plan's dtype."""
        check(self.lib.hz_gemm_plan_run(b.handle, torch.cuda.current_stream(self.device).cuda_stream, 0, b.n_steps))
        logits.copy_(b.out[1][:, :self.A])
        return b.state
