"""Adam + GradScaler for the NeRF step in two launches (row f-4 of SURVEY.md section 8: "Optimizer + AMP glue on the
12.2 M-param table"), for the NeRF network and for the edit stage's style network (row a-13).

The reference trains with `torch.optim.Adam(lr 1e-2, betas (0.9, 0.99), eps 1e-15)` under `torch.cuda.amp.GradScaler`
(main_nerf.py:223, nerf/utils.py:1474-1484) and casts the whole hash table to fp16 on every forward
(gridencoder/grid.py:43-44).  Per step that is ~610 MB of HBM traffic in six or more launches around the 49 MB table.
`AmpAdam` keeps, for every *persistent* parameter tensor,

  * a persistent fp16 shadow (what the kernels read under fp16 autocast), rewritten by the update,
  * a persistent gradient buffer the backward kernels accumulate into (cleared by the update),

and runs `lnrf_grad_nonfinite_check` + `lnrf_adam_step` + `lnrf_amp_update` (csrc/optim.cu): GradScaler's inf check,
unscale, skip-on-inf, scale growth/backoff and torch's Adam arithmetic, with no host synchronisation, so the whole
training step stays capturable in a CUDA graph.  Tensors whose gradient arrives through autograd (`p.grad`, e.g. the
two small FFMLPs and the palette of the style network) ride in the same launches.

Checkpoints: `state_dict()` has torch.optim.Adam's layout with the reference's parameter groups (`model.get_params()`:
encoder / sigma_net / encoder_dir (empty) / color_net, network_ff.py:139-153), so `torch.optim.Adam.load_state_dict`
accepts it and vice versa; the GradScaler state is separate (`scaler_state_dict()`), as in the reference's
`state['scaler']` (nerf/utils.py:1793).

Ray-sharded training (world_size > 1, SURVEY.md section 8e): the exchange step and the optimizer are fused ZeRO-1 style.
Instead of all-reduce(24.5 MB) followed by the full 367 MB Adam pass on every rank, the hash-table gradient is
REDUCE-SCATTERED (mean over ranks, fp16), every rank runs Adam on its 1/N slice of the table only (fp32 master, moments and
the slice of the fp16 shadow), and the updated fp16 shadow slices are ALL-GATHERED -- the same NVLink bytes as the
all-reduce, but the HBM-bound optimizer pass shrinks N-fold, which more than pays for the exchange.  In that mode the fp32
masters exist only as per-rank slices: the modules' fp32 parameters are refreshed from the (complete, local) fp16 shadow
whenever somebody reads them through `state_dict()` or switches the model to eval (`refresh_params()`, not a collective),
and `gather_master()` (a collective) restores the exact fp32 values for checkpoints.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import torch

from . import _native as N
from ._shadow import mark_current


class _Owner:
    """One parameter tensor of the step.  persistent = fp16 shadow + persistent gradient buffer on `module`."""
    __slots__ = ("module", "param", "lr_mult", "persistent", "group")

    def __init__(self, module, param, lr_mult=1.0, persistent=True, group=0):
        self.module, self.param, self.lr_mult, self.persistent, self.group = module, param, float(lr_mult), bool(persistent), int(group)


class AmpAdam:
    def __init__(self, model, lr=1e-2, betas=(0.9, 0.99), eps=1e-15, weight_decay=0.0, fp16=True, init_scale=2.0 ** 16,
                 growth_factor=2.0, backoff_factor=0.5, growth_interval=2000, world_size=1, rank=0, group=None, owners=None,
                 n_groups=None):
        """`owners`: None = the NeRF network (table, sigma-net, colour-net; torch.optim order of NeRFNetwork.get_params), or a list
        of (module, parameter, lr_multiplier, persistent, param_group_index).  fp16 = train under fp16 autocast with a GradScaler
        (persistent tensors get fp16 shadows and fp16 gradient buffers); fp16 = False keeps everything fp32 without a scaler."""
        self.model = model
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), (float(betas[0]), float(betas[1])), float(eps), float(weight_decay)
        self.fp16 = bool(fp16)
        self.growth_factor, self.backoff_factor, self.growth_interval = float(growth_factor), float(backoff_factor), int(growth_interval)
        self.world, self.rank, self.group = int(world_size), int(rank), group
        self.sharded = self.world > 1 and self.fp16
        if owners is None:
            # (owner module, parameter) in torch.optim order of NeRFNetwork.get_params (network_ff.py:139-153): groups 0, 1, (2 empty), 3
            self.owners = [_Owner(model.encoder, model.encoder.embeddings, group=0), _Owner(model.sigma_net, model.sigma_net.weights, group=1),
                           _Owner(model.color_net, model.color_net.weights, group=3)]
            self.n_groups = 4
        else:
            self.owners = [o if isinstance(o, _Owner) else _Owner(*o) for o in owners]
            self.n_groups = int(n_groups) if n_groups is not None else 1 + max(o.group for o in self.owners)
        if not self.fp16:
            for o in self.owners:
                o.persistent = False
        dev = self.owners[0].param.device
        if dev.type != "cuda":
            raise RuntimeError("AmpAdam: the model must live on a CUDA device (there is no CPU path)")
        self.state = []
        if self.sharded:
            if any(not o.persistent for o in self.owners):
                raise RuntimeError("AmpAdam: ray-sharded mode needs persistent (fp16 shadow) tensors only")
            self._init_sharded(dev)
        else:
            for o in self.owners:
                p = o.param
                self.state.append({"exp_avg": torch.zeros_like(p.data), "exp_avg_sq": torch.zeros_like(p.data)})
                if o.persistent:
                    o.module._shadow_f16 = p.data.half()
                    o.module._grad_f16 = torch.zeros_like(o.module._shadow_f16)
                    o.module._shadow_resync = None
                    mark_current(o.module, p)
        self.step_count = torch.ones(1, dtype=torch.float32, device=dev)       # 1-based number of the NEXT update
        self.found_inf = torch.zeros(1, dtype=torch.float32, device=dev)
        self._scale = torch.full((1,), float(init_scale), dtype=torch.float32, device=dev) if self.fp16 else None
        self._growth_tracker = torch.zeros(1, dtype=torch.int32, device=dev) if self.fp16 else None
        self.lr_scale = torch.ones(1, dtype=torch.float32, device=dev)  # schedule factor (LambdaLR), read on the device
        self._sync_words = torch.zeros(4, dtype=torch.int32, device=dev)  # grid barrier / last-block ticket of lnrf_adam_amp_step
        # one launch for check + Adam + scale update (grid barrier inside) measured 11 us SLOWER than the three launches on one B200
        # (0.425 vs 0.414 ms/step: the co-resident grid is 3 blocks per SM and the gradient is read twice); kept as an option
        self.one_launch = os.environ.get("LNRF_ADAM_ONE_LAUNCH", "0") == "1"
        self._snapshot = torch.zeros(8, dtype=torch.float32, device=dev)  # {found_inf, scale, step} of the running step + a ticket
        self.early_amp_update = os.environ.get("LNRF_EARLY_AMP_UPDATE", "1") == "1"
        self._stale_params = False
        if model is not None:
            model._amp_adam = weakref.ref(self)
            if self.sharded and hasattr(model, "register_state_dict_pre_hook"):
                # the fp32 parameters of the modules are NOT updated by the sharded step: refresh them before anybody serialises them
                self._sd_hook = model.register_state_dict_pre_hook(lambda m, prefix, keep_vars: self.refresh_params())

    # ---- ray-sharded layout -------------------------------------------------------------------------------------------
    def _init_sharded(self, dev):
        """One flat parameter vector [table | sigma-net weights | colour-net weights | pad] whose [lo, hi) slice this rank owns:
        the fp32 master and the Adam moments exist for that slice only; the fp16 shadow and the fp16 gradient exist in full on
        every rank and the modules' `_shadow_f16` / `_grad_f16` are views of them.  With torch symmetric memory the two flat
        fp16 vectors are peer-mapped and the whole exchange is one kernel (lnrf_adam_step_sharded); otherwise NCCL
        reduce-scatter / all-gather move the same bytes."""
        sizes = [o.param.numel() for o in self.owners]
        T = sum(sizes)
        unit = self.world * 8  # every slice a multiple of 8 elements: 16-byte fp16 vectors
        self.P, self.P_pad = T, (T + unit - 1) // unit * unit
        self.Sz = self.P_pad // self.world
        self.lo, self.hi = self.rank * self.Sz, (self.rank + 1) * self.Sz
        self._sizes = sizes
        flat32 = self._flat_from_params(dev)
        self.p2p = None
        if os.environ.get("LNRF_P2P", "1") == "1":
            try:
                self.p2p = self._init_symmetric(dev)
            except Exception as e:  # never silently: bench.py reports which exchange path ran
                self.p2p_error = f"{type(e).__name__}: {e}"[:300]
                self.p2p = None
                self.__dict__.pop("_grad_bufs", None)
        if self.p2p is None:
            self.shadow_flat = torch.empty(self.P_pad, dtype=torch.half, device=dev)
            self.grad_flat = torch.zeros(self.P_pad, dtype=torch.half, device=dev)
            self.grad_shard = torch.zeros(self.Sz, dtype=torch.half, device=dev)
        self.shadow_flat.copy_(flat32)
        self.master_shard = flat32[self.lo:self.hi].clone()
        del flat32
        self._phase = None        # None: one gradient buffer, closing clear (every eager step); 0 / 1: pipelined, see select_phase
        self._dirty_buf = None    # pipelined: the buffer the last step left for the NEXT step's kernel to clear
        self._grad_views = [[], []]
        off = 0
        for o, n in zip(self.owners, sizes):
            o.module._shadow_f16 = self.shadow_flat[off:off + n].view_as(o.param)
            for b_, buf in enumerate(getattr(self, "_grad_bufs", [self.grad_flat])):
                self._grad_views[b_].append(buf[off:off + n].view_as(o.param))
            o.module._grad_f16 = self.grad_flat[off:off + n].view_as(o.param)
            o.module._shadow_resync = self._resync_from_params  # an outside write to ANY fp32 parameter re-derives shadow + master slice
            mark_current(o.module, o.param)
            off += n
        # ONE state entry in sharded mode: the moments of this rank's slice of the flat vector
        self.state.append({"exp_avg": torch.zeros(self.Sz, dtype=torch.float32, device=dev),
                           "exp_avg_sq": torch.zeros(self.Sz, dtype=torch.float32, device=dev)})

    @property
    def can_pipeline(self) -> bool:
        """Two peer-mapped gradient buffers exist (symmetric memory, barrier-bracketed exchange): steps may alternate between them."""
        return bool(self.sharded and self.p2p is not None and not self.inkernel_sync and len(getattr(self, "_grad_bufs", [])) == 2)

    def select_phase(self, phase):
        """Software-pipelined sharded training (GraphedTrainStep(lookahead=True) at world_size > 1): consecutive steps accumulate into
        alternating gradient buffers, so the exchange kernel of a step can clear the buffer of the step before it -- no closing
        "clear + scale update" launch, no flag memset (csrc/optim.cu ExchangeExtra).  phase 0 / 1: the modules' `_grad_f16` point into
        that buffer and step() takes the pipelined path; None: back to one buffer with the closing clear."""
        if phase is not None and not self.can_pipeline:
            raise RuntimeError("select_phase: needs the symmetric-memory exchange with barrier launches")
        self._phase = phase
        b_ = 0 if phase is None else int(phase)
        self.grad_flat = self._grad_bufs[b_] if hasattr(self, "_grad_bufs") else self.grad_flat
        for o, v in zip(self.owners, self._grad_views[b_]):
            o.module._grad_f16 = v

    def _settle_buffers(self):
        """Eager step after pipelined ones: the buffer the last pipelined step filled was to be cleared by its successor."""
        if self._dirty_buf is not None:
            self._grad_bufs[self._dirty_buf].zero_()
            self.flag_buf[:8].zero_()
            self._dirty_buf = None

    def _flat_from_params(self, dev):
        flat = torch.zeros(self.P_pad, dtype=torch.float32, device=dev)
        off = 0
        for o, n in zip(self.owners, self._sizes):
            flat[off:off + n] = o.param.data.reshape(-1)
            off += n
        return flat

    def _init_symmetric(self, dev):
        """Peer-mapped gradient / shadow / flag buffers (torch.distributed._symmetric_memory): returns the handles and the
        per-rank device pointers the fused kernel dereferences over NVLink."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        group = self.group if self.group is not None else dist.group.WORLD
        bufs, hdls = {}, {}
        for name, numel, dt in (("grad", self.P_pad, torch.half), ("shadow", self.P_pad, torch.half), ("flag", 32, torch.float32),
                                ("grad_b", self.P_pad, torch.half)):  # grad_b: the second buffer of the software-pipelined step (select_phase)
            t = symm.empty(numel, dtype=dt, device=dev)
            hdls[name] = symm.rendezvous(t, group)
            bufs[name] = t
        self.grad_flat, self.shadow_flat, self.flag_buf = bufs["grad"], bufs["shadow"], bufs["flag"]
        self._grad_bufs = [bufs["grad"], bufs["grad_b"]]
        self.grad_flat.zero_()
        bufs["grad_b"].zero_()
        self.flag_buf.zero_()
        ptrs = {k: [int(x) for x in hdls[k].buffer_ptrs] for k in hdls}
        if any(len(v) != self.world or not all(v) for v in ptrs.values()):
            raise RuntimeError(f"symmetric memory rendezvous returned {ptrs}")
        mk = lambda v: (C.c_void_p * self.world)(*v)
        self._peer_arrays = (mk(ptrs["grad"]), mk(ptrs["shadow"]), mk(ptrs["flag"]))
        # phase 1 of the pipelined step: the second gradient buffer, flag word 4 of every rank's flag buffer (word 0 is phase 0's)
        self._peer_arrays_b = (mk(ptrs["grad_b"]), self._peer_arrays[1], mk([x + 16 for x in ptrs["flag"]]))
        # LNRF_INKERNEL_SYNC=1: rank synchronisation inside the exchange kernels instead of symmetric-memory barrier launches
        self.inkernel_sync = os.environ.get("LNRF_INKERNEL_SYNC", "0") == "1" and self.world <= 8
        self._sync_state = torch.zeros(2, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        hdls["grad"].barrier(channel=0)
        return hdls

    # ---- optional timing of the exchange pieces (diagnostics; never inside graph capture) --------------------------
    def _mark(self, name):
        if os.environ.get("LNRF_TIME_EXCHANGE", "0") != "1" or torch.cuda.is_current_stream_capturing():
            return
        if not hasattr(self, "_marks"):
            self._marks = []
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self._marks.append((name, e))

    def exchange_timing(self):
        """Mean microseconds between consecutive marks of _step_sharded over the eager steps run so far (LNRF_TIME_EXCHANGE=1)."""
        marks = getattr(self, "_marks", [])
        torch.cuda.synchronize()
        acc, cnt = {}, {}
        for (n0, e0), (n1, e1) in zip(marks, marks[1:]):
            if n1 == "start":
                continue
            acc[n1] = acc.get(n1, 0.0) + e0.elapsed_time(e1) * 1e3
            cnt[n1] = cnt.get(n1, 0) + 1
        return {k: acc[k] / cnt[k] for k in acc}

    # ---- GradScaler surface -------------------------------------------------------------------------------------
    def scale(self, loss):
        return loss * self._scale if self.fp16 else loss

    def get_scale(self) -> float:
        return float(self._scale.item()) if self.fp16 else 1.0

    def grads(self):
        """The gradient tensors the next step() will consume (the all-reduce of ray-sharded training acts on these)."""
        out = []
        for o in self.owners:
            g = o.module._grad_f16 if o.persistent else o.param.grad
            if g is not None:
                out.append(g)
        return out

    def zero_grad(self, set_to_none=True):
        for o in self.owners:
            if not o.persistent:
                o.param.grad = None  # autograd allocates; the update kernel has consumed them

    def _descriptors(self, owners, states):
        arr = (N.OptTensor * len(owners))()
        keep = []
        for i, (o, st) in enumerate(zip(owners, states)):
            p = o.param
            g = o.module._grad_f16 if o.persistent else p.grad
            if g is None:
                raise RuntimeError("AmpAdam.step(): a parameter has no gradient (call backward first)")
            if o.persistent and p.grad is not None:
                raise RuntimeError("AmpAdam.step(): a persistent parameter received an autograd .grad -- under fp16 autocast the kernels "
                                   "accumulate into its fp16 buffer (NeRFNetwork.fused = True / GridEncoder with a shadow); a module path that "
                                   "bypasses them was used")
            g = g.contiguous()
            keep.append(g)
            arr[i].params, arr[i].exp_avg, arr[i].exp_avg_sq = p.data.data_ptr(), st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr()
            arr[i].grad = g.data_ptr()
            arr[i].params_f16 = o.module._shadow_f16.data_ptr() if o.persistent else None
            arr[i].n = p.numel()
            if g.dtype not in (torch.float16, torch.float32):
                raise RuntimeError(f"AmpAdam.step(): unsupported gradient dtype {g.dtype}")
            arr[i].grad_dtype = N.F16 if g.dtype == torch.float16 else N.F32
        return arr, keep

    def _one(self, params, st, grad, shadow, n):
        arr = (N.OptTensor * 1)()
        arr[0].params, arr[0].exp_avg, arr[0].exp_avg_sq = N.ptr(params), N.ptr(st["exp_avg"]) if st else None, N.ptr(st["exp_avg_sq"]) if st else None
        arr[0].grad, arr[0].params_f16, arr[0].n, arr[0].grad_dtype = grad.data_ptr(), N.ptr(shadow), n, N.F16
        return arr

    @torch.no_grad()
    def _step_sharded(self):
        """world_size > 1: exchange + Adam on this rank's slice + broadcast of the new fp16 values (see the module docstring)."""
        import torch.distributed as dist
        lib, st = N.lib(), N.stream()
        hyper = (self.lr, self.betas[0], self.betas[1], self.eps, self.weight_decay)
        self._stale_params = True
        if self.p2p is not None:
            # own gradient checked locally, flag published beside it; barrier; ONE kernel averages the R gradients of the slice
            # over NVLink, updates, and writes the new fp16 slice into every rank's table; barrier; clear the local gradient
            mark = self._mark  # LNRF_TIME_EXCHANGE=1: CUDA events between the pieces (eager steps only), see exchange_timing()
            mark("start")
            if self._phase is not None:
                # pipelined: inf check (+ snapshot of scale / step) -> barrier -> ONE kernel: exchange + Adam + table broadcast + clear of
                # the OTHER gradient buffer and flag + GradScaler.update() -> barrier.  4 launches (6 on the one-buffer path below).
                ph = self._phase
                g, sh, fl = self._peer_arrays if ph == 0 else self._peer_arrays_b
                my_flag = self.flag_buf.data_ptr() + 16 * ph
                other = self._grad_bufs[1 - ph]
                N.check(lib.lnrf_grad_nonfinite_check_snapshot(C.cast(self._one(None, None, self._grad_bufs[ph], None, self.P_pad), C.c_void_p), 1,
                                                               my_flag, N.ptr(self._scale), N.ptr(self.step_count), N.ptr(self._snapshot), st))
                self.p2p["grad"].barrier(channel=0)
                N.check(lib.lnrf_adam_step_sharded_pipelined(
                    C.cast(g, C.c_void_p), C.cast(sh, C.c_void_p), C.cast(fl, C.c_void_p), self.world, self.lo, self.Sz, N.ptr(self.master_shard),
                    N.ptr(self.state[0]["exp_avg"]), N.ptr(self.state[0]["exp_avg_sq"]), *hyper, N.ptr(self._snapshot), N.ptr(self.lr_scale),
                    other.data_ptr(), self.P_pad, self.flag_buf.data_ptr() + 16 * (1 - ph), N.ptr(self._scale), N.ptr(self._growth_tracker),
                    N.ptr(self.found_inf), N.ptr(self.step_count), self.growth_factor, self.backoff_factor, self.growth_interval, st))
                self.p2p["grad"].barrier(channel=1)
                self._dirty_buf = ph
                return
            self._settle_buffers()
            if self.inkernel_sync:
                # the ranks meet INSIDE the kernels (signal + poll on the peer-mapped flag words, csrc/optim.cu): no barrier launches,
                # and the closing wait clears the gradient -- 3 launches instead of 6
                self.flag_buf[:1].zero_()  # word 0 only: the other words carry the epochs of the synchronisation
                N.check(lib.lnrf_grad_nonfinite_check(C.cast(self._one(None, None, self.grad_flat, None, self.P_pad), C.c_void_p), 1,
                                                      N.ptr(self.flag_buf), st))
                mark("inf check")
                g, sh, fl = self._peer_arrays
                N.check(lib.lnrf_adam_step_sharded_sync(C.cast(g, C.c_void_p), C.cast(sh, C.c_void_p), C.cast(fl, C.c_void_p), self.world,
                                                        self.rank, self.lo, self.Sz, N.ptr(self.master_shard),
                                                        N.ptr(self.state[0]["exp_avg"]), N.ptr(self.state[0]["exp_avg_sq"]), *hyper,
                                                        N.ptr(self._scale), N.ptr(self.found_inf), N.ptr(self.step_count),
                                                        N.ptr(self.lr_scale), N.ptr(self._sync_state), st))
                mark("exchange + Adam kernel (arrive sync inside)")
                N.check(lib.lnrf_exchange_finish(N.ptr(self.flag_buf), self.world, N.ptr(self._sync_state), N.ptr(self.grad_flat), self.P_pad, st))
                mark("done sync + gradient clear")
                N.check(lib.lnrf_amp_update(N.ptr(self._scale), N.ptr(self._growth_tracker), N.ptr(self.found_inf), N.ptr(self.step_count),
                                            self.growth_factor, self.backoff_factor, self.growth_interval, st))
                return
            self.flag_buf.zero_()
            N.check(lib.lnrf_grad_nonfinite_check(C.cast(self._one(None, None, self.grad_flat, None, self.P_pad), C.c_void_p), 1,
                                                  N.ptr(self.flag_buf), st))
            mark("inf check")
            self.p2p["grad"].barrier(channel=0)
            mark("barrier A")
            g, sh, fl = self._peer_arrays
            N.check(lib.lnrf_adam_step_sharded(C.cast(g, C.c_void_p), C.cast(sh, C.c_void_p), C.cast(fl, C.c_void_p), self.world, self.lo,
                                               self.Sz, N.ptr(self.master_shard), N.ptr(self.state[0]["exp_avg"]),
                                               N.ptr(self.state[0]["exp_avg_sq"]), *hyper, N.ptr(self._scale), N.ptr(self.found_inf),
                                               N.ptr(self.step_count), N.ptr(self.lr_scale), st))
            mark("exchange + Adam kernel")
            self.p2p["grad"].barrier(channel=1)
            mark("barrier B")
            # gradient clear + GradScaler.update() in one launch
            N.check(lib.lnrf_exchange_tail(N.ptr(self.grad_flat), self.P_pad, N.ptr(self._scale), N.ptr(self._growth_tracker), N.ptr(self.found_inf),
                                           N.ptr(self.step_count), self.growth_factor, self.backoff_factor, self.growth_interval, st))
            mark("gradient clear + amp update")
            return
        else:
            nccl = dist.get_backend(self.group) == "nccl"
            if nccl:  # mean inside the collective (pre-scaled sum: no fp16 overflow from adding `world` loss-scaled gradients)
                dist.reduce_scatter_tensor(self.grad_shard, self.grad_flat, op=dist.ReduceOp.AVG, group=self.group)
            else:     # gloo (CPU tests of the host logic): sum, slice, divide
                dist.all_reduce(self.grad_flat, op=dist.ReduceOp.SUM, group=self.group)
                self.grad_shard.copy_(self.grad_flat[self.lo:self.hi])
                self.grad_shard.div_(self.world)
            self.grad_flat.zero_()
            arr = self._one(self.master_shard, self.state[0], self.grad_shard, self.shadow_flat[self.lo:self.hi], self.Sz)
            N.check(lib.lnrf_grad_nonfinite_check(C.cast(arr, C.c_void_p), 1, N.ptr(self.found_inf), st))
            dist.all_reduce(self.found_inf, op=dist.ReduceOp.MAX, group=self.group)  # an inf may sit in another rank's slice only
            N.check(lib.lnrf_adam_step(C.cast(arr, C.c_void_p), 1, *hyper, N.ptr(self._scale), N.ptr(self.found_inf), N.ptr(self.step_count),
                                       N.ptr(self.lr_scale), st))
            dist.all_gather_into_tensor(self.shadow_flat, self.shadow_flat[self.lo:self.hi], group=self.group)
        N.check(lib.lnrf_amp_update(N.ptr(self._scale), N.ptr(self._growth_tracker), N.ptr(self.found_inf), N.ptr(self.step_count),
                                    self.growth_factor, self.backoff_factor, self.growth_interval, st))

    def _allreduce_autograd_grads(self):
        """world_size > 1 without fp16 sharding (e.g. the fp32 style network): plain mean all-reduce of every gradient."""
        import torch.distributed as dist
        for g in self.grads():
            dist.all_reduce(g, op=dist.ReduceOp.SUM, group=self.group)
            g.div_(self.world)

    @torch.no_grad()
    def step(self):
        N.join_pending()  # e.g. the weight-gradient reduction of the fused network, queued on a side stream beside the encoder backward
        if self.sharded:
            return self._step_sharded()
        if self.world > 1:
            self._allreduce_autograd_grads()
        lib = N.lib()
        st = N.stream()
        arr, keep = self._descriptors(self.owners, self.state)
        n = len(self.owners)
        if self.fp16 and self.one_launch and len({o.lr_mult for o in self.owners}) == 1:
            # non-finite check + Adam + GradScaler.update() in ONE launch (csrc/optim.cu k_adam_amp_fused)
            N.check(lib.lnrf_adam_amp_step(C.cast(arr, C.c_void_p), n, self.lr * self.owners[0].lr_mult, self.betas[0], self.betas[1], self.eps,
                                           self.weight_decay, N.ptr(self._scale), N.ptr(self._growth_tracker), N.ptr(self.found_inf),
                                           N.ptr(self.step_count), N.ptr(self.lr_scale), self.growth_factor, self.backoff_factor,
                                           self.growth_interval, N.ptr(self._sync_words), st))
            del keep
            return
        scale_p, found_p, count_p = N.ptr(self._scale), N.ptr(self.found_inf), N.ptr(self.step_count)
        early_update = self.fp16 and self.early_amp_update
        if early_update:
            # non-finite check + GradScaler.update() in one launch AHEAD of Adam, which then reads the frozen {found_inf, scale, step}
            # of this step from the snapshot (csrc/optim.cu k_grad_nonfinite_amp): one launch fewer on the step's critical path
            N.check(lib.lnrf_grad_nonfinite_check_amp_update(C.cast(arr, C.c_void_p), n, scale_p, N.ptr(self._growth_tracker), found_p, count_p,
                                                             self.growth_factor, self.backoff_factor, self.growth_interval,
                                                             N.ptr(self._snapshot), st))
            base = self._snapshot.data_ptr()
            found_p, scale_p, count_p = base, base + 4, base + 8
        elif self.fp16:
            N.check(lib.lnrf_grad_nonfinite_check(C.cast(arr, C.c_void_p), n, N.ptr(self.found_inf), st))
        # one launch per distinct learning rate (the style network trains its palette at 2 x lr, style_encoder.py:247-255)
        for mult in sorted({o.lr_mult for o in self.owners}):
            idx = [i for i, o in enumerate(self.owners) if o.lr_mult == mult]
            if len(idx) == n:
                sub = arr
            else:
                sub, _k = self._descriptors([self.owners[i] for i in idx], [self.state[i] for i in idx])
                keep += _k
            N.check(lib.lnrf_adam_step(C.cast(sub, C.c_void_p), len(idx), self.lr * mult, self.betas[0], self.betas[1], self.eps, self.weight_decay,
                                       scale_p, found_p, count_p, N.ptr(self.lr_scale), st))
        if not early_update:
            N.check(lib.lnrf_amp_update(N.ptr(self._scale), N.ptr(self._growth_tracker), N.ptr(self.found_inf), N.ptr(self.step_count),
                                        self.growth_factor, self.backoff_factor, self.growth_interval, st))
        del keep

    # ---- sharded mode: where the fp32 parameters live ----------------------------------------------------------------
    def _gather_flat(self, shard):
        import torch.distributed as dist
        full = torch.empty(self.P_pad, dtype=shard.dtype, device=shard.device)
        dist.all_gather_into_tensor(full, shard.contiguous(), group=self.group)
        return full

    def _split_flat(self, full):
        out, off = [], 0
        for o, n in zip(self.owners, self._sizes):
            out.append(full[off:off + n].view_as(o.param))
            off += n
        return out

    def _write_params(self, tensors):
        for o, t in zip(self.owners, tensors):
            o.param.data.copy_(t)
            mark_current(o.module, o.param)  # our own write: the shadow is (still) the truth
        self._stale_params = False

    @torch.no_grad()
    def refresh_params(self):
        """Sharded mode, NOT a collective: bring the modules' fp32 parameters up to date from this rank's complete fp16 shadow
        (the values every kernel reads; fp16-rounded).  Runs automatically before `model.state_dict()` and on `model.eval()`.
        For the exact fp32 masters use gather_master()."""
        if not self.sharded or not self._stale_params:
            return
        self._resync_if_params_changed()
        self._write_params([o.module._shadow_f16 for o in self.owners])

    @torch.no_grad()
    def gather_master(self):
        """Sharded mode (collective): bring the fp32 masters of every slice back into the modules' parameters (checkpoints)."""
        if not self.sharded:
            return
        self._resync_if_params_changed()
        self._write_params(self._split_flat(self._gather_flat(self.master_shard)))

    def _resync_if_params_changed(self):
        if any(o.param._version != getattr(o.module, "_shadow_version", None) for o in self.owners if o.persistent):
            self.sync_shadows()

    @torch.no_grad()
    def _resync_from_params(self):
        """Sharded mode: the fp32 parameters were written from outside (load_state_dict, manual edit): they are the truth now."""
        for o in self.owners:
            o.module._shadow_f16.copy_(o.param.data)
            mark_current(o.module, o.param)
        self.master_shard.copy_(self._flat_from_params(self.master_shard.device)[self.lo:self.hi])
        self._stale_params = False

    @torch.no_grad()
    def sync_shadows(self):
        """Re-derive the fp16 shadows (and, sharded, this rank's master slice) from the fp32 parameters.  Happens by itself when a
        parameter was written through torch (see _shadow.py); call it after writing through raw pointers."""
        if self.sharded:
            return self._resync_from_params()
        for o in self.owners:
            if o.persistent:
                o.module._shadow_f16.copy_(o.param.data)
                mark_current(o.module, o.param)

    def detach(self):
        """Give the modules back to the plain torch path (drops the shadows and persistent gradient buffers)."""
        if self.sharded:
            self.refresh_params()
        for o in self.owners:
            if o.persistent:
                o.module._shadow_f16 = o.module._grad_f16 = None
                o.module._shadow_resync = None
        if self.model is not None and getattr(self.model, "_amp_adam", None) is not None and self.model._amp_adam() is self:
            self.model._amp_adam = None
        hook = getattr(self, "_sd_hook", None)
        if hook is not None:
            hook.remove()
            self._sd_hook = None

    # ---- torch.optim.Adam-compatible checkpoint layout ------------------------------------------------------------
    def state_dict(self):
        """torch.optim.Adam's layout with the reference's parameter groups.  Sharded mode: a collective (every rank calls it)."""
        step = float(self.step_count.item()) - 1.0
        if self.sharded:  # the moments are gathered back into the per-parameter layout
            ea = self._split_flat(self._gather_flat(self.state[0]["exp_avg"]))
            es = self._split_flat(self._gather_flat(self.state[0]["exp_avg_sq"]))
        else:
            ea = [st["exp_avg"] for st in self.state]
            es = [st["exp_avg_sq"] for st in self.state]
        state = {i: {"step": torch.tensor(step), "exp_avg": ea[i], "exp_avg_sq": es[i]} for i in range(len(self.owners))}
        groups = []
        for gi in range(self.n_groups):
            idx = [i for i, o in enumerate(self.owners) if o.group == gi]
            mult = self.owners[idx[0]].lr_mult if idx else 1.0
            groups.append({"lr": self.lr * mult, "betas": self.betas, "eps": self.eps, "weight_decay": self.weight_decay, "amsgrad": False,
                           "maximize": False, "foreach": None, "capturable": False, "differentiable": False, "fused": None,
                           "decoupled_weight_decay": False, "params": idx})
        return {"state": state, "param_groups": groups}

    def scaler_state_dict(self):
        """torch.amp.GradScaler.state_dict() layout (the reference stores it beside the optimizer's, nerf/utils.py:1793)."""
        if not self.fp16:
            return {}
        return {"scale": self.get_scale(), "growth_factor": self.growth_factor, "backoff_factor": self.backoff_factor,
                "growth_interval": self.growth_interval, "_growth_tracker": int(self._growth_tracker.item())}

    def load_scaler_state_dict(self, sd):
        if self.fp16 and sd:
            self._scale.fill_(float(sd["scale"]))
            self._growth_tracker.fill_(int(sd["_growth_tracker"]))
            self.growth_factor, self.backoff_factor = float(sd["growth_factor"]), float(sd["backoff_factor"])
            self.growth_interval = int(sd["growth_interval"])

    def load_state_dict(self, sd):
        """Accepts this class's state_dict() and torch.optim.Adam's (full per-parameter tensors in both).  The fp32 parameters
        themselves are not part of an optimizer checkpoint: if the caller loaded the MODEL beforehand, the shadows (and the sharded
        master slice) follow that write by themselves (_shadow.py); nothing is derived from parameters that were not touched."""
        n = len(self.owners)
        if len(sd["state"]) not in (0, n):
            raise RuntimeError(f"AmpAdam.load_state_dict: {len(sd['state'])} state entries for {n} parameter tensors")
        if len(sd["state"]) == n:
            if self.sharded:
                for k in ("exp_avg", "exp_avg_sq"):
                    flat = torch.zeros(self.P_pad, dtype=torch.float32, device=self.master_shard.device)
                    off = 0
                    for i, cnt in enumerate(self._sizes):
                        flat[off:off + cnt] = sd["state"][i][k].reshape(-1)
                        off += cnt
                    self.state[0][k].copy_(flat[self.lo:self.hi])
            else:
                for i, st in enumerate(self.state):
                    src = sd["state"][i]
                    st["exp_avg"].copy_(src["exp_avg"])
                    st["exp_avg_sq"].copy_(src["exp_avg_sq"])
            self.step_count.fill_(float(sd["state"][0]["step"]) + 1.0)
        g = next((g for g in sd["param_groups"] if g["params"]), sd["param_groups"][0])
        first = self.owners[g["params"][0]].lr_mult if g["params"] else 1.0
        self.lr = float(g["lr"]) / first
        self.betas, self.eps, self.weight_decay = tuple(map(float, g["betas"])), float(g["eps"]), float(g["weight_decay"])
        if "scaler" in sd:  # round-1 checkpoints nested the scaler state here
            self.load_scaler_state_dict(sd["scaler"])
        self._resync_if_params_changed()


class ShardedFlatAdam(AmpAdam):
    """Data-parallel Adam + GradScaler for a network trained in fp32 without fp16 shadows (the edit-stage style network, row a-13),
    sharded ZeRO-1 style over torch symmetric memory.

    The parameters of all owners are views of ONE flat fp32 vector (each tensor starts on a multiple of 8 elements, the vector is
    padded to a multiple of 8 x world), peer-mapped on every rank; so is the flat fp32 gradient vector.  Owners with `persistent` set
    accumulate into it from their kernels (GridEncoder's `_grad_f32`: the 49 MB table gradient is never copied); the gradients of the
    others arrive through autograd and are copied into their place by step() (the two small nets and the palette: ~10 K values).
    step() = inf check of the local gradient (flag published beside it) -> barrier -> ONE kernel (lnrf_adam_step_sharded_f32): this
    rank averages the R gradients of its slice in rank order, runs Adam on it with per-owner learning rates and stores the new values
    into every rank's parameter vector -> barrier -> gradient clear + GradScaler.update().  Adam moments exist for the slice only.
    No host synchronisation, so the step can be captured in a CUDA graph.

    world_size = 1 needs no process group: the vectors are ordinary device memory and the only peer is the rank itself.  Construction
    raises when the symmetric-memory rendezvous fails; nothing has been re-pointed then."""

    def __init__(self, owners, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, init_scale=2.0 ** 16, growth_factor=2.0,
                 backoff_factor=0.5, growth_interval=2000, world_size=1, rank=0, group=None, n_groups=None):
        self.model = None
        self.lr, self.betas, self.eps, self.weight_decay = float(lr), (float(betas[0]), float(betas[1])), float(eps), float(weight_decay)
        self.fp16, self.sharded = True, False
        self.growth_factor, self.backoff_factor, self.growth_interval = float(growth_factor), float(backoff_factor), int(growth_interval)
        self.world, self.rank, self.group = int(world_size), int(rank), group
        self.owners = [o if isinstance(o, _Owner) else _Owner(*o) for o in owners]
        self.n_groups = int(n_groups) if n_groups is not None else 1 + max(o.group for o in self.owners)
        dev = self.owners[0].param.device
        if dev.type != "cuda":
            raise RuntimeError("ShardedFlatAdam: the parameters must live on a CUDA device (there is no CPU path)")
        if any(o.param.dtype != torch.float32 for o in self.owners):
            raise RuntimeError("ShardedFlatAdam: fp32 parameters only")
        self._offsets, off = [], 0
        for o in self.owners:
            self._offsets.append(off)
            off += (o.param.numel() + 7) // 8 * 8
        unit = 8 * self.world
        self.P_pad = (off + unit - 1) // unit * unit
        self.Sz = self.P_pad // self.world
        self.lo, self.hi = self.rank * self.Sz, (self.rank + 1) * self.Sz
        # learning-rate segments: runs of owners with the same multiplier
        starts, mults = [], []
        for o, o_off in zip(self.owners, self._offsets):
            if not mults or mults[-1] != o.lr_mult:
                starts.append(o_off)
                mults.append(o.lr_mult)
        if len(starts) > 8:
            raise RuntimeError("ShardedFlatAdam: at most 8 learning-rate segments")
        self._seg_start, self._seg_mult = (C.c_uint64 * len(starts))(*starts), (C.c_double * len(mults))(*mults)
        self.p2p = None
        if self.world > 1:
            self._init_symmetric(dev)
        else:
            self.param_flat = torch.zeros(self.P_pad, dtype=torch.float32, device=dev)
            self.grad_flat = torch.zeros(self.P_pad, dtype=torch.float32, device=dev)
            self.flag_buf = torch.zeros(32, dtype=torch.float32, device=dev)
            self._peer_arrays = tuple((C.c_void_p * 1)(t.data_ptr()) for t in (self.grad_flat, self.param_flat, self.flag_buf))
        # re-point every parameter into the flat vector (a leaf stays the same leaf: the palette is a plain tensor, not an nn.Parameter)
        self._grad_views = []
        with torch.no_grad():
            for o, o_off in zip(self.owners, self._offsets):
                n = o.param.numel()
                view = self.param_flat[o_off:o_off + n].view_as(o.param)
                view.copy_(o.param)
                o.param.set_(view)
                gview = self.grad_flat[o_off:o_off + n].view_as(o.param)
                self._grad_views.append(gview)
                if o.persistent:
                    o.module._grad_f32 = gview
        if self.world > 1:
            torch.cuda.synchronize()
            self.p2p["grad"].barrier(channel=0)
        self.state = [{"exp_avg": torch.zeros(self.Sz, dtype=torch.float32, device=dev),
                       "exp_avg_sq": torch.zeros(self.Sz, dtype=torch.float32, device=dev)}]
        self.step_count = torch.ones(1, dtype=torch.float32, device=dev)
        self.found_inf = torch.zeros(1, dtype=torch.float32, device=dev)
        self._scale = torch.full((1,), float(init_scale), dtype=torch.float32, device=dev)
        self._growth_tracker = torch.zeros(1, dtype=torch.int32, device=dev)
        self.lr_scale = torch.ones(1, dtype=torch.float32, device=dev)

    def _init_symmetric(self, dev):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        group = self.group if self.group is not None else dist.group.WORLD
        bufs, hdls = {}, {}
        for name, numel in (("grad", self.P_pad), ("param", self.P_pad), ("flag", 32)):
            t = symm.empty(numel, dtype=torch.float32, device=dev)
            hdls[name] = symm.rendezvous(t, group)
            bufs[name] = t
        ptrs = {k: [int(x) for x in hdls[k].buffer_ptrs] for k in hdls}
        if any(len(v) != self.world or not all(v) for v in ptrs.values()):
            raise RuntimeError(f"symmetric memory rendezvous returned {ptrs}")
        self.grad_flat, self.param_flat, self.flag_buf = bufs["grad"], bufs["param"], bufs["flag"]
        self.grad_flat.zero_()
        self.param_flat.zero_()
        self.flag_buf.zero_()
        self._peer_arrays = tuple((C.c_void_p * self.world)(*ptrs[k]) for k in ("grad", "param", "flag"))
        self.p2p = hdls

    def grads(self):
        return [self.grad_flat]

    def zero_grad(self, set_to_none=True):
        for o in self.owners:
            if not o.persistent:
                o.param.grad = None

    @torch.no_grad()
    def step(self):
        N.join_pending()
        lib, st = N.lib(), N.stream()
        for o, gview in zip(self.owners, self._grad_views):
            if o.persistent:
                continue
            if o.param.grad is None:
                raise RuntimeError("ShardedFlatAdam.step(): a parameter has no gradient (call backward first)")
            gview.copy_(o.param.grad)
        self.flag_buf[:1].zero_()
        N.check(lib.lnrf_grad_nonfinite_check(C.cast(self._one_f32(self.grad_flat), C.c_void_p), 1, N.ptr(self.flag_buf), st))
        if self.p2p is not None:
            self.p2p["grad"].barrier(channel=0)   # every rank's gradient and flag are complete
        g, p, f = self._peer_arrays
        N.check(lib.lnrf_adam_step_sharded_f32(C.cast(g, C.c_void_p), C.cast(p, C.c_void_p), C.cast(f, C.c_void_p), self.world, self.rank,
                                               self.lo, self.Sz, self._seg_start, self._seg_mult, len(self._seg_mult),
                                               N.ptr(self.state[0]["exp_avg"]), N.ptr(self.state[0]["exp_avg_sq"]), self.lr, self.betas[0],
                                               self.betas[1], self.eps, self.weight_decay, N.ptr(self._scale), N.ptr(self.found_inf),
                                               N.ptr(self.step_count), N.ptr(self.lr_scale), st))
        if self.p2p is not None:
            self.p2p["grad"].barrier(channel=1)   # every rank has stored into this rank's parameters and read its gradient
        # gradient clear (the fp32 vector as 2 x P_pad fp16 words) + GradScaler.update() in one launch
        N.check(lib.lnrf_exchange_tail(N.ptr(self.grad_flat), 2 * self.P_pad, N.ptr(self._scale), N.ptr(self._growth_tracker),
                                       N.ptr(self.found_inf), N.ptr(self.step_count), self.growth_factor, self.backoff_factor,
                                       self.growth_interval, st))

    def _one_f32(self, t):
        arr = (N.OptTensor * 1)()
        arr[0].grad, arr[0].n, arr[0].grad_dtype = t.data_ptr(), t.numel(), N.F32
        return arr

    # ---- checkpoints: torch.optim.Adam's per-parameter layout (a collective at world_size > 1) ------------------------
    def _full(self, shard):
        if self.world == 1:
            return shard
        import torch.distributed as dist
        full = torch.empty(self.P_pad, dtype=shard.dtype, device=shard.device)
        dist.all_gather_into_tensor(full, shard.contiguous(), group=self.group)
        return full

    def state_dict(self):
        step = float(self.step_count.item()) - 1.0
        ea, es = self._full(self.state[0]["exp_avg"]), self._full(self.state[0]["exp_avg_sq"])
        state = {}
        for i, (o, off) in enumerate(zip(self.owners, self._offsets)):
            n = o.param.numel()
            state[i] = {"step": torch.tensor(step), "exp_avg": ea[off:off + n].view_as(o.param).clone(),
                        "exp_avg_sq": es[off:off + n].view_as(o.param).clone()}
        groups = []
        for gi in range(self.n_groups):
            idx = [i for i, o in enumerate(self.owners) if o.group == gi]
            mult = self.owners[idx[0]].lr_mult if idx else 1.0
            groups.append({"lr": self.lr * mult, "betas": self.betas, "eps": self.eps, "weight_decay": self.weight_decay, "amsgrad": False,
                           "maximize": False, "foreach": None, "capturable": False, "differentiable": False, "fused": None,
                           "decoupled_weight_decay": False, "params": idx})
        return {"state": state, "param_groups": groups}

    @torch.no_grad()
    def load_state_dict(self, sd):
        n = len(self.owners)
        if len(sd["state"]) not in (0, n):
            raise RuntimeError(f"ShardedFlatAdam.load_state_dict: {len(sd['state'])} state entries for {n} parameter tensors")
        if len(sd["state"]) == n:
            for k in ("exp_avg", "exp_avg_sq"):
                flat = torch.zeros(self.P_pad, dtype=torch.float32, device=self.param_flat.device)
                for i, (o, off) in enumerate(zip(self.owners, self._offsets)):
                    flat[off:off + o.param.numel()] = sd["state"][i][k].reshape(-1)
                self.state[0][k].copy_(flat[self.lo:self.hi])
            self.step_count.fill_(float(sd["state"][0]["step"]) + 1.0)
        g = next((g for g in sd["param_groups"] if g["params"]), sd["param_groups"][0])
        first = self.owners[g["params"][0]].lr_mult if g["params"] else 1.0
        self.lr = float(g["lr"]) / first
        self.betas, self.eps, self.weight_decay = tuple(map(float, g["betas"])), float(g["eps"]), float(g["weight_decay"])
