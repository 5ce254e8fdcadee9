"""``FunctionalEnsemble`` — M sparse autoencoders trained in lock-step on one GPU.

Drop-in for the reference's ``autoencoders/ensemble.py`` (FunctionalEnsemble :68-193, stack_dict/unstack_dict
:50-65, optim_str_to_func :25-31): same constructor, same attributes (``params``, ``buffers``, ``optim_states``,
``n_models``, ``sig``, ``device``, ``no_stacking``), same methods (``step_batch``, ``unstack``, ``state_dict`` /
``from_state``, ``to_device``, ``to_shared_memory``). Parameters, buffers and Adam moments stay torch tensors owned
by Python and are updated in place, so ``unstack``/export/IPC keep working.

What differs is *how* a step is computed. The reference builds ``vmap(grad(sig.loss))`` + ``vmap(torchopt.adam)``
out of ~70 stock PyTorch launches that stream the fp32 code tensor [M, B, n] through HBM a dozen times. Here
``step_batch`` is one call into libsce.so (include/sce.h): four tcgen05 split-operand GEMMs with fused epilogues plus a
handful of streaming kernels; the code tensor exists only as operand planes (4 bytes per element) consumed by the next GEMM.
``aux["c"]`` is therefore a lazy :class:`CodeProxy` — ``aux["c"].count_nonzero(dim=-1).float().mean(dim=-1)``
(the only use in the reference loop, big_sweep.py:171) is answered from fused counters, and ``.dense()``
materialises the real [M, B, n] tensor on demand.

There is no CPU path and no generic-autograd path: a signature without an engine ``variant`` raises.

Range contract of the default arithmetic (``arith="auto"`` -> f16f8 where the shape allows, include/sce.h): operand
values must fit fp16. The engine guards this on the device — a batch holding |x| >= 65520 / NaN, or a step whose loss
is not finite, SKIPS its Adam update (parameters, moments and operand planes stay untouched) and raises a sticky
health flag. ``step_batch`` reads that flag after the first step of a plan and every ``health_check_every`` steps
(one small D2H copy), ``check_health()`` on demand (the chunk loops call it at the end of every chunk): with
``arith="auto"`` the ensemble then rebuilds its plan on the fp32-range bf16x3 arithmetic, re-runs the current batch
and warns; with an explicitly requested arithmetic it raises ``FloatingPointError``.
"""
from __future__ import annotations

import ctypes as C
import warnings
from typing import Dict, List, Optional

import torch

from . import _lib
from .optim import AdamConfig, adam, resolve_optimizer
from .signatures import DictSignature
from .tracing import nvtx_range

Tensor = torch.Tensor

_VARIANT_CODE = {"tied": _lib.SCE_TIED, "masked_tied": _lib.SCE_TIED, "untied": _lib.SCE_UNTIED,
                 "masked_untied": _lib.SCE_UNTIED, "topk": _lib.SCE_TOPK}
_LOSS_KEYS = {
    "tied": ("loss", "l_reconstruction", "l_l1"),
    "masked_tied": ("loss", "l_reconstruction", "l_l1"),
    "masked_untied": ("loss", "l_reconstruction", "l_l1"),
    "untied": ("loss", "l_reconstruction", "l_l1", "l_bias_decay"),
    "topk": ("loss",),
}


def optim_str_to_func(optim_str):
    """ensemble.py:25-31."""
    if optim_str == "adam":
        return adam
    raise ValueError("Unknown optimizer string: {}".format(optim_str))


def construct_stacked_leaf(tensors, device=None) -> Tensor:
    """ensemble.py:35-46."""
    all_rg = all(t.requires_grad for t in tensors)
    none_rg = all(not t.requires_grad for t in tensors)
    if not all_rg and not none_rg:
        raise RuntimeError("Expected tensors from each model to have the same .requires_grad")
    result = torch.stack(list(tensors)).to(device=device)
    if all_rg:
        result = result.detach().requires_grad_()
    return result


def stack_dict(models: List[dict], device=None) -> dict:
    """Stack the same-keyed (possibly nested) dicts of M models along a new dim 0 (ensemble.py:50-56)."""
    first = models[0]
    out = {}
    for k, v in first.items():
        if isinstance(v, dict):
            out[k] = stack_dict([m[k] for m in models], device=device)
        else:
            out[k] = construct_stacked_leaf([m[k] for m in models], device=device)
    return out


def unstack_dict(params: dict, n_models: int, device=None) -> List[dict]:
    """ensemble.py:59-65."""
    outs = [dict() for _ in range(n_models)]
    for k, v in params.items():
        if isinstance(v, dict):
            subs = unstack_dict(v, n_models, device=device)
            for i in range(n_models):
                outs[i][k] = subs[i]
        else:
            for i in range(n_models):
                outs[i][k] = v[i].to(device=device)
    return outs


def _tree_map(fn, tree):
    return {k: (_tree_map(fn, v) if isinstance(v, dict) else fn(v)) for k, v in tree.items()}


class _RowCount:
    """Result of ``CodeProxy.count_nonzero(dim=-1)``: supports the reference's ``.float().mean(dim=-1)``."""

    def __init__(self, proxy):
        self._p = proxy

    def float(self):
        return self

    def mean(self, dim=-1):
        if dim not in (-1, 1):
            return self._p.dense().count_nonzero(dim=-1).float().mean(dim=dim)
        return self._p.mean_nnz

    def __getattr__(self, name):  # anything else: fall back to the real per-row counts
        return getattr(self._p.dense().count_nonzero(dim=-1), name)


class CodeProxy:
    """Lazy stand-in for ``aux["c"]`` ([M, B, n] fp32). Valid until the next engine call on the ensemble."""

    def __init__(self, ens, B, mean_nnz, serial):
        self._ens, self._B, self.mean_nnz, self._serial = ens, B, mean_nnz, serial
        self._dense = None

    @property
    def shape(self):
        return torch.Size((self._ens.n_models, self._B, self._ens._n))

    def count_nonzero(self, dim=-1):
        if dim in (-1, 2):
            return _RowCount(self)
        return self.dense().count_nonzero(dim=dim)

    def dense(self) -> Tensor:
        if self._dense is None:
            if self._serial != self._ens._serial:
                raise RuntimeError("aux['c'] was read after a later engine call overwrote the code buffers; call "
                                   ".dense() before the next step_batch, or construct the ensemble with "
                                   "materialize_code=True")
            self._dense = self._ens._read_code(self._B)
        return self._dense

    def __getattr__(self, name):
        return getattr(self.dense(), name)

    def __getitem__(self, idx):
        return self.dense()[idx]


class FunctionalEnsemble:
    def __init__(self, models, sig, optimizer_func, optimizer_kwargs, device=None, no_stacking=False,
                 adam_count_mode: str = "frozen_t1", fwd_passes: int = 3, bwd_passes: int = 3,
                 materialize_code: bool = False, arith: str = "auto", health_check_every: int = 64):
        """``models``: list of (params, buffers) from ``sig.init``; ``optimizer_func``: ``torchopt.adam`` (if
        installed), :func:`sparse_coding_b200.optim.adam`, or the string "adam"; ``optimizer_kwargs``: ``{"lr": …}``.
        ``no_stacking`` is accepted for API compatibility (the reference needs it for TopK because ``torch.topk``
        with a data-dependent k cannot be vmapped; the engine batches TopK models natively).
        Extra keywords (engine-only): ``adam_count_mode`` "frozen_t1" (reference behaviour, SURVEY.md Q2) or
        "standard"; ``fwd_passes`` / ``bwd_passes`` 3 (split operands, fp32-grade) or 1 (16-bit plane only);
        ``arith`` "auto" | "bf16x3" | "f16f8": how fp32 operands reach the tensor cores (include/sce.h, sce_arith);
        ``health_check_every``: steps between reads of the device-side health flag (module docstring; 0 = never)."""
        if device is None:
            first = next(iter(models[0][0].values()))
            self.device = first.device
        else:
            self.device = device
        self.n_models = len(models)
        params, buffers = tuple(zip(*models))
        self.params = stack_dict(list(params), device=self.device)
        self.buffers = stack_dict(list(buffers), device=self.device)
        self.sig = sig
        self.no_stacking = no_stacking
        self.optimizer_func = optimizer_func
        self.optimizer_kwargs = optimizer_kwargs
        self.optimizer = resolve_optimizer(optimizer_func, optimizer_kwargs)
        self.adam_count_mode = adam_count_mode
        self.fwd_passes, self.bwd_passes = fwd_passes, bwd_passes
        if arith not in _lib.ARITH_CODE:
            raise ValueError(f"arith must be one of {sorted(_lib.ARITH_CODE)}, got {arith!r}")
        self.arith = arith
        self.materialize_code = materialize_code
        self.health_check_every = int(health_check_every)
        self.optim_states = {
            "mu": _tree_map(torch.zeros_like, self.params),
            "nu": _tree_map(torch.zeros_like, self.params),
            "count": _tree_map(lambda t: torch.zeros(t.shape[0], dtype=torch.int64, device=t.device), self.params),
        }
        self.init_functions()

    # ------------------------------------------------------------------------------------------------------
    def init_functions(self):
        variant = getattr(self.sig, "variant", None)
        if variant not in _VARIANT_CODE:
            raise NotImplementedError(
                f"{getattr(self.sig, '__name__', self.sig)} has no engine variant: only the signatures of the sweep hot "
                "path (FunctionalTiedSAE, FunctionalSAE, the Masked variants, TopKEncoder) are implemented in the "
                "sm_100a engine, and there is deliberately no generic autograd fallback")
        self._variant = variant
        self._plan = None
        self._plan_key = None
        self._plan_k_max = 0              # TopK: the largest sparsity the current plan was built for
        self._ws = None
        self._centering = None
        self._serial = 0
        self._steps = 0
        main = "dict" if variant == "topk" else "encoder"
        self._main = main
        self._n, self._d = self.params[main].shape[1], self.params[main].shape[2]
        self._engine_buffers = None
        self._arith_fallback = None       # "bf16x3" once an auto plan left the fp16 range (sticky for this object)
        self._since_health = 0            # steps since the health flag was last read
        self._plan_steps = 0              # steps taken on the current plan

    # ------------------------------------------------------------------------------------------------------
    # engine plumbing
    # ------------------------------------------------------------------------------------------------------
    def _require_cuda(self):
        dev = torch.device(self.device)
        if dev.type != "cuda":
            raise RuntimeError(f"FunctionalEnsemble computes in the sm_100a CUDA engine; device is {dev}. "
                               "Move it with to_device('cuda:…') — there is no CPU implementation.")
        return dev

    def _needs_centering(self) -> bool:
        """Whether the tied signature's centring is non-trivial. Evaluated once (it costs three device
        reductions and a host sync) and cached until ``refresh()`` / ``to_device()``."""
        if self._variant != "tied":
            return False
        if self._centering is None:
            self._centering = self._centering_is_nontrivial()
        return self._centering

    def _centering_is_nontrivial(self) -> bool:
        b = self.buffers
        d = self._d
        eye = torch.eye(d, device=b["center_rot"].device, dtype=b["center_rot"].dtype)
        return not (bool((b["center_rot"] == eye).all()) and bool((b["center_trans"] == 0).all())
                    and bool((b["center_scale"] == 1).all()))

    def _topk_k_max(self) -> int:
        """Largest ``buffers["sparsity"]`` of a TopK ensemble (0 for the other variants); raises ``ValueError`` naming
        the model when a k is outside [1, n] (``torch.topk`` raises for k > n in the reference)."""
        if self._variant != "topk":
            return 0
        ks = [int(k) for k in self.buffers["sparsity"].reshape(-1).tolist()]
        for m, k in enumerate(ks):
            if not 1 <= k <= self._n:
                raise ValueError(f"model {m}: sparsity k = {k} is outside [1, n = {self._n}]")
        return max(ks)

    def _build_plan(self, batch_max: int, x_per_model: bool, centering: int = 0):
        dev = self._require_cuda()
        k_max = self._topk_k_max()
        lib = _lib.load()
        for k, v in self.params.items():
            if v.dtype != torch.float32:
                raise TypeError(f"the engine trains fp32 parameters; params['{k}'] is {v.dtype}")
            if not v.is_contiguous():
                self.params[k] = v.contiguous()
        self._destroy_plan()
        cfg: AdamConfig = self.optimizer
        desc = _lib.SceDesc(
            variant=_VARIANT_CODE[self._variant], n_models=self.n_models, d=self._d, n=self._n,
            batch_max=batch_max, x_per_model=int(x_per_model), lr=cfg.lr, beta1=cfg.b1, beta2=cfg.b2, eps=cfg.eps,
            eps_root=cfg.eps_root,
            adam_count_mode=_lib.SCE_ADAM_FROZEN_T1 if self.adam_count_mode == "frozen_t1" else _lib.SCE_ADAM_STANDARD,
            fwd_passes=self.fwd_passes, bwd_passes=self.bwd_passes,
            norm_floor=0.0 if self._variant == "topk" else 1e-8,
            arith=_lib.ARITH_CODE[getattr(self, "_arith_fallback", None) or getattr(self, "arith", "auto")],
            topk_k_max=k_max,
            centering=centering)
        nbytes = lib.sce_workspace_bytes(C.byref(desc))
        if nbytes == 0:
            _lib.check(-1, "sce_workspace_bytes")
        with torch.cuda.device(dev):
            self._ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
        ws_ptr = (self._ws.data_ptr() + 1023) // 1024 * 1024
        M = self.n_models
        eb = {}

        def f32vec(name):  # [M] fp32 hyper-parameter buffers
            t = self.buffers.get(name)
            if t is None:
                return None
            eb[name] = t.to(device=dev, dtype=torch.float32).contiguous()
            return eb[name].data_ptr()

        ptr = lambda t: t.data_ptr() if t is not None else None
        mu, nu = self.optim_states["mu"], self.optim_states["nu"]
        bufs = _lib.SceBuffers()
        bufs.encoder = ptr(self.params[self._main])
        bufs.encoder_m, bufs.encoder_v = ptr(mu[self._main]), ptr(nu[self._main])
        if self._variant != "topk":
            bufs.encoder_bias = ptr(self.params["encoder_bias"])
            bufs.bias_m, bufs.bias_v = ptr(mu["encoder_bias"]), ptr(nu["encoder_bias"])
            bufs.l1_alpha = f32vec("l1_alpha")
            if self._variant in ("tied", "untied"):
                bufs.bias_decay = f32vec("bias_decay")
        if self._variant in ("untied", "masked_untied"):
            bufs.decoder = ptr(self.params["decoder"])
            bufs.decoder_m, bufs.decoder_v = ptr(mu["decoder"]), ptr(nu["decoder"])
        if self._variant in ("masked_tied", "masked_untied"):
            eb["coef_mask"] = self.buffers["coef_mask"].to(device=dev, dtype=torch.uint8).contiguous()
            bufs.coef_mask = eb["coef_mask"].data_ptr()
        if self._variant == "topk":
            eb["sparsity"] = self.buffers["sparsity"].to(device=dev, dtype=torch.int64).contiguous()
            bufs.sparsity = eb["sparsity"].data_ptr()
        if centering:
            # FunctionalTiedSAE.center (sae_ensemble.py:126-128) runs on the device: (x - trans) planes, GEMM with rot, * scale
            for name in ("center_trans", "center_rot", "center_scale"):
                eb[name] = self.buffers[name].to(device=dev, dtype=torch.float32).contiguous()
            bufs.center_trans, bufs.center_rot, bufs.center_scale = (eb["center_trans"].data_ptr(), eb["center_rot"].data_ptr(),
                                                                     eb["center_scale"].data_ptr())
        bufs.workspace, bufs.workspace_bytes = ws_ptr, nbytes
        plan = C.c_void_p()
        with torch.cuda.device(dev):
            _lib.check(lib.sce_plan_create(C.byref(desc), C.byref(bufs), C.byref(plan)), "sce_plan_create")
            self._plan = plan
            self._engine_buffers = eb
            self._plan_key = (batch_max, bool(x_per_model), int(centering))
            self._plan_k_max = k_max
            _lib.check(lib.sce_set_step_count(plan, self._steps), "sce_set_step_count")
            _lib.check(lib.sce_prepare(plan, self._stream()), "sce_prepare")
        self._plan_steps = 0
        self._since_health = 0
        self._new_outputs()

    def _new_outputs(self):
        """Fresh result tensors for the next engine call (the reference returns new tensors every step; allocating
        them from torch's caching allocator costs no kernel, unlike cloning a fixed output buffer)."""
        dev = torch.device(self.device)
        self._out_losses = torch.empty(self.n_models, _lib.SCE_LOSS_COLS, dtype=torch.float32, device=dev)
        self._out_nnz = torch.empty(self.n_models, dtype=torch.float32, device=dev)

    def _destroy_plan(self):
        if getattr(self, "_plan", None) is not None:
            _lib.load().sce_plan_destroy(self._plan)
            self._plan = None

    def __del__(self):
        try:
            self._destroy_plan()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(torch.device(self.device)).cuda_stream)

    def _prep_batch(self, minibatches: Tensor, expand_dims: bool):
        dev = self._require_cuda()
        x = minibatches
        if x.device != dev:
            x = x.to(dev, non_blocking=True)
        if x.dtype != torch.float32:
            x = x.float()
        per_model = not expand_dims
        # non-identity centring (sae_ensemble.py:126-128) is applied by the engine (sce_desc.centering): 1 = this batch is
        # one [B,d] array for all models, 2 = [M,B,d]; the centred batch is per model either way
        centering = (1 if expand_dims else 2) if self._needs_centering() else 0
        x = x.contiguous()
        B = x.shape[-2]
        if x.shape[-1] != self._d or (per_model and (x.dim() != 3 or x.shape[0] != self.n_models)):
            raise ValueError(f"batch shape {tuple(x.shape)} does not match ensemble (M={self.n_models}, d={self._d})")
        plan_per_model = per_model or centering != 0
        key = self._plan_key
        if self._plan is None or key is None or key[1] != plan_per_model or key[2] != centering or B > key[0]:
            self._build_plan(max(B, key[0]) if key else B, plan_per_model, centering)
        return x, B

    def _losses_dict(self) -> Dict[str, Tensor]:
        cols = self._out_losses
        return {k: cols[:, i] for i, k in enumerate(("loss", "l_reconstruction", "l_l1", "l_bias_decay"))
                if k in _LOSS_KEYS[self._variant]}

    def _aux(self, B):
        self._serial += 1
        proxy = CodeProxy(self, B, self._out_nnz, self._serial)
        if self.materialize_code:
            return {"c": proxy.dense()}
        return {"c": proxy}

    def _results(self, B):
        """(loss_data, aux) of the engine call that just wrote the current output tensors; hands those tensors to
        the caller and allocates fresh ones for the next call."""
        out = (self._losses_dict(), self._aux(B))
        self._new_outputs()
        return out

    def _read_code(self, B) -> Tensor:
        out = torch.empty(self.n_models, B, self._n, dtype=torch.float32, device=self.device)
        with torch.cuda.device(out.device):
            _lib.check(_lib.load().sce_read_code(self._plan, B, out.data_ptr(), self._stream()), "sce_read_code")
        return out

    # ------------------------------------------------------------------------------------------------------
    # public API (reference names)
    # ------------------------------------------------------------------------------------------------------
    def step_batch(self, minibatches, expand_dims=True):
        """One Adam step of every model on one batch (ensemble.py:175-193). Returns (loss_data, aux)."""
        with torch.no_grad(), nvtx_range("sce.step_batch"):
            every = getattr(self, "health_check_every", 64)
            while True:
                x, B = self._prep_batch(minibatches, expand_dims)
                self._launch_step(x, B)
                self._plan_steps += 1
                self._since_health += 1
                if not every or not (self._plan_steps == 1 or self._since_health >= every):
                    break
                if self._health_action(rerun=True) != "rerun":
                    break
                # the plan was rebuilt on bf16x3 (the update of this batch was skipped on the device): take the step again
            self._steps += 1
            if self.adam_count_mode != "frozen_t1":
                for t in self.optim_states["count"].values():
                    t.add_(1)
            return self._results(B)

    def _launch_step(self, x, B):
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().sce_step(self._plan, x.data_ptr(), B, self._out_losses.data_ptr(),
                                            self._out_nnz.data_ptr(), self._stream()), "sce_step")

    # ------------------------------------------------------------------------------------------------------
    # health (range contract of the f16f8 arithmetic, non-finite losses)
    # ------------------------------------------------------------------------------------------------------
    def health(self):
        """(bad, absmax) from the device: ``bad`` — some step since the plan was prepared skipped its update because
        the batch left the fp16 range or the loss was not finite; ``absmax`` — largest |x| fed (f16f8 plans)."""
        if self._plan is None:
            return False, 0.0
        bad, amax = C.c_int(0), C.c_float(0.0)
        with torch.cuda.device(torch.device(self.device)):
            _lib.check(_lib.load().sce_health(self._plan, C.byref(bad), C.byref(amax), self._stream()), "sce_health")
        self._since_health = 0
        return bool(bad.value), float(amax.value)

    def _health_action(self, rerun=None):
        bad, amax = self.health()
        if not bad:
            return "ok"
        resolved = self.resolved_arith()
        lost = max(self._plan_steps - 1, 0) if rerun else self._plan_steps
        lost = min(lost, getattr(self, "health_check_every", 64))
        if resolved == "f16f8" and getattr(self, "arith", "auto") == "auto":
            self._arith_fallback = "bf16x3"
            key = self._plan_key
            self._build_plan(key[0], key[1], key[2])
            warnings.warn(
                f"a batch left the range of the f16f8 operand arithmetic (largest |activation| {amax:g}; fp16 holds "
                "|v| < 65504) or produced a non-finite loss: the affected updates were skipped on the device, the "
                f"ensemble now runs on arith='bf16x3' (fp32 range). Up to {lost} earlier step(s) since the last health "
                "check made no update.", RuntimeWarning)
            return "rerun"
        raise FloatingPointError(
            f"the engine skipped parameter updates: largest |activation| fed = {amax:g}, arithmetic = {resolved} "
            + ("(values beyond 65504 do not fit its fp16 operand plane: construct the ensemble with arith='bf16x3' "
               "or arith='auto')" if resolved == "f16f8" else "(a loss was not finite)")
            + "; parameters and Adam moments were left untouched by the offending steps")

    def check_health(self) -> None:
        """Read the device-side health flag now (the chunk loops call this at the end of every chunk)."""
        if self._plan is not None:
            self._health_action(rerun=None)

    def forward_batch(self, minibatches, expand_dims=True, return_x_hat=False):
        """Forward only: losses and code statistics (and optionally x̂ [M,B,d]) without touching parameters."""
        with torch.no_grad():
            x, B = self._prep_batch(minibatches, expand_dims)
            x_hat = torch.empty(self.n_models, B, self._d, dtype=torch.float32, device=x.device) if return_x_hat else None
            with torch.cuda.device(x.device):
                _lib.check(_lib.load().sce_forward(self._plan, x.data_ptr(), B,
                                                   x_hat.data_ptr() if return_x_hat else None,
                                                   self._out_losses.data_ptr(), self._out_nnz.data_ptr(),
                                                   self._stream()), "sce_forward")
            out = self._results(B)
            return out + (x_hat,) if return_x_hat else out

    def grads_batch(self, minibatches, expand_dims=True):
        """Parameter gradients exactly as ``vmap(grad(sig.loss))`` would return them (parity tests)."""
        with torch.no_grad():
            x, B = self._prep_batch(minibatches, expand_dims)
            g = {k: torch.empty_like(v) for k, v in self.params.items()}
            ptr = lambda k: g[k].data_ptr() if k in g else None
            with torch.cuda.device(x.device):
                _lib.check(_lib.load().sce_grads(self._plan, x.data_ptr(), B, ptr(self._main), ptr("encoder_bias"),
                                                 ptr("decoder"), self._out_losses.data_ptr(),
                                                 self._out_nnz.data_ptr(), self._stream()), "sce_grads")
            return g, self._results(B)

    def calc_grads(self, params, buffers, minibatches):
        """Reference-shaped entry point (``self.calc_grads`` of ensemble.py:99-123): gradients of ``sig.loss`` for
        the stacked models on ``minibatches`` [M, B, d]. ``params`` / ``buffers`` must be this ensemble's own trees
        (the engine reads the tensors it was planned on). Returns ``(grads, (loss_data, aux))``."""
        if params is not self.params or buffers is not self.buffers:
            raise ValueError("calc_grads operates on the ensemble's own params/buffers (in-place engine)")
        if minibatches.dim() == 3 and minibatches.stride(0) == 0:      # an expand()-ed shared batch: don't copy it M times
            return self.grads_batch(minibatches[0], expand_dims=True)
        return self.grads_batch(minibatches, expand_dims=False)

    def refresh(self):
        """Call after modifying ``params`` / ``buffers`` from outside the engine (re-derives the operand
        copies and the cached centring check). A TopK ensemble whose largest ``sparsity`` changed gets a new plan:
        the list capacity, the gather-path choice and the slice count all follow from it."""
        self._centering = None
        k_max = self._topk_k_max()
        if self._plan is not None and k_max != self._plan_k_max:
            key = self._plan_key
            self._build_plan(key[0], key[1], key[2])
        elif self._plan is not None:
            # engine-side copies of the buffers (dtype-converted hyper-parameter vectors, uint8 coef_mask, int64
            # sparsity) keep their addresses — the plan holds the pointers — and are refilled in place
            for name, t in (self._engine_buffers or {}).items():
                t.copy_(self.buffers[name].to(device=t.device, dtype=t.dtype))
            with torch.cuda.device(torch.device(self.device)):
                _lib.check(_lib.load().sce_prepare(self._plan, self._stream()), "sce_prepare")
            self._plan_steps = 0

    def profile_begin(self):
        """Start per-phase device timing of the following ``step_batch`` calls (up to 64 steps)."""
        if self._plan is None:
            raise RuntimeError("profile_begin needs a built plan: run one step_batch first")
        _lib.check(_lib.load().sce_profile_begin(self._plan), "sce_profile_begin")

    def profile_end(self) -> Dict[str, float]:
        """Stop timing; returns {"steps": k, phase: total milliseconds over those k steps, ...}."""
        ms = (C.c_float * len(_lib.PHASES))()
        steps = C.c_int(0)
        _lib.check(_lib.load().sce_profile_end(self._plan, ms, C.byref(steps)), "sce_profile_end")
        out = {name: float(ms[i]) for i, name in enumerate(_lib.PHASES)}
        out["steps"] = int(steps.value)
        return out

    def gpu_launches_last_call(self) -> int:
        return int(_lib.load().sce_last_launch_count(self._plan)) if self._plan is not None else 0

    def resolved_arith(self):
        """"bf16x3" or "f16f8": what the current plan runs (``arith="auto"`` resolves per shape); None before the
        first step."""
        if self._plan is None:
            return None
        return _lib.ARITH_NAME.get(int(_lib.load().sce_plan_arith(self._plan)))

    def input_absmax(self) -> float:
        """f16f8 plans: the largest |x| the engine has been fed since the plan was (re)prepared (one 4-byte D2H copy +
        stream sync; 0.0 for bf16x3 / before the first step). Values beyond 65504 overflow the fp16 operand plane
        (losses turn inf/NaN), magnitudes far below 1e-3 lose relative precision: switch such data to
        ``arith="bf16x3"``. ``ensemble_train_loop`` checks this once per chunk."""
        if self._plan is None:
            return 0.0
        out = C.c_float(0.0)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().sce_input_absmax(self._plan, C.byref(out), self._stream()), "sce_input_absmax")
        return float(out.value)

    def active_counts(self, B: int, counts: Optional[Tensor] = None) -> Tensor:
        """Add, per model and feature, the number of the ``B`` rows of the most recent engine call whose code is
        non-zero to ``counts`` ([M, n] int32 on the device; created zeroed when None) and return it — the reference's
        ``(c != 0).sum(0)`` (standard_metrics.py:441-454; ``/ rows`` gives :305-308). Fused: column sums of the
        activity-mask plane the encode epilogue wrote; the dense code is never materialised."""
        if self._plan is None:
            raise RuntimeError("active_counts needs a built plan: run forward_batch / step_batch first")
        dev = torch.device(self.device)
        if counts is None:
            counts = torch.zeros(self.n_models, self._n, dtype=torch.int32, device=dev)
        if counts.dtype != torch.int32 or tuple(counts.shape) != (self.n_models, self._n) or not counts.is_contiguous():
            raise ValueError("counts must be a contiguous int32 tensor of shape [n_models, n]")
        with torch.cuda.device(dev):
            _lib.check(_lib.load().sce_active_counts(self._plan, int(B), counts.data_ptr(), self._stream()),
                       "sce_active_counts")
        return counts

    def unstack(self, device=None):
        params = unstack_dict(self.params, self.n_models, device=device)
        buffers = unstack_dict(self.buffers, self.n_models, device=device)
        return list(zip(params, buffers))

    def state_dict(self):
        """ensemble.py:150-161 keys, plus the engine-only settings."""
        return {
            "device": self.device, "n_models": self.n_models, "params": self.params, "buffers": self.buffers,
            "sig": self.sig, "no_stacking": self.no_stacking, "optimizer_func": self.optimizer_func,
            "optimizer_kwargs": self.optimizer_kwargs, "optim_states": self.optim_states,
            "adam_count_mode": self.adam_count_mode, "fwd_passes": self.fwd_passes, "bwd_passes": self.bwd_passes,
            "arith": getattr(self, "arith", "auto"), "arith_fallback": getattr(self, "_arith_fallback", None),
            "health_check_every": getattr(self, "health_check_every", 64),
            "materialize_code": self.materialize_code, "steps": self._steps,
        }

    @staticmethod
    def from_state(state_dict):
        self = FunctionalEnsemble.__new__(FunctionalEnsemble)
        for k in ("device", "n_models", "params", "buffers", "sig", "no_stacking", "optimizer_func",
                  "optimizer_kwargs", "optim_states"):
            setattr(self, k, state_dict[k])
        self.adam_count_mode = state_dict.get("adam_count_mode", "frozen_t1")
        self.arith = state_dict.get("arith", "auto")
        self.fwd_passes = state_dict.get("fwd_passes", 3)
        self.bwd_passes = state_dict.get("bwd_passes", 3)
        self.materialize_code = state_dict.get("materialize_code", False)
        self.health_check_every = state_dict.get("health_check_every", 64)
        self.optimizer = resolve_optimizer(self.optimizer_func, self.optimizer_kwargs)
        self.init_functions()
        self._arith_fallback = state_dict.get("arith_fallback")
        self._steps = state_dict.get("steps", 0)
        if self.adam_count_mode != "frozen_t1":
            # The reference's dispatch hands state_dict() to a freshly spawned worker per chunk (cluster_runs.py:113-125):
            # the worker's Python step counter dies with it, but optim_states["count"] is shared memory updated in
            # place, so the bias correction continues from there.
            counts = [int(t.max()) for t in self.optim_states.get("count", {}).values() if t.numel()]
            if counts:
                self._steps = max(self._steps, max(counts))
        return self

    def to_device(self, device):
        self._destroy_plan()
        self._plan_key = None
        self._centering = None
        self.device = device
        self.params = _tree_map(lambda t: t.to(device), self.params)
        self.buffers = _tree_map(lambda t: t.to(device), self.buffers)
        self.optim_states = _tree_map(lambda t: t.to(device), self.optim_states)

    def to_shared_memory(self):
        for tree in (self.params, self.buffers, self.optim_states):
            _tree_map(lambda t: t.share_memory_(), tree)
