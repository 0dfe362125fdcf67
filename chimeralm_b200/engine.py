"""Python handle on one native context (one per GPU).

PyTorch is used here only for device memory, streams and tensors handed to the C-ABI as raw
pointers; every computation happens in the CUDA library.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _lib
from .config import DEFAULT_CONFIG, HyenaConfig
from .weights import BACKBONE_PREFIX, HEAD_PREFIX

_IDS_DTYPES = {torch.uint8: _lib.CLM_U8, torch.int32: _lib.CLM_I32, torch.int64: _lib.CLM_I64}


def _full_name(name: str) -> str:
    """State-dict key of a head tensor given as "net.head.x", "head.x" or "x"."""
    if name.startswith("net."):
        return name
    return "net." + name if name.startswith("head.") else HEAD_PREFIX + name


def tail_keys(n_layer: int) -> list[str]:
    """State-dict keys of the last block's tail and ln_f, the tensors `Engine.tail_train_begin` adds to training."""
    p = f"{BACKBONE_PREFIX}layers.{n_layer - 1}."
    return [p + "mixer.out_proj.weight", p + "mixer.out_proj.bias", p + "norm2.weight", p + "norm2.bias",
            p + "mlp.fc1.weight", p + "mlp.fc1.bias", p + "mlp.fc2.weight", p + "mlp.fc2.bias",
            BACKBONE_PREFIX + "ln_f.weight", BACKBONE_PREFIX + "ln_f.bias"]


def _stream_ptr(device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Engine:
    """Owns a `clm_ctx`: weights, filter tables, workspaces (include/chimeralm_b200.h)."""

    def __init__(self, state_dict, device: int | str | torch.device = 0, cfg: HyenaConfig = DEFAULT_CONFIG,
                 max_batch: int = 32, max_tokens: int = 8193, token_budget: int | None = None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise _lib.ChimeraLMNativeError("no CUDA device: chimeralm_b200 has no CPU path")
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        self.cfg = cfg
        torch.cuda.set_device(self.device)
        torch.zeros(1, device=self.device)  # make sure the primary context exists
        ccfg = _lib.clm_config()
        self.lib.clm_default_config(C.byref(ccfg))
        ccfg.d_model, ccfg.n_layer, ccfg.d_inner = cfg.d_model, cfg.n_layer, cfg.d_inner
        ccfg.vocab_rows, ccfg.max_seq_len = cfg.vocab_rows, cfg.max_seq_len
        ccfg.filter_order, ccfg.emb_dim = cfg.filter_order, cfg.emb_dim
        ccfg.short_filter_order, ccfg.num_inner_mlps = cfg.short_filter_order, cfg.num_inner_mlps
        ccfg.head_hidden, ccfg.num_classes = cfg.head_hidden, cfg.num_classes
        ccfg.layer_norm_eps, ccfg.filter_shift = cfg.layer_norm_epsilon, cfg.shift
        if cfg.pooling_type not in _lib.POOLING:
            raise ValueError(f"Unsupported pooling type: {cfg.pooling_type}")   # the reference's message (components/hyena.py:135)
        ccfg.pooling = _lib.POOLING[cfg.pooling_type]
        self.ctx = C.c_void_p()
        rc = self.lib.clm_create(C.byref(ccfg), self.device.index or 0, C.byref(self.ctx))
        if rc < 0:
            msg = self.lib.clm_last_error(self.ctx).decode() if self.ctx else "clm_create rejected the configuration"
            raise _lib.ChimeraLMNativeError(f"clm_create failed (status {rc}): {msg}")
        self.load_state_dict(state_dict)
        self._check(self.lib.clm_finalize(self.ctx), "clm_finalize")
        self.max_batch = self.max_tokens = self.token_budget = 0
        self.last_seq = 0
        self.tc_fallbacks = 0   # batches redone with the fp32 convolution by forward(check=True)
        self._debug_stop = False
        self.reserve(max_batch, max_tokens, token_budget)
        # CLM_OPTIONS="name=value,name=value": kernel-selection switches (clm_set_option) for A/B runs of the test suite / bench
        for item in filter(None, os.environ.get("CLM_OPTIONS", "").split(",")):
            name, _, val = item.partition("=")
            self.set_option(name.strip(), int(val))

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc, what):
        _lib.check(self.ctx, rc, what)

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.clm_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_state_dict(self, sd) -> None:
        self._head_shapes = getattr(self, "_head_shapes", {})
        self._tail_shapes = getattr(self, "_tail_shapes", {})
        tail = set(tail_keys(self.cfg.n_layer))
        for name, t in sd.items():
            if not name.startswith("net."):
                name = "net." + name
            if name.startswith(HEAD_PREFIX):
                self._head_shapes[name] = tuple(t.shape)
            if name in tail:
                self._tail_shapes[name] = tuple(t.shape)
            a = t.detach().to(torch.float32).cpu().contiguous().numpy()
            shape = (C.c_int64 * max(a.ndim, 1))(*a.shape) if a.ndim else (C.c_int64 * 1)(1)
            rc = self.lib.clm_load_tensor(self.ctx, name.encode(), a.ctypes.data_as(C.c_void_p), _lib.CLM_F32,
                                          shape, a.ndim)
            self._check(rc, f"clm_load_tensor({name})")

    def reserve(self, max_batch: int, max_tokens: int, token_budget: int | None = None) -> None:
        """Workspaces for batches of <= max_batch reads of <= max_tokens tokens each; `token_budget` (default
        max_batch * max_tokens) caps the padded size B * T of a batch (length-bucketed prediction: many short reads or
        few long ones per batch)."""
        budget = max_batch * max_tokens if token_budget is None else min(token_budget, max_batch * max_tokens)
        if max_batch <= self.max_batch and max_tokens <= self.max_tokens and budget <= self.token_budget:
            return
        max_batch, max_tokens = max(max_batch, self.max_batch), max(max_tokens, self.max_tokens)
        budget = min(max(budget, self.token_budget, max_tokens), max_batch * max_tokens)
        self.max_batch = self.max_tokens = self.token_budget = 0   # a failed clm_reserve leaves the context without workspaces
        self._check(self.lib.clm_reserve_tokens(self.ctx, max_batch, max_tokens, budget), "clm_reserve")
        self.max_batch, self.max_tokens, self.token_budget = max_batch, max_tokens, budget

    @property
    def native_tc_fallbacks(self) -> int:
        """Batches `clm_predict_host` redid with the fp32 convolution."""
        return int(self.lib.clm_tc_fallback_count(self.ctx))

    @property
    def launch_count(self) -> int:
        return int(self.lib.clm_launch_count(self.ctx))

    def profile(self, on: bool) -> None:
        self._check(self.lib.clm_profile_enable(self.ctx, int(on)), "clm_profile_enable")

    def profile_reset(self) -> None:
        self._check(self.lib.clm_profile_reset(self.ctx), "clm_profile_reset")

    def profile_read(self) -> dict:
        """{kernel class: (total device ms, launches)} accumulated while profiling was on."""
        out = {}
        for cat in range(self.lib.clm_profile_num()):
            ms, n = C.c_double(), C.c_longlong()
            self._check(self.lib.clm_profile_get(self.ctx, cat, C.byref(ms), C.byref(n)), "clm_profile_get")
            if n.value:
                out[self.lib.clm_profile_name(cat).decode()] = (ms.value, n.value)
        return out

    # ------------------------------------------------------------------ hot path
    def forward(self, input_ids: torch.Tensor, return_labels: bool = False, check: bool = False):
        """ClassificationLit.forward: int ids [B,T] on this device -> float32 logits [B,2].  Asynchronous on the current
        stream unless `check` (see `forward_status`)."""
        if input_ids.dim() != 2:
            raise ValueError("input_ids must be [B, T]")
        if input_ids.dtype not in _IDS_DTYPES:
            raise TypeError(f"input_ids dtype {input_ids.dtype} not supported (uint8/int32/int64)")
        ids = input_ids.to(self.device).contiguous()
        B, T = ids.shape
        self.reserve(B, T, B * T)
        logits = torch.empty(B, 2, dtype=torch.float32, device=self.device)
        labels = torch.empty(B, dtype=torch.uint8, device=self.device)
        rc = self.lib.clm_forward(self.ctx, C.c_void_p(ids.data_ptr()), _IDS_DTYPES[ids.dtype], B, T,
                                  C.c_void_p(logits.data_ptr()), C.c_void_p(labels.data_ptr()),
                                  _stream_ptr(self.device))
        self._check(rc, "clm_forward")
        self.last_seq = int(self.lib.clm_forward_seq(self.ctx))
        if check:
            # synchronous form: wait, read the forward's status word and, if the batch left the fp16 range of the
            # tensor-core convolution, redo it with the fp32 FFT kernel (the reference's fftconv is fp32)
            torch.cuda.current_stream(self.device).synchronize()
            try:
                self.forward_status(self.last_seq)
            except _lib.Fp16RangeError:
                self.tc_fallbacks += 1
                self.set_option("tc_conv", 0)
                try:
                    return self.forward(ids, return_labels=return_labels, check=True)
                finally:
                    self.set_option("tc_conv", 1)
        return (logits, labels) if return_labels else logits

    def forward_status(self, seq: int | None = None) -> None:
        """Raise if forward `seq` (default: the last one) saw a token id outside the embedding table (IndexError, like
        `nn.Embedding`) or left the fp16 range of the tensor-core convolution (Fp16RangeError).  The forward's stream
        work must be complete; the status word sits in mapped host memory, so this is a plain read."""
        if self._debug_stop:
            return   # a stopped forward never reaches the kernel that publishes the status
        self._check(self.lib.clm_forward_status(self.ctx, self.last_seq if seq is None else seq), "forward")

    def encode(self, bases: torch.Tensor, offsets: torch.Tensor, T_pad: int, *, add_cls: bool, add_sep: bool,
               pad_left: bool, max_bases: int):
        """Device tokenisation + padding: uint8 ASCII bases, int64 offsets[B+1] -> uint8 ids [B,T_pad], int32 lens."""
        B = offsets.numel() - 1
        bases = bases.to(self.device, torch.uint8).contiguous()
        offsets = offsets.to(self.device, torch.int64).contiguous()
        if bases.numel() == 0:
            bases = torch.zeros(1, dtype=torch.uint8, device=self.device)
        ids = torch.empty(B, T_pad, dtype=torch.uint8, device=self.device)
        lens = torch.empty(B, dtype=torch.int32, device=self.device)
        rc = self.lib.clm_encode_batch(self.ctx, C.c_void_p(bases.data_ptr()), C.c_void_p(offsets.data_ptr()), B, T_pad,
                                       int(add_cls), int(add_sep), int(pad_left), int(max_bases),
                                       C.c_void_p(ids.data_ptr()), C.c_void_p(lens.data_ptr()), _stream_ptr(self.device))
        self._check(rc, "clm_encode_batch")
        return ids, lens

    def predict_host(self, bases: torch.Tensor, offsets: torch.Tensor, T_pad: int, *, add_cls: bool, add_sep: bool,
                     pad_left: bool, max_bases: int, logits_out: torch.Tensor | None = None,
                     labels_out: torch.Tensor | None = None):
        """End-to-end with HOST tensors (pinned recommended): H2D, encode, forward, D2H, sync."""
        B = offsets.numel() - 1
        self.reserve(B, T_pad, B * T_pad)
        if logits_out is None:
            logits_out = torch.empty(B, 2, dtype=torch.float32).pin_memory()
        if labels_out is None:
            labels_out = torch.empty(B, dtype=torch.uint8).pin_memory()
        rc = self.lib.clm_predict_host(self.ctx, C.c_void_p(bases.data_ptr()), C.c_void_p(offsets.data_ptr()), B, T_pad,
                                       int(add_cls), int(add_sep), int(pad_left), int(max_bases),
                                       C.c_void_p(logits_out.data_ptr()), C.c_void_p(labels_out.data_ptr()))
        self._check(rc, "clm_predict_host")
        return logits_out, labels_out

    def predict_host_submit(self, bases: torch.Tensor, offsets: torch.Tensor, T_pad: int, *, add_cls: bool, add_sep: bool,
                            pad_left: bool, max_bases: int, logits_out: torch.Tensor, labels_out: torch.Tensor | None = None) -> int:
        """Enqueue one batch (HOST tensors, pinned) and return a ticket at once; `predict_host_wait(ticket)` blocks until
        `logits_out` / `labels_out` are valid.  Up to 3 batches in flight; the tensors must stay alive until the wait."""
        B = offsets.numel() - 1
        self.reserve(B, T_pad, B * T_pad)
        ticket = C.c_int(-1)
        rc = self.lib.clm_predict_host_submit(self.ctx, C.c_void_p(bases.data_ptr()), C.c_void_p(offsets.data_ptr()), B, T_pad,
                                              int(add_cls), int(add_sep), int(pad_left), int(max_bases),
                                              C.c_void_p(logits_out.data_ptr()),
                                              C.c_void_p(labels_out.data_ptr() if labels_out is not None else 0), C.byref(ticket))
        self._check(rc, "clm_predict_host_submit")
        return ticket.value

    def predict_host_wait(self, ticket: int) -> None:
        self._check(self.lib.clm_predict_host_wait(self.ctx, int(ticket)), "clm_predict_host_wait")

    # ------------------------------------------------------------------ head fine-tuning (backbone frozen)
    def head_train_begin(self, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.01,
                         dropout: float = 0.1, seed: int = 0) -> None:
        """AdamW state and step buffers for batches of up to `max_batch` reads (clm_head_train_begin): the defaults are
        torch.optim.AdamW's and the reference head's dropout p = 0.1.  Call `reserve` for the largest batch first."""
        cfg = _lib.clm_head_train_cfg(float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay),
                                      float(dropout), int(seed) & 0xFFFFFFFF)
        self._check(self.lib.clm_head_train_begin(self.ctx, C.byref(cfg)), "clm_head_train_begin")
        self.train_steps = 0

    def head_train_step(self, input_ids: torch.Tensor, targets: torch.Tensor, check: bool = True) -> torch.Tensor:
        """One optimizer step on a batch (clm_head_train_step): ids [B,T] and 0/1 targets [B] -> the batch's mean
        cross-entropy as a 0-d device tensor.  With `check` the step is synchronised and its status read: an id outside
        the embedding table raises IndexError; a batch that left the fp16 range of the tensor-core convolution changed
        no weight and is redone with the fp32 FFT convolution."""
        if input_ids.dim() != 2 or input_ids.dtype not in _IDS_DTYPES:
            raise ValueError("input_ids must be [B, T] of uint8/int32/int64")
        ids = input_ids.to(self.device).contiguous()
        B, T = ids.shape
        tgt = torch.as_tensor(targets).to(self.device, torch.int64).contiguous()
        if tgt.shape != (B,):
            raise ValueError(f"targets must have shape ({B},), got {tuple(tgt.shape)}")
        if bool(((tgt != 0) & (tgt != 1)).any()):
            raise ValueError("targets must be 0 or 1")
        if T > self.max_tokens or B * T > self.token_budget:
            raise ValueError(f"batch {B}x{T} exceeds the workspaces reserved before head_train_begin "
                             f"({self.max_batch} reads, {self.max_tokens} tokens, {self.token_budget} in all)")
        loss = torch.empty((), dtype=torch.float32, device=self.device)
        rc = self.lib.clm_head_train_step(self.ctx, C.c_void_p(ids.data_ptr()), _IDS_DTYPES[ids.dtype], B, T,
                                          C.c_void_p(tgt.data_ptr()), C.c_void_p(loss.data_ptr()), _stream_ptr(self.device))
        self._check(rc, "clm_head_train_step")
        self.last_seq = int(self.lib.clm_forward_seq(self.ctx))
        self.train_steps += 1
        if check:
            torch.cuda.current_stream(self.device).synchronize()
            try:
                self.forward_status(self.last_seq)
            except _lib.Fp16RangeError:
                self.tc_fallbacks += 1
                self.set_option("tc_conv", 0)
                try:
                    return self.head_train_step(ids, tgt, check=True)
                finally:
                    self.set_option("tc_conv", 1)
        return loss

    def tail_train_begin(self, lr: float) -> None:
        """Train the last block's tail (out_proj, norm2, fc1, fc2) and ln_f together with the head from the next step on,
        with learning rate `lr` and the head's other AdamW settings (clm_tail_train_begin).  Call after
        `head_train_begin` and before the first `head_train_step`."""
        self._check(self.lib.clm_tail_train_begin(self.ctx, float(lr)), "clm_tail_train_begin")

    def _shape(self, name: str):
        name = _full_name(name)
        return self._tail_shapes[name] if name in self._tail_shapes else self._head_shapes[name]

    def head_grad(self, name: str) -> torch.Tensor:
        """Gradient of head or tail tensor `name` (state-dict key; tail keys in full) from the last training step,
        float32 on this device."""
        shape = self._shape(name)
        out = torch.empty(int(np.prod(shape)), dtype=torch.float32, device=self.device)
        self._check(self.lib.clm_head_grad_copy(self.ctx, _full_name(name).encode(), C.c_void_p(out.data_ptr()),
                                                _stream_ptr(self.device)), "clm_head_grad_copy")
        return out.view(shape)

    def head_export(self, name: str) -> torch.Tensor:
        """Current value of head or tail tensor `name` as a CPU float32 tensor (synchronises the device)."""
        shape = self._shape(name)
        out = torch.empty(shape, dtype=torch.float32)
        self._check(self.lib.clm_head_export(self.ctx, _full_name(name).encode(), C.c_void_p(out.data_ptr())),
                    "clm_head_export")
        return out

    def head_state_dict(self) -> dict:
        """Every trainable head tensor under its state-dict name."""
        return {k: self.head_export(k) for k in self._head_shapes}

    def tail_state_dict(self) -> dict:
        """The ten tensors of the last block's tail and ln_f under their state-dict names (their loaded values when the
        tail is not in training)."""
        return {k: self.head_export(k) for k in tail_keys(self.cfg.n_layer)}

    # ------------------------------------------------------------------ evaluation on labelled reads
    def eval_step(self, input_ids: torch.Tensor, targets: torch.Tensor, check: bool = True):
        """The forward on a labelled batch plus its per-read loss (clm_eval_step): ids [B,T] and 0/1 targets [B] ->
        (logits float32 [B,2], labels uint8 [B], cross-entropy float32 [B], probability of class 1 float32 [B]), all on
        this device.  Logits and labels are `forward`'s.  With `check` (as `forward(check=True)`) the call synchronises:
        an id outside the embedding table raises IndexError, and a batch that left the fp16 range of the tensor-core
        convolution is redone with the fp32 FFT convolution."""
        if input_ids.dim() != 2 or input_ids.dtype not in _IDS_DTYPES:
            raise ValueError("input_ids must be [B, T] of uint8/int32/int64")
        ids = input_ids.to(self.device).contiguous()
        B, T = ids.shape
        tgt = torch.as_tensor(targets).to(self.device, torch.int64).contiguous()
        if tgt.shape != (B,):
            raise ValueError(f"targets must have shape ({B},), got {tuple(tgt.shape)}")
        if bool(((tgt != 0) & (tgt != 1)).any()):
            raise ValueError("targets must be 0 or 1")
        self.reserve(B, T, B * T)
        logits = torch.empty(B, 2, dtype=torch.float32, device=self.device)
        labels = torch.empty(B, dtype=torch.uint8, device=self.device)
        loss = torch.empty(B, dtype=torch.float32, device=self.device)
        prob = torch.empty(B, dtype=torch.float32, device=self.device)
        rc = self.lib.clm_eval_step(self.ctx, C.c_void_p(ids.data_ptr()), _IDS_DTYPES[ids.dtype], B, T,
                                    C.c_void_p(tgt.data_ptr()), C.c_void_p(logits.data_ptr()), C.c_void_p(labels.data_ptr()),
                                    C.c_void_p(loss.data_ptr()), C.c_void_p(prob.data_ptr()), _stream_ptr(self.device))
        self._check(rc, "clm_eval_step")
        self.last_seq = int(self.lib.clm_forward_seq(self.ctx))
        if check:
            torch.cuda.current_stream(self.device).synchronize()
            try:
                self.forward_status(self.last_seq)
            except _lib.Fp16RangeError:
                self.tc_fallbacks += 1
                self.set_option("tc_conv", 0)
                try:
                    return self.eval_step(ids, tgt, check=True)
                finally:
                    self.set_option("tc_conv", 1)
        return logits, labels, loss, prob

    # ------------------------------------------------------------------ unit-level access (tests)
    def gemm(self, A, W, bias, epi, res=None, w2=None, b2=0.0):
        M, K = A.shape
        N = W.shape[0]
        st = _stream_ptr(self.device)
        null = C.c_void_p(0)
        if epi == _lib.EPI_SCORE:
            score = torch.empty(M, dtype=torch.float32, device=self.device)
            rc = self.lib.clm_gemm(self.ctx, C.c_void_p(A.data_ptr()), C.c_void_p(W.data_ptr()), C.c_void_p(bias.data_ptr()),
                                   M, N, K, epi, null, null, C.c_void_p(w2.data_ptr()), float(b2),
                                   C.c_void_p(score.data_ptr()), st)
            self._check(rc, "clm_gemm")
            return score
        if epi == _lib.EPI_BIAS_RES_F32:
            out = torch.empty(M, N, dtype=torch.float32, device=self.device)
            rc = self.lib.clm_gemm(self.ctx, C.c_void_p(A.data_ptr()), C.c_void_p(W.data_ptr()), C.c_void_p(bias.data_ptr()),
                                   M, N, K, epi, C.c_void_p(out.data_ptr()), C.c_void_p(res.data_ptr()), null, 0.0, null, st)
        else:
            out = torch.empty(M, N, dtype=torch.bfloat16, device=self.device)
            rc = self.lib.clm_gemm(self.ctx, C.c_void_p(A.data_ptr()), C.c_void_p(W.data_ptr()), C.c_void_p(bias.data_ptr()),
                                   M, N, K, epi, C.c_void_p(out.data_ptr()), null, null, 0.0, null, st)
        self._check(rc, "clm_gemm")
        return out

    def block_in(self, layer: int, res_rows: torch.Tensor, B: int, T: int):
        """Fused LN1+in_proj+short conv+gate: res_rows fp32 [B*T,256] (row-major here) -> (vx, x0) bf16 [B,256,Tp]."""
        Tp = (T + 63) // 64 * 64
        self.reserve(B, T)
        blocked = rows_to_r32(torch.cat([res_rows, torch.zeros(160, 256, dtype=res_rows.dtype, device=res_rows.device)]))
        vx = torch.zeros(B, 256, Tp, dtype=torch.bfloat16, device=self.device)
        x0 = torch.zeros_like(vx)
        rc = self.lib.clm_block_in(self.ctx, layer, C.c_void_p(blocked.data_ptr()), B, T, Tp, C.c_void_p(vx.data_ptr()),
                                   C.c_void_p(x0.data_ptr()), _stream_ptr(self.device))
        self._check(rc, "clm_block_in")
        return vx, x0

    def block_mlp(self, layer: int, y: torch.Tensor, res: torch.Tensor) -> torch.Tensor:
        """Fused block tail: y (bf16 [M,256]), res (fp32 [M,256], row-major here; converted to the
        device's blocked layout and back) -> block output [M,256]."""
        M = y.shape[0]
        blocked = rows_to_r32(res)
        rc = self.lib.clm_block_mlp(self.ctx, layer, C.c_void_p(y.data_ptr()), C.c_void_p(blocked.data_ptr()), M,
                                    _stream_ptr(self.device))
        self._check(rc, "clm_block_mlp")
        return r32_to_rows(blocked, M)

    def block_mlp_cm(self, layer: int, y_cm: torch.Tensor, res: torch.Tensor, T: int) -> torch.Tensor:
        """Fused block tail from the channel-major conv output y_cm bf16 [B,256,Tp]; res fp32 [B*T,256]."""
        B, _, Tp = y_cm.shape
        blocked = rows_to_r32(torch.cat([res, torch.zeros(160, 256, dtype=res.dtype, device=res.device)]))
        rc = self.lib.clm_block_mlp_cm(self.ctx, layer, C.c_void_p(y_cm.data_ptr()), C.c_void_p(blocked.data_ptr()), B, T, Tp,
                                       _stream_ptr(self.device))
        self._check(rc, "clm_block_mlp_cm")
        return r32_to_rows(blocked, B * T)

    def set_option(self, name: str, value: int) -> None:
        self._check(self.lib.clm_set_option(self.ctx, name.encode(), int(value)), "clm_set_option")

    def longconv(self, layer: int, vx: torch.Tensor, x0: torch.Tensor, T: int):
        B, D, Tp = vx.shape
        out = torch.zeros_like(vx)
        rc = self.lib.clm_longconv(self.ctx, layer, C.c_void_p(vx.data_ptr()), C.c_void_p(x0.data_ptr()),
                                   C.c_void_p(out.data_ptr()), B, T, Tp, _stream_ptr(self.device))
        self._check(rc, "clm_longconv")
        return out

    def longconv_tc(self, layer: int, vx_f16: torch.Tensor, x0: torch.Tensor, T: int):
        """Tensor-core FFT long conv (2057 <= T <= 32769; zeros past T): vx fp16 [B,D,Tp], x0 bf16 -> bf16 [B,D,Tp]."""
        if vx_f16.dtype != torch.float16 or x0.dtype != torch.bfloat16:
            raise TypeError("longconv_tc takes fp16 vx and bf16 x0")
        B, D, Tp = vx_f16.shape
        out = torch.zeros_like(x0)
        rc = self.lib.clm_longconv_tc(self.ctx, layer, C.c_void_p(vx_f16.data_ptr()), C.c_void_p(x0.data_ptr()),
                                      C.c_void_p(out.data_ptr()), B, T, Tp, _stream_ptr(self.device))
        self._check(rc, "clm_longconv_tc")
        return out

    def longconv_tc_auto(self, layer: int, vx: torch.Tensor, x0: torch.Tensor, T: int):
        """Tensor-core FFT long conv on bf16 vx of any magnitude: per-channel power-of-two input scale from the data,
        fp16 conversion, kernel, output scaled back (what block_in + longconv_tc do together in the forward)."""
        if vx.dtype != torch.bfloat16 or x0.dtype != torch.bfloat16:
            raise TypeError("longconv_tc_auto takes bf16 vx and x0")
        B, D, Tp = vx.shape
        out = torch.zeros_like(x0)
        rc = self.lib.clm_longconv_tc_auto(self.ctx, layer, C.c_void_p(vx.data_ptr()), C.c_void_p(x0.data_ptr()),
                                           C.c_void_p(out.data_ptr()), B, T, Tp, _stream_ptr(self.device))
        self._check(rc, "clm_longconv_tc_auto")
        return out

    def attention_weights(self, B: int, T: int) -> torch.Tensor:
        """softmax_t of the attention-pooling scores of the last forward: float32 [B, T]."""
        out = torch.empty(B, T, dtype=torch.float32, device=self.device)
        self._check(self.lib.clm_attention_weights(self.ctx, C.c_void_p(out.data_ptr()), B, T, _stream_ptr(self.device)),
                    "clm_attention_weights")
        return out

    def longconv_variant(self, T: int) -> str:
        """Name of the long-convolution kernel `forward` uses for reads of T tokens."""
        return {0: "fft_fp32", 1: "fft_fp32_tuned", 2: "fft_tensor_core"}.get(self.lib.clm_longconv_variant(self.ctx, int(T)), "?")

    def get_filter(self, layer: int, L: int) -> torch.Tensor:
        out = torch.empty(self.cfg.d_model, L, dtype=torch.float32, device=self.device)
        self._check(self.lib.clm_get_filter(self.ctx, layer, C.c_void_p(out.data_ptr()), L, _stream_ptr(self.device)),
                    "clm_get_filter")
        return out

    def set_debug_stop(self, layer: int = -1, stage: int = -1) -> None:
        self._check(self.lib.clm_set_debug_stop(self.ctx, layer, stage), "clm_set_debug_stop")
        self._debug_stop = layer >= 0

    def debug_copy(self, what: str, shape, dtype) -> torch.Tensor:
        out = torch.empty(shape, dtype=dtype, device=self.device)
        rc = self.lib.clm_debug_copy(self.ctx, what.encode(), C.c_void_p(out.data_ptr()), out.numel() * out.element_size(),
                                     _stream_ptr(self.device))
        self._check(rc, "clm_debug_copy")
        return out


def r32_to_rows(blocked: torch.Tensor, M: int) -> torch.Tensor:
    """Undo the residual stream's blocked device layout (csrc/ptx.cuh r32_off): -> [M, 256]."""
    G = (M + 31) // 32
    return blocked.reshape(-1)[: G * 32 * 256].reshape(G, 64, 32, 4).permute(0, 2, 1, 3).reshape(G * 32, 256)[:M]


def rows_to_r32(rows: torch.Tensor) -> torch.Tensor:
    """[M, 256] -> the blocked layout, padded to whole 32-row groups."""
    M = rows.shape[0]
    G = (M + 31) // 32
    pad = torch.zeros(G * 32, 256, dtype=rows.dtype, device=rows.device)
    pad[:M] = rows
    return pad.reshape(G, 32, 64, 4).permute(0, 2, 1, 3).contiguous().reshape(-1)


def pack_reads(seqs: list[str] | list[bytes], pinned: bool = False):
    """Concatenate reads into one uint8 buffer + int64 offsets (the C-ABI's input layout)."""
    bs = [s.encode("ascii", "replace") if isinstance(s, str) else bytes(s) for s in seqs]
    offsets = np.zeros(len(bs) + 1, dtype=np.int64)
    np.cumsum([len(b) for b in bs], out=offsets[1:])
    flat = np.frombuffer(b"".join(bs), dtype=np.uint8).copy() if offsets[-1] else np.zeros(1, dtype=np.uint8)
    tb, to = torch.from_numpy(flat), torch.from_numpy(offsets)
    if pinned:
        tb, to = tb.pin_memory(), to.pin_memory()
    return tb, to
