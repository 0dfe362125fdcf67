"""ORACLE (test infrastructure, never shipped): CPU fp32 restatement of the
`chimeralm predict` model forward.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU-baseline legs may import
this module.  The product path (`chimeralm_b200`) never does.

What is restated, and from where
--------------------------------
* Wrapper: `HyenaDna.forward` = `head(backbone(input_ids)[0], None)`
  (reference `chimeralm/models/components/hyena.py:244-256`) — no attention mask ever
  reaches the head; PAD tokens are ordinary tokens.
* Head: `BinarySequenceClassifier.forward`, attention-pooling branch
  (`components/hyena.py:79-95,117-132,142-146`), layer stack from the ctor
  (`:50-74`) and `ResidualBlock` (`:149-180`).  PINNED: `oracle/make_golden.py` imports
  the reference class by file path, loads the same weights and records its outputs in
  `tests/golden/head_golden.npz`; `tests/test_oracle.py` checks this restatement
  against them.
* Backbone: HF Hub remote code `LongSafari/hyenadna-small-32k-seqlen-hf`
  (`modeling_hyena.py`; call site `components/hyena.py:237`, executed by
  transformers 4.57.0 per the reference's `uv.lock`).  It is NOT in `/root/reference`
  and no revision is pinned there, so this part restates the published algorithm
  (SURVEY.md Appendix A.2-A.6).  PARITY UNPINNED for the backbone numerics: the
  reference holds no golden logits, forward test or fixture for it.  Independent
  cross-checks kept in `tests/test_oracle.py`: the FFT long convolution against a
  float64 direct causal sum, parameter counts against the advertised model size, and
  `fftconv` / the `pos_emb.z` table against outputs of the independent implementation of
  the same lineage in the `fla` package (`fla/modules/conv/long_conv.py`), stored in
  `tests/golden/fla_long_conv.npz` by `oracle/make_fla_golden.py`.
"""

from __future__ import annotations

import math

import torch
import torch.nn.functional as F

BB = "net.backbone.backbone."
HD = "net.head."


def implicit_filter(sd, layer: int, L: int, cfg) -> torch.Tensor:
    """HyenaFilter.filter(L) -> k [L, d_model] (A.4): MLP with sin activations over the
    positional embedding, then exponential-decay modulation."""
    p = f"{BB}layers.{layer}.mixer.filter_fn."
    z = sd[p + "pos_emb.z"][:, :L]
    t = sd[p + "pos_emb.t"][:, :L]
    h = z
    n_lin = cfg.num_inner_mlps + 1
    for j in range(n_lin):
        h = F.linear(h, sd[p + f"implicit_filter.{2 * j}.weight"], sd[p + f"implicit_filter.{2 * j}.bias"])
        h = torch.sin(sd[p + f"implicit_filter.{2 * j + 1}.freq"] * h)
    h = F.linear(h, sd[p + f"implicit_filter.{2 * n_lin}.weight"])
    decay = torch.exp(-t * sd[p + "modulation.deltas"].abs())
    return (h * (decay + cfg.shift))[0]  # [L, D]


def fftconv(u: torch.Tensor, k: torch.Tensor, D: torch.Tensor) -> torch.Tensor:
    """A.5: causal long convolution through rFFT of size 2L, fp32, plus the bias skip."""
    seqlen = u.shape[-1]
    fft_size = 2 * seqlen
    k_f = torch.fft.rfft(k, n=fft_size) / fft_size
    u_f = torch.fft.rfft(u.to(dtype=k.dtype), n=fft_size)
    y = torch.fft.irfft(u_f * k_f, n=fft_size, norm="forward")[..., :seqlen]
    out = y + u * D.unsqueeze(-1)
    return out.to(dtype=u.dtype)


def hyena_operator(sd, layer: int, u: torch.Tensor, cfg) -> torch.Tensor:
    """A.3: order-2 Hyena operator, u [B,T,D] -> [B,T,D]."""
    p = f"{BB}layers.{layer}.mixer."
    T = u.size(-2)
    l_filter = min(T, cfg.max_seq_len)
    u = F.linear(u, sd[p + "in_proj.weight"], sd[p + "in_proj.bias"])
    u = u.transpose(1, 2)  # b d l
    uc = F.conv1d(u, sd[p + "short_filter.weight"], sd[p + "short_filter.bias"],
                  padding=cfg.short_filter_order - 1, groups=cfg.inner_width)[..., :l_filter]
    x0, x1, v = uc.split(cfg.d_model, dim=1)
    k = implicit_filter(sd, layer, l_filter, cfg).transpose(0, 1)  # [D, L]
    v = fftconv(v * x1, k, sd[p + "filter_fn.bias"])
    y = (v * x0).transpose(1, 2)
    return F.linear(y, sd[p + "out_proj.weight"], sd[p + "out_proj.bias"])


def block(sd, layer: int, h: torch.Tensor, cfg) -> torch.Tensor:
    """A.6: pre-norm block with an fp32 residual stream."""
    p = f"{BB}layers.{layer}."
    D, eps = cfg.d_model, cfg.layer_norm_epsilon
    res = h.float()
    x = F.layer_norm(res, (D,), sd[p + "norm1.weight"], sd[p + "norm1.bias"], eps)
    res = hyena_operator(sd, layer, x, cfg) + res
    x = F.layer_norm(res, (D,), sd[p + "norm2.weight"], sd[p + "norm2.bias"], eps)
    y = F.linear(x, sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"])
    y = F.gelu(y, approximate="tanh")
    y = F.linear(y, sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"])
    return y + res


def backbone(sd, input_ids: torch.Tensor, cfg) -> torch.Tensor:
    """A.2: embedding -> n_layer blocks -> ln_f.  Returns last hidden state [B,T,D]."""
    h = F.embedding(input_ids, sd[BB + "embeddings.word_embeddings.weight"])
    for i in range(cfg.n_layer):
        h = block(sd, i, h, cfg)
    return F.layer_norm(h, (cfg.d_model,), sd[BB + "ln_f.weight"], sd[BB + "ln_f.bias"], cfg.layer_norm_epsilon)


def head(sd, hidden: torch.Tensor, return_attention: bool = False, return_features: bool = False,
         pooling: str = "attention"):
    """BinarySequenceClassifier.forward(hidden, attention_mask=None), attention pooling.

    components/hyena.py:117-132: scores = Linear(256->1)(GELU(Linear(256->256)(h)));
    weights = softmax over the sequence axis (dim=1) of ALL positions (mask is None);
    pooled = sum_t w_t h_t.  Classifier (:55-74): Lin(256,512) GELU Lin(512,512) GELU
    ResidualBlock(512) then output_layer Lin(512,2); dropouts are identity in eval.
    GELU here is the exact-erf flavour (nn.GELU default).
    """
    w = None
    if pooling == "attention":
        a = F.linear(hidden, sd[HD + "attention.0.weight"], sd[HD + "attention.0.bias"])
        a = F.gelu(a)
        s = F.linear(a, sd[HD + "attention.2.weight"], sd[HD + "attention.2.bias"])  # [B,T,1]
        w = torch.softmax(s, dim=1)
        pooled = (hidden * w).sum(dim=1)
    elif pooling == "mean":      # components/hyena.py:97-106 with attention_mask None
        pooled = hidden.mean(dim=1)
    elif pooling == "max":       # :107-115
        pooled = hidden.max(dim=1)[0]
    elif pooling == "cls":       # :134-136: the FIRST position
        pooled = hidden[:, 0, :]
    else:
        raise ValueError(f"Unsupported pooling type: {pooling}")
    x = F.gelu(F.linear(pooled, sd[HD + "classifier.0.weight"], sd[HD + "classifier.0.bias"]))
    x = F.gelu(F.linear(x, sd[HD + "classifier.3.weight"], sd[HD + "classifier.3.bias"]))
    r = F.linear(x, sd[HD + "classifier.6.layers.0.weight"], sd[HD + "classifier.6.layers.0.bias"])
    r = F.gelu(r)
    r = F.linear(r, sd[HD + "classifier.6.layers.3.weight"], sd[HD + "classifier.6.layers.3.bias"])
    x = r + x
    logits = F.linear(x, sd[HD + "output_layer.weight"], sd[HD + "output_layer.bias"])
    if return_features:   # input of `output_layer` (components/hyena.py:142-146), for the probe-head fit
        return logits, x
    if return_attention:
        return logits, w.squeeze(-1)
    return logits


@torch.inference_mode()
def forward(sd, input_ids: torch.Tensor, cfg, return_hidden: bool = False, return_features: bool = False):
    """ClassificationLit.forward (basic_module.py:67-77) -> logits [B,2] float32."""
    input_ids = input_ids.long()
    h = backbone(sd, input_ids, cfg)
    pooling = getattr(cfg, "pooling_type", "attention")
    if return_features:
        return head(sd, h, return_features=True, pooling=pooling)
    logits = head(sd, h, pooling=pooling)
    if return_hidden:
        return logits, h
    return logits


@torch.inference_mode()
def predict_labels(sd, input_ids: torch.Tensor, cfg) -> torch.Tensor:
    """PredictionWriter's label rule: argmax(dim=1) of the logits, no softmax
    (chimeralm/models/callbacks.py:107); exact ties resolve to index 0."""
    return forward(sd, input_ids, cfg).argmax(dim=1)


def direct_causal_conv(u: torch.Tensor, k: torch.Tensor, D: torch.Tensor) -> torch.Tensor:
    """float64 O(T^2) statement of A.5 used to cross-check `fftconv` on small cases:
    y[c,t] = sum_{s<=t} k[c,s] u[c,t-s] + D[c] u[c,t]."""
    u64, k64 = u.double(), k.double()
    Bn, C, T = u64.shape
    y = torch.zeros_like(u64)
    for s in range(T):
        y[..., s:] += k64[:, s].view(1, C, 1) * u64[..., : T - s]
    return y + u64 * D.double().view(1, C, 1)


def param_count(sd) -> dict:
    bb = sum(v.numel() for k, v in sd.items() if k.startswith(BB) and not k.endswith("pos_emb.t")
             and not (k.endswith(".freq") and ".1.freq" not in k))
    hd = sum(v.numel() for k, v in sd.items() if k.startswith(HD))
    return {"backbone": bb, "head": hd}
