"""Model-side mirror of the reference's predict interface.

`ChimeraLM.new()` / `.from_pretrained()` mirror `chimeralm/models/lm.py:12-61`;
`ClassificationLit.forward / predict_step` mirror `chimeralm/models/basic_module.py:67-77,
177-187` (same names, arguments and return values).  The arithmetic runs in the CUDA library
through `Engine`; there is no CPU implementation behind these classes.
"""

from __future__ import annotations

from pathlib import Path

import torch

from .config import DEFAULT_CONFIG, HyenaConfig
from .engine import Engine
from .weights import load_checkpoint, make_state_dict


class ClassificationLit:
    """Stand-in for the reference LightningModule: inference, and training of the head with the backbone frozen."""

    def __init__(self, state_dict, *, device: int | str = 0, cfg: HyenaConfig = DEFAULT_CONFIG, max_batch: int = 12,
                 max_tokens: int = 8193, save_attention: bool = False):
        self.cfg = cfg
        # `save_attention=True` (chimeralm/models/lm.py:14,30): after every forward `attention_weights` holds the pooling
        # weights [B, T, 1], like `BinarySequenceClassifier.attention_weights` (components/hyena.py:129-130)
        self.save_attention = save_attention
        self.attention_weights = None
        self.last_device_labels, self.last_forward_seq = None, 0
        self._state_dict = state_dict
        self.engine = Engine(state_dict, device=device, cfg=cfg, max_batch=max_batch, max_tokens=max_tokens)
        self.device = self.engine.device
        self.training = False

    # Lightning/torch API surface the predict path touches
    def eval(self):
        return self

    def to(self, device):
        if torch.device(device) != self.device:
            raise RuntimeError("a chimeralm_b200 model is bound to its CUDA device at construction")
        return self

    def state_dict(self):
        return self._state_dict

    def load_state_dict(self, sd, strict: bool = True):
        """Re-binds the engine to new weights (what `trainer.predict(ckpt_path=...)` does)."""
        mb, mt = self.engine.max_batch, self.engine.max_tokens
        self.engine.close()
        self._state_dict = sd
        self.engine = Engine(sd, device=self.device, cfg=self.cfg, max_batch=mb, max_tokens=mt)

    def forward(self, input_ids: torch.Tensor, input_quals: torch.Tensor | None = None) -> torch.Tensor:
        """logits [B, 2] float32; `input_quals` is accepted and ignored exactly like
        `HyenaDna.forward` ignores it (chimeralm/models/components/hyena.py:244-256).  Synchronous: the forward's
        status is checked (an out-of-range token id raises IndexError like `nn.Embedding`; a batch that leaves the
        fp16 range of the tensor-core convolution is redone with the fp32 FFT kernel)."""
        logits = self.engine.forward(input_ids, check=True)
        if self.save_attention:
            self.attention_weights = self.engine.attention_weights(*input_ids.shape).unsqueeze(-1)
        return logits

    __call__ = forward

    def configure_optimizers(self, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.01,
                             dropout: float = 0.1, seed: int = 0):
        """AdamW over the head's parameters with the backbone frozen (the reference's configure_optimizers,
        basic_module.py:200-223, optimises the whole net; here only `net.head.*` is trainable).  Workspaces must already
        cover the largest training batch (`engine.reserve`)."""
        self.engine.head_train_begin(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, dropout=dropout, seed=seed)
        self._train_begun = True
        self.training = True

    def training_step(self, batch: dict, batch_idx: int) -> torch.Tensor:
        """One optimizer step on `batch` (input_ids [B,T], labels [B] of 0/1) and its mean cross-entropy, like the
        reference's training_step (basic_module.py:87-104, model_step's F.cross_entropy) followed by the optimizer step
        Lightning takes; returns the loss as a 0-d device tensor."""
        if not getattr(self, "_train_begun", False):
            B, T = batch["input_ids"].shape
            self.engine.reserve(B, T, B * T)
            self.configure_optimizers()
        return self.engine.head_train_step(batch["input_ids"], batch["labels"])

    def predict_step(self, batch: dict, batch_idx: int):
        """Returns exactly `(logits, batch["labels"])` like the reference (basic_module.py:177-187).  The step is
        asynchronous on the current stream; the device-side argmax labels (same rule as PredictionWriter,
        callbacks.py:107) and the forward's sequence number (for `Engine.forward_status`) are left in
        `last_device_labels` / `last_forward_seq` for a caller that wants to pipeline - `Trainer.predict` does."""
        logits, labels = self.engine.forward(batch["input_ids"], return_labels=True)
        self.last_device_labels, self.last_forward_seq = labels, self.engine.last_seq
        if self.save_attention:
            self.attention_weights = self.engine.attention_weights(*batch["input_ids"].shape).unsqueeze(-1)
        return logits, batch["labels"]


class ChimeraLM:
    """Factory with the reference's two constructors."""

    @classmethod
    def new(cls, *, save_attention: bool = False, seed: int = 0, device: int | str = 0, **kw) -> ClassificationLit:
        """Random-init model of the named architecture.  (The reference's `new()` still pulls the
        pretrained HyenaDNA backbone from the Hub, components/hyena.py:237; offline the backbone
        is random-init too, seeded for reproducibility.)"""
        return ClassificationLit(make_state_dict(seed), device=device, save_attention=save_attention, **kw)

    @classmethod
    def from_pretrained(cls, model_name: str = "yangliz5/chimeralm", *, save_attention: bool = False,
                        device: int | str = 0, **kw) -> ClassificationLit:
        """Load weights from a local checkpoint: a Lightning `.ckpt`, a `.pt` state dict, a
        `.safetensors` file, or a directory holding `model.safetensors` (the Hub layout written by
        PyTorchModelHubMixin).  There is no network here, so a Hub id must already be on disk."""
        p = Path(model_name)
        if p.is_dir():
            for cand in ("model.safetensors", "pytorch_model.bin", "model.ckpt"):
                if (p / cand).exists():
                    p = p / cand
                    break
        if not p.is_file():
            raise FileNotFoundError(
                f"'{model_name}' is not a local checkpoint; downloading from the Hugging Face Hub is not possible "
                "offline. Pass --ckpt / a local path.")
        return ClassificationLit(load_checkpoint(p), device=device, save_attention=save_attention, **kw)
