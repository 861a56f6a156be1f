"""SFT loss / step on the B200 kernels -- mirror of align_anything/trainers/text_to_text/sft.py
(SupervisedTrainer.loss :95-98, .train_step :100-109).  The reference takes `outputs.loss` from the HF
model, which upcasts the whole logits tile to fp32 and materialises a (rows, V) log-softmax; here the
model is called WITHOUT labels and the cross-entropy comes from K1 + the mean-NLL epilogue
(ops.causal_lm_loss; SURVEY.md section 8f row 4).  With `fused_lm_head` there is no logits tile at all: the model
returns its last hidden states and the lm_head runs on the tcgen05 kernels over the valid rows only
(causal_lm_loss_from_model)."""
from __future__ import annotations

import warnings
from typing import Any

import torch

from ... import ops

__all__ = ['SupervisedTrainer', 'causal_lm_loss_from_model']


def causal_lm_loss_from_model(owner, model, batch: dict, labels: torch.Tensor, loss_scale: float = 1.0,
                              ignore_index: int = -100):
    """The causal-LM cross-entropy of `model(**batch)` against `labels` from the last hidden states (ops.
    causal_lm_loss_from_hidden_scaled) -> (loss_scale * loss, loss), or None where the model cannot take that path and the
    caller has to ask it for logits:
      * its forward rejects `logits_to_keep` (Qwen2AudioForConditionalGeneration): `owner.fused_lm_head` is switched off
        for good, as `_actor_logits` does with `tail_logits`;
      * its `hidden_states[-1]` is not (B, L, H) for labels (B, L) (a model that splices image / audio embeddings into the
        sequence inside its forward): this batch only.
    Order of the calls: the row plan (ops.ce_rows) is launched BEFORE the forward is enqueued, the loss reads the row
    count AFTER it -- the count copy has long finished by then, so the path adds no pipeline bubble."""
    module = getattr(model, 'module', model)
    weight = ops.lm_head_weight(module)
    rows = ops.ce_rows(labels, weight.size(0), ignore_index)
    try:
        out = model(**batch, output_hidden_states=True, logits_to_keep=1)
    except TypeError as e:
        if 'logits_to_keep' not in str(e):
            raise
        warnings.warn(f'fused_lm_head: {type(module).__name__}.forward does not take `logits_to_keep`; the cross-entropy '
                      'falls back to the logits tile', RuntimeWarning, stacklevel=3)
        owner.fused_lm_head = False
        return None
    hidden = out.hidden_states[-1]
    if hidden.dim() != 3 or tuple(hidden.shape[:2]) != tuple(labels.shape):
        warnings.warn(f'fused_lm_head: hidden states {tuple(hidden.shape)} do not line up with labels {tuple(labels.shape)}; '
                      'the cross-entropy of this batch falls back to the logits tile', RuntimeWarning, stacklevel=3)
        return None
    return ops.causal_lm_loss_from_hidden_scaled(hidden, weight, labels, loss_scale, ignore_index,
                                                 chunk_rows=getattr(owner, 'lm_head_chunk_rows', None), rows=rows)


class SupervisedTrainer:
    ignore_index = -100
    # Opt-in, as DPOTrainer.fused_lm_head: no (B, L, V) logits tile.  The model is asked for its last hidden states
    # (`output_hidden_states=True, logits_to_keep=1`) and the cross-entropy runs the lm_head on the valid rows only: K6
    # forward, K6b + the two backward GEMMs (tcgen05).  lm_head_chunk_rows: rows per d(logits) chunk of that backward.
    fused_lm_head = False
    lm_head_chunk_rows = None

    def __init__(self, cfgs, model, tokenizer=None, infer_batch=None) -> None:
        self.cfgs = cfgs
        self.model = model
        self.tokenizer = tokenizer
        self.infer_batch = infer_batch or (lambda batch: {k: v for k, v in batch.items() if k != 'meta_info'})

    def loss(self, sft_batch) -> dict[str, torch.Tensor]:
        """trainers/text_to_text/sft.py:95-98."""
        batch = dict(self.infer_batch(sft_batch))
        labels = batch.pop('labels')
        if self.fused_lm_head:
            out = causal_lm_loss_from_model(self, self.model, batch, labels, 1.0, self.ignore_index)
            if out is not None:
                return {'loss': out[0]}
        logits = self.model(**batch).logits
        return {'loss': ops.causal_lm_loss(logits, labels, self.ignore_index)}

    def train_step(self, sft_batch) -> dict[str, Any]:
        """trainers/text_to_text/sft.py:100-109."""
        loss = self.loss(sft_batch)['loss']
        self.model.backward(loss)
        self.model.step()
        with torch.no_grad():  # the loss and the device status word (out-of-range label ...) in ONE host read
            loss_val, status = torch.cat([loss.detach().float().reshape(1), ops.status_lane(loss.device)]).tolist()
        ops.raise_for_status(status, loss.device)
        return {'train/loss': loss_val, 'train/lr': self.model.optimizer.param_groups[0]['lr']}
