"""Multimodal PPO rollout and rl_step on the B200 kernels -- mirror of
align_anything/trainers/text_image_to_text/ppo.py (move_padding_left :56-87, actor_step :174-204,
rollout :206-269, rl_step :271-379); the audio trainer (text_audio_to_text/ppo.py:217-277) runs the same
arithmetic per micro-batch (`micro_batched_rollout`).

Differences from the text trainer that matter here: sequences are rotated to full left padding,
per-sample response tails are scored (`logits[b, :-1][-R:]` against `input_ids[b, 1:][-R:]`),
`response_mask = (log_probs != 0)`, GAE starts at 0 and the losses run over the padded width."""
from __future__ import annotations

import copy
from typing import Any

import torch

from ... import ops
from ...utils.multi_process import all_reduce_packed, fused_allreduce
from ..text_to_text.ppo import METRIC_KEYS
from ..text_to_text.ppo import PPOTrainer as _TextPPOTrainer

__all__ = ['PPOTrainer', 'move_padding_left']


def move_padding_left(input_tensor: torch.Tensor, padding_value: int = 0) -> torch.Tensor:
    """trainers/text_image_to_text/ppo.py:56-87."""
    return ops.move_padding_left(input_tensor, padding_value)


def _tail_values(values_2d: torch.Tensor, lens) -> torch.Tensor:
    """pad_sequence([v[b][-R_b:] for b]) for a (B, L') tensor: one launch (and one for its gradient)."""
    return ops.tail_rows(values_2d, lens)


class PPOTrainer(_TextPPOTrainer):
    # Ask the HF model for the logits of the last W + 1 positions only (`logits_to_keep`, transformers >= 4.45 causal
    # LMs), W = the number of generated positions.  Sequences are fully left-padded after move_padding_left, so every
    # scored row lives in that tail; the (B, L, V) tile shrinks to (B, W + 1, V) -- less lm_head work, and K1b no longer
    # writes the prompt rows of zeros.  A model whose forward does not take `logits_to_keep` gets the plain call (the
    # first TypeError switches the option off); one that ignores it returns the whole tile, which works the same.
    tail_logits = True
    # Opt-in (SURVEY.md 8f rank 1): no logits tile at all.  The models are asked for their last hidden states
    # (`output_hidden_states=True, logits_to_keep=1`); rollout scoring (no gradient) runs K6, one tcgen05 kernel per
    # model, the actor's rl_step K6 + K6b + the two backward GEMMs (ops.tail_log_probs_from_hidden).
    fused_lm_head = False
    lm_head_chunk_rows = None
    # text+image / text+video: the whole prompt batch is generated and scored at once (:206-269); the audio trainer
    # loops over micro-batches of per_device_train_batch_size (text_audio_to_text/ppo.py:217-277)
    micro_batched_rollout = False

    def _tail_log_probs(self, model, batch, lens, input_ids, **kw):
        """(B, W) log-probs of the response tails, right-padded with 0 (W = lens.bound)."""
        lens = ops.as_device_lens(lens, input_ids.device)
        if self.fused_lm_head:
            out = model(**batch, output_hidden_states=True, logits_to_keep=1, **kw)
            module = getattr(model, 'module', model)
            # lens.tolist(): the host wait of the fused path (the row gather is sized on the host; cached on the DeviceLens,
            # so once per rollout).  Its cross-entropy sibling (ptx_step, SupervisedTrainer) waits on the valid-row count
            # instead, copied before the forward was enqueued (ops.CERows).
            return ops.tail_log_probs_from_hidden(out.hidden_states[-1], ops.lm_head_weight(module), input_ids,
                                                  lens.tolist(), chunk_rows=self.lm_head_chunk_rows, mode=self.mode)
        logits = self._actor_logits(model, batch, lens, **kw)
        return ops.response_tail_log_probs(logits, input_ids, lens, mode=self.mode)

    def _actor_logits(self, model, batch, lens, **kw):
        if self.tail_logits:
            try:
                return model(**batch, logits_to_keep=lens.bound + 1, **kw).logits
            except TypeError as e:  # a forward without the keyword (older / custom models): whole tiles from now on
                if 'logits_to_keep' not in str(e):
                    raise
                self.tail_logits = False
        return model(**batch, **kw).logits

    # ---- trainers/text_image_to_text/ppo.py:185-204 (after generate) -------------------------
    def postprocess_generation(self, prompt_ids: torch.Tensor, sequences: torch.Tensor):
        """move_padding_left + attention mask + response_lens = nonpad(sequence) - nonpad(prompt): ONE launch, nothing
        goes to the host (the reference does 2 `.tolist()` per sample).  The lengths come back as ops.DeviceLens."""
        return ops.rollout_layout(prompt_ids, sequences, self.tokenizer.pad_token_id)

    # ---- trainers/text_image_to_text/ppo.py:174-204 -----------------------------------------
    def actor_step(self, mini_prompt_only_batch):
        """generate, then everything the reference does on the host per sample (2 `.tolist()` + list filtering per
        sample, :190-203) as three launches and one transfer: -> (actor_batch, response_lens)."""
        infer_batch = self.infer_batch(mini_prompt_only_batch)
        actor_batch = copy.deepcopy(infer_batch)
        sequences = self.actor_model.module.generate(**infer_batch, generation_config=self.generation_config,
                                                     synced_gpus=True, do_sample=True)
        sequences, attention_mask, response_lens = self.postprocess_generation(mini_prompt_only_batch['input_ids'], sequences)
        actor_batch['input_ids'] = sequences
        actor_batch['attention_mask'] = attention_mask
        return actor_batch, response_lens

    # ---- trainers/text_image_to_text/ppo.py:206-269, text_audio_to_text/ppo.py:217-277 --------
    @torch.no_grad()
    def rollout(self, prompt_only_batch):
        self.set_train(mode=False)
        if self.micro_batched_rollout:
            total = prompt_only_batch['input_ids'].size(0)
            micro = int(self.cfgs.train_cfgs.per_device_train_batch_size)
            minis = [{key: prompt_only_batch[key][i:i + micro] for key in prompt_only_batch} for i in range(0, total, micro)]
        else:
            minis = [prompt_only_batch.copy()]
        inference_batches, training_batches = [], []
        for mini_batch in minis:
            actor_batch, response_lens = self.actor_step(mini_batch)
            inference, training = self.score_rollout(actor_batch, response_lens)
            mini_batch['input_ids'] = inference['input_ids']
            mini_batch['attention_mask'] = actor_batch['attention_mask']
            inference_batches.append(mini_batch)
            training_batches.append(training)
        self.set_train()
        return inference_batches, training_batches

    # ---- trainers/text_image_to_text/ppo.py:224-262 -----------------------------------------
    @torch.no_grad()
    def score_rollout(self, actor_batch, response_lens) -> tuple[dict, dict]:
        reward_batch = self.reward_model_step(actor_batch)
        ids = actor_batch['input_ids']
        lens = ops.as_device_lens(response_lens, ids.device)
        if ops._DUAL_K1 and not self.fused_lm_head:  # EXPERIMENTAL: both models' tiles through ONE K1 launch
            log_probs, ref_log_probs = ops.response_tail_log_probs_pair(
                self._actor_logits(self.actor_model, actor_batch, lens),
                self._actor_logits(self.actor_reference_model, actor_batch, lens), ids, lens, mode=self.mode)
        else:
            log_probs = self._tail_log_probs(self.actor_model, actor_batch, lens, ids)
            ref_log_probs = self._tail_log_probs(self.actor_reference_model, actor_batch, lens, ids)
        training = {
            'response_lens': lens,  # ops.DeviceLens: list-like for reference code, device tensor for ours
            'log_probs': log_probs,
            'ref_log_probs': ref_log_probs,
            'reward': reward_batch['reward'],
            'reward_values': _tail_values(reward_batch['reward_values'], lens),
            'response_mask': (log_probs != 0),
        }
        inference = dict(actor_batch)
        inference['input_ids'] = reward_batch['input_ids']
        return inference, training

    # ---- trainers/text_image_to_text/ppo.py:271-379 -----------------------------------------
    def rl_step(self, inference_batch, training_batch) -> dict[str, Any]:
        old_log_probs = training_batch['log_probs']
        ref_log_probs = training_batch['ref_log_probs']
        reward = training_batch['reward']
        old_reward_values = training_batch['reward_values']
        sequence_mask = training_batch['response_mask']
        input_ids = inference_batch['input_ids']
        lens = ops.as_device_lens(training_batch['response_lens'], input_ids.device)

        old_rewards, reward_advantages, reward_returns, row_stats = ops.kl_rewards_and_gae(
            reward, old_log_probs, ref_log_probs, old_reward_values, sequence_mask, 0, self.kl_coeff,
            self.clip_range_score, self.gamma, self.gae_lambda, mode=self.mode)

        # actor: K1 over the response tails + K5 as ONE autograd node; its backward is K1b alone (:296-316)
        batch = self.infer_batch(inference_batch)
        if self.fused_lm_head:
            log_probs = self._tail_log_probs(self.actor_model, batch, lens, input_ids, use_cache=False)
            actor_loss = actor_loss32 = ops.actor_loss(log_probs, old_log_probs, reward_advantages, sequence_mask,
                                                       self.clip_range_ratio, mode=self.mode)
        else:
            logits = self._actor_logits(self.actor_model, batch, lens, use_cache=False)
            actor_loss, _, actor_loss32 = ops.tail_actor_loss(logits, input_ids, lens, old_log_probs, reward_advantages,
                                                              sequence_mask, self.clip_range_ratio, mode=self.mode)
        self.actor_model.backward(actor_loss)
        self.actor_model.step()

        # critic: K5 reads `scores.squeeze(-1)[:, :-1]` through the per-sample tail indexing; one scatter launch back (:318-337)
        scores = self.reward_critic_model(**self.infer_batch(inference_batch)).scores
        reward_critic_loss, value_row_mean, critic_loss32 = ops.tail_critic_loss(
            scores, lens, old_reward_values, reward_returns, sequence_mask, self.clip_range_value, mode=self.mode)
        self.reward_critic_model.backward(reward_critic_loss)
        self.reward_critic_model.step()

        with torch.no_grad():
            fused = fused_allreduce(row_stats.device)
            stats = ops.ppo_pack_metrics(row_stats, reward, value_row_mean, actor_loss32, critic_loss32,
                                         coll=fused.next((9, 10)) if fused is not None else None)
            if fused is None:
                stats = all_reduce_packed(stats, max_lanes=(9, 10))
            v = stats.tolist()  # the ONE host sync of rollout scoring + rl_step
        ops.raise_for_status(v[10], stats.device)  # lane 10 = device status word (MAX over ranks): raise like the reference
        out = dict(zip(METRIC_KEYS, v[:10]))
        out['train/actor_lr'] = self.actor_model.optimizer.param_groups[0]['lr']
        out['train/reward_critic_lr'] = self.reward_critic_model.optimizer.param_groups[0]['lr']
        self.last_rl_tensors = {'old_rewards': old_rewards, 'advantages': reward_advantages, 'returns': reward_returns}
        return out
