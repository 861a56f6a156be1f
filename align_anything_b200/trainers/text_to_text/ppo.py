"""PPO rollout scoring and rl_step on the B200 kernels -- mirror of
align_anything/trainers/text_to_text/ppo.py (reward_model_step :224-242, rollout :244-289,
actor_loss_fn :291-307, rl_step :309-398, get_advantages_and_returns :487-508, critic_loss_fn
:510-526, add_kl_divergence_regularization :528-547).

Generation itself (`model.generate`), engine construction and the data loaders are out of scope and stay
in the reference; the methods below read the same attributes from `self`:
    self.actor_model, self.actor_reference_model, self.reward_model, self.reward_critic_model,
    self.kl_coeff, self.clip_range_ratio, self.clip_range_score, self.clip_range_value,
    self.gamma, self.gae_lambda, self.tokenizer, self.reward_tokenizer
"""
from __future__ import annotations

import copy
from typing import Any

import torch

from ... import ops
from ...utils.multi_process import all_reduce_packed, fused_allreduce
from .sft import causal_lm_loss_from_model

__all__ = ['PPOTrainer']

METRIC_KEYS = ('train/actor_loss', 'train/reward_critic_loss', 'train/reward', 'train/reward_with_kl_penalty',
               'train/reward_advantage', 'train/reward_return', 'train/reward_value', 'train/kl_divergence',
               'train/mean_generated_length', 'train/max_generated_length')


class PPOTrainer:
    mode = None  # None -> 'faithful'

    def __init__(self, cfgs=None, actor_model=None, actor_reference_model=None, reward_model=None,
                 reward_critic_model=None, tokenizer=None, reward_tokenizer=None, *, kl_coeff=0.02,
                 clip_range_ratio=0.2, clip_range_score=50.0, clip_range_value=5.0, gamma=1.0,
                 gae_lambda=0.95) -> None:
        self.cfgs = cfgs
        self.actor_model = actor_model
        self.actor_reference_model = actor_reference_model
        self.reward_model = reward_model
        self.reward_critic_model = reward_critic_model
        self.tokenizer = tokenizer
        self.reward_tokenizer = reward_tokenizer if reward_tokenizer is not None else tokenizer
        tc = getattr(cfgs, 'train_cfgs', None) if cfgs is not None else None

        def pick(name, default):  # trainers/text_to_text/ppo.py:87-93 reads these from cfgs.train_cfgs
            v = getattr(tc, name, None) if tc is not None else None
            return default if v is None else v

        self.kl_coeff = pick('kl_coeff', kl_coeff)
        self.clip_range_ratio = pick('clip_range_ratio', clip_range_ratio)
        self.clip_range_score = pick('clip_range_score', clip_range_score)
        self.clip_range_value = pick('clip_range_value', clip_range_value)
        self.gamma = pick('gamma', gamma)
        self.gae_lambda = pick('gae_lambda', gae_lambda)
        self.ptx_coeff = pick('ptx_coeff', 16.0)
        self.infer_batch = lambda batch: {k: v for k, v in batch.items() if k != 'meta_info'}
        self.reward_infer_batch = self.infer_batch

    # ---- the four loss-path functions, drop-in signatures -----------------------------------
    def actor_loss_fn(self, log_probs, old_log_probs, advantages, mask) -> torch.Tensor:
        """trainers/text_to_text/ppo.py:291-307."""
        return ops.actor_loss(log_probs, old_log_probs, advantages, mask, self.clip_range_ratio, mode=self.mode)

    def critic_loss_fn(self, values, old_values, returns, mask) -> torch.Tensor:
        """trainers/text_to_text/ppo.py:510-526."""
        return ops.critic_loss(values, old_values, returns, mask, self.clip_range_value, mode=self.mode)

    def add_kl_divergence_regularization(self, reward, log_probs, ref_log_probs, sequence_mask) -> torch.Tensor:
        """trainers/text_to_text/ppo.py:528-547 (K4; rl_step below fuses it with the GAE scan)."""
        W = log_probs.size(-1)
        dummy = torch.zeros((log_probs.size(0), W), dtype=torch.float32, device=log_probs.device)
        old_rewards, _, _, _ = ops.kl_rewards_and_gae(
            reward, log_probs, ref_log_probs, dummy, sequence_mask, W - 1, self.kl_coeff, self.clip_range_score,
            self.gamma, self.gae_lambda, mode=self.mode)
        return old_rewards

    def get_advantages_and_returns(self, values, rewards, sequence_mask, start):
        """trainers/text_to_text/ppo.py:487-508."""
        adv, ret, _ = ops.gae_from_rewards(values, rewards, sequence_mask, start, self.gamma, self.gae_lambda,
                                           mode=self.mode)
        return adv.detach(), ret

    # ---- trainers/text_to_text/ppo.py:224-242 -----------------------------------------------
    def reward_model_step(self, actor_batch) -> dict[str, Any]:
        reward_batch = copy.copy(actor_batch)
        if self.reward_tokenizer is not self.tokenizer:
            raise NotImplementedError('re-tokenisation for a different reward tokenizer is host-side text '
                                      'processing (utils/tools.py batch_retokenize) and out of scope')
        reward_batch['reward'] = self.reward_model(**self.reward_infer_batch(reward_batch)).end_scores.squeeze(dim=-1)
        scores = self.reward_critic_model(**self.reward_infer_batch(actor_batch)).scores
        reward_batch['reward_values'] = scores.squeeze(dim=-1)[:, :-1]
        return reward_batch

    # ---- trainers/text_to_text/ppo.py:209-222 and base/rl_trainer.py:274-286 -------------------
    def actor_step(self, mini_prompt_only_batch) -> dict[str, Any]:
        """Generation + attention mask.  patch.install() keeps the reference's own method for the text trainer (it is
        already free of host syncs); this one serves the stand-alone mirror."""
        infer_batch = self.infer_batch(mini_prompt_only_batch)
        actor_batch = copy.deepcopy(infer_batch)
        sequences = self.actor_model.module.generate(**infer_batch, generation_config=self.generation_config,
                                                     synced_gpus=True, do_sample=True)
        actor_batch['input_ids'] = sequences
        actor_batch['attention_mask'] = sequences.not_equal(self.tokenizer.pad_token_id)
        return actor_batch

    def set_train(self, mode: bool = True) -> None:
        for engine in (self.actor_model, self.reward_critic_model):
            fn = getattr(engine, 'train' if mode else 'eval', None)
            if callable(fn):
                fn()

    # ---- trainers/text_to_text/ppo.py:244-289 -------------------------------------------------
    @torch.no_grad()
    def rollout(self, prompt_only_batch):
        """Micro-batched generation + scoring -> (inference_batches, training_batches), the lists the reference's
        train() loop zips into rl_step (:430-447)."""
        self.set_train(mode=False)
        total = prompt_only_batch['input_ids'].size(0)
        micro = int(self.cfgs.train_cfgs.per_device_train_batch_size)
        inference_batches, training_batches = [], []
        for i in range(0, total, micro):
            mini_batch = {key: prompt_only_batch[key][i:i + micro] for key in prompt_only_batch}
            actor_batch = self.actor_step(mini_batch)
            inference, training = self.score_rollout(actor_batch, mini_batch['input_ids'].size(-1))
            mini_batch['input_ids'] = inference['input_ids']
            mini_batch['attention_mask'] = inference['attention_mask']
            inference_batches.append(mini_batch)
            training_batches.append(training)
        self.set_train()
        return inference_batches, training_batches

    # ---- scoring half of rollout(), trainers/text_to_text/ppo.py:262-283 ---------------------
    @torch.no_grad()
    def score_rollout(self, actor_batch, prompt_len: int) -> tuple[dict, dict]:
        """Everything rollout() does after generation for one mini-batch: reward / critic scoring and
        the actor / reference log-probs of every next token."""
        reward_batch = self.reward_model_step(actor_batch)
        logits = self.actor_model(**actor_batch).logits
        ref_logits = self.actor_reference_model(**actor_batch).logits
        ids = actor_batch['input_ids']
        training = {
            'prompt_idx': prompt_len - 1,
            'log_probs': ops.gather_log_probabilities(logits[:, :-1], ids[:, 1:], mode=self.mode),
            'ref_log_probs': ops.gather_log_probabilities(ref_logits[:, :-1], ids[:, 1:], mode=self.mode),
            'reward': reward_batch['reward'],
            'reward_values': reward_batch['reward_values'],
        }
        inference = {'input_ids': reward_batch['input_ids'], 'attention_mask': actor_batch['attention_mask']}
        return inference, training

    # ---- trainers/text_to_text/ppo.py:400-408 -----------------------------------------------
    def ptx_step(self, ptx_batch) -> dict[str, Any]:
        """PTX (pre-training mix) term: the HF causal-LM loss, taken from K1 instead of `outputs.loss`."""
        from ...utils.multi_process import get_all_reduce_mean

        batch = dict(self.infer_batch(ptx_batch))
        labels = batch.pop('labels')
        out = None
        if getattr(self, 'fused_lm_head', False):  # multimodal trainers: the lm_head on the valid rows, no logits tile
            out = causal_lm_loss_from_model(self, self.actor_model, batch, labels, self.ptx_coeff)
        if out is None:
            logits = self.actor_model(**batch).logits
            # `ptx_coeff * ptx_loss` (:405): the gradient tile comes out of the single pass already multiplied
            out = ops.causal_lm_loss_scaled(logits, labels, self.ptx_coeff)
        scaled_loss, ptx_loss = out
        self.actor_model.backward(scaled_loss)
        self.actor_model.step()
        ptx_loss = get_all_reduce_mean(ptx_loss.detach())
        return {'train/ptx_loss': ptx_loss.item()}

    # ---- trainers/text_to_text/ppo.py:309-398 -----------------------------------------------
    def rl_step(self, inference_batch, training_batch) -> dict[str, Any]:
        old_log_probs = training_batch['log_probs']
        ref_log_probs = training_batch['ref_log_probs']
        reward = training_batch['reward']
        old_reward_values = training_batch['reward_values']
        start = training_batch['prompt_idx']
        input_ids = inference_batch['input_ids']
        sequence_mask = inference_batch['attention_mask'][:, 1:]

        old_rewards, reward_advantages, reward_returns, row_stats = ops.kl_rewards_and_gae(
            reward, old_log_probs, ref_log_probs, old_reward_values, sequence_mask, start, self.kl_coeff,
            self.clip_range_score, self.gamma, self.gae_lambda, mode=self.mode)

        logits = self.actor_model(**inference_batch, use_cache=False).logits
        # the reference scores every position and then slices `[:, start:]` (:338-346); only those rows are ever used, so
        # only they are read here.  One autograd node (K1f): log-probs, d loss / d log-prob and the gradient tile in a
        # single pass over the response rows; the prompt rows of the tile are written as zeros by the same kernel.
        actor_loss, _, actor_loss32 = ops.dense_actor_loss(logits, input_ids, start, old_log_probs[:, start:],
                                                           reward_advantages, sequence_mask[:, start:],
                                                           self.clip_range_ratio, mode=self.mode)
        self.actor_model.backward(actor_loss)
        self.actor_model.step()

        reward_values = self.reward_critic_model(**inference_batch).scores
        reward_values = reward_values.squeeze(dim=-1)[:, :-1]
        reward_critic_loss, value_row_mean = ops.critic_loss(
            reward_values[:, start:], old_reward_values[:, start:], reward_returns, sequence_mask[:, start:],
            self.clip_range_value, mode=self.mode, return_row_mean=True)
        self.reward_critic_model.backward(reward_critic_loss)
        self.reward_critic_model.step()

        with torch.no_grad():
            fused = fused_allreduce(row_stats.device)
            stats = ops.ppo_pack_metrics(row_stats, reward, value_row_mean, actor_loss32, reward_critic_loss,
                                         coll=fused.next((9, 10)) if fused is not None else None)
            if fused is None:
                stats = all_reduce_packed(stats, max_lanes=(9, 10))  # ONE collective (reference: 10 + barrier)
            v = stats.tolist()  # ONE host sync (reference: 12 .item())
        ops.raise_for_status(v[10], stats.device)  # lane 10 = device status word (MAX over ranks): raise like the reference
        out = dict(zip(METRIC_KEYS, v[:10]))
        out['train/actor_lr'] = self.actor_model.optimizer.param_groups[0]['lr']
        out['train/reward_critic_lr'] = self.reward_critic_model.optimizer.param_groups[0]['lr']
        # the per-token tensors stay OUT of the returned dict: the reference hands it to Logger.log -> add_scalar /
        # wandb.log (utils/logger.py:130-138), which takes scalars only.  Tests read them from this attribute.
        self.last_rl_tensors = {'old_rewards': old_rewards, 'advantages': reward_advantages, 'returns': reward_returns}
        return out
