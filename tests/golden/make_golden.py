"""Generate tests/golden/*.pt by running the UNMODIFIED reference (/root/reference, imported
through oracle/ref_shim.py) on small seeded inputs.  Run in the authoring container only:

    python tests/golden/make_golden.py

The fixtures hold inputs AND the reference's outputs, so the oracle port and the CUDA path
can be checked on the GPU box where /root/reference does not exist.  Sizes are tiny (odd
vocab 1031 to exercise the unaligned-row path; bf16 and fp32 variants).
"""
from __future__ import annotations

import gzip
import io
import os
import sys
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_shim  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
PAD = 1030  # resized-vocab style pad id = V - 1 (models/pretrained_model.py:118-149)


def synth_preference_batch(gen, n_pairs, L, V, pad, lens=None, interior_pad=False):
    """Mirror of PreferenceCollator's layout (datasets/text_to_text/preference.py:179-201):
    rows 0..B-1 chosen, B..2B-1 rejected, left padding, response_lens chosen first."""
    n = 2 * n_pairs
    ids = torch.randint(2, V - 1, (n, L), generator=gen)
    if lens is None:
        lens = torch.randint(2, L // 2, (n,), generator=gen).tolist()
    total = [min(L, r + int(torch.randint(1, L // 2, (1,), generator=gen))) for r in lens]
    for i in range(n):
        ids[i, : L - total[i]] = pad
    if interior_pad:  # pad == eos style tokenizers: a pad id inside the text (dpo.py:52-54 quirk)
        ids[0, L - 2] = pad
        ids[n - 1, L - lens[n - 1]] = pad
    return ids, lens


def golden_logprob(gen):
    t = ref_shim.tools()
    out = {}
    for name, dtype in (('bf16', torch.bfloat16), ('f32', torch.float32), ('f16', torch.float16)):
        logits = (torch.randn(3, 9, 1031, generator=gen) * 2.5).to(dtype)
        labels = torch.randint(0, 1031, (3, 9), generator=gen)
        view = logits[:, :-1]
        lab = labels[:, 1:]
        leaf = logits.clone().requires_grad_(True)
        res = t.gather_log_probabilities(leaf[:, :-1], lab)
        g = torch.randn(res.shape, generator=gen).to(dtype)
        res.backward(g)
        out[name] = dict(logits=logits, labels=labels, out=t.gather_log_probabilities(view, lab).detach(),
                         grad_out=g, grad_logits=leaf.grad)
    x = torch.randn(4, 11, generator=gen)
    m = torch.rand(4, 11, generator=gen) > 0.4
    out['masked_mean'] = dict(x=x, mask=m, out=t.masked_mean(x, m), out_nomask=t.masked_mean(x))
    return out


def golden_dpo(gen):
    out = {}
    V, L, B, PAD = 517, 20, 3, 516
    for modality in ('text', 'audio'):
        for name, dtype in (('bf16', torch.bfloat16), ('f32', torch.float32)):
            ids, lens = synth_preference_batch(gen, B, L, V, PAD, interior_pad=(modality == 'text'))
            if modality == 'audio':  # identical pair -> dropped (text_audio_to_text/dpo.py:138-139)
                ids[B + 1] = ids[1]
                lens[B + 1] = lens[1]
            pol = (torch.randn(2 * B, L, V, generator=gen) * 2.5).to(dtype)
            ref = (pol.float() + 0.3 * torch.randn(2 * B, L, V, generator=gen)).to(dtype)
            leaf = pol.clone().requires_grad_(True)
            tr = ref_shim.make_dpo_trainer(leaf, ref, PAD, 0.1, modality)
            batch = {'input_ids': ids, 'attention_mask': ids != PAD, 'meta_info': {'response_lens': lens}}
            lp = tr.compute_log_probs(tr.model.module, batch).detach()
            with torch.no_grad():
                rlp = tr.compute_log_probs(tr.reference_model.module, batch)
            res = tr.loss(batch)
            res['loss'].backward()
            out[f'{modality}_{name}'] = dict(
                policy_logits=pol, ref_logits=ref, input_ids=ids, response_lens=lens, pad=PAD,
                scale_coeff=0.1, policy_lp=lp, ref_lp=rlp,
                loss={k: v.detach() for k, v in res.items()}, grad_logits=leaf.grad,
            )
    return out


def golden_ppo(gen):
    out = {}
    B, Lp, V = 3, 20, 1031
    for name, dtype, vdtype in (('bf16_f32v', torch.bfloat16, torch.float32),
                                ('bf16_bf16v', torch.bfloat16, torch.bfloat16),
                                ('f32', torch.float32, torch.float32)):
        p = ref_shim.make_ppo_trainer()
        lp = (-3 * torch.rand(B, Lp, generator=gen)).to(dtype)
        rlp = (lp.float() + 0.2 * torch.randn(B, Lp, generator=gen)).to(dtype)
        newlp = (lp.float() + 0.3 * torch.randn(B, Lp, generator=gen)).to(dtype).requires_grad_(True)
        mask = torch.zeros(B, Lp, dtype=torch.bool)
        start = 6
        for b, n in enumerate((14, 9, 11)):
            mask[b, 2 : start + n] = True  # left pad of 2, prompt to `start`, n response tokens
        reward = torch.randn(B, generator=gen)
        vals = torch.randn(B, Lp, generator=gen).to(vdtype)
        newvals = (vals.float() + 0.5 * torch.randn(B, Lp, generator=gen)).to(vdtype).requires_grad_(True)
        rew = p.add_kl_divergence_regularization(reward, lp, rlp, mask)
        adv, ret = p.get_advantages_and_returns(vals, rew, mask, start)
        al = p.actor_loss_fn(newlp[:, start:], lp[:, start:], adv, mask[:, start:])
        al.backward()
        cl = p.critic_loss_fn(newvals[:, start:], vals[:, start:], ret, mask[:, start:])
        cl.backward()
        out[name] = dict(log_probs=lp, ref_log_probs=rlp, new_log_probs=newlp.detach(), mask=mask, start=start,
                         reward=reward, values=vals, new_values=newvals.detach(), rewards=rew, advantages=adv,
                         returns=ret, actor_loss=al.detach(), critic_loss=cl.detach(),
                         grad_new_log_probs=newlp.grad, grad_new_values=newvals.grad)
    return out


def golden_ppo_step(gen):
    """Whole rollout-scoring + rl_step of the text and multimodal trainers, driven through the
    reference classes with stub engines (models return fixed tensors)."""
    from oracle.ref_port import ppo_mm_rl_step, ppo_mm_rollout_scoring  # noqa: F401  (doc pointer only)

    out = {}
    B, L, V, H = 2, 18, 1031, 32
    prompt_len = 7
    ids = torch.randint(2, V - 1, (B, L), generator=gen)
    ids[0, :2] = PAD
    ids[1, :1] = PAD
    ids[0, 15:] = PAD  # right pads after eos (generation output)
    attn = ids != PAD
    for name, dtype in (('bf16', torch.bfloat16), ('f32', torch.float32)):
        actor = (torch.randn(B, L, V, generator=gen) * 2.5).to(dtype)
        refl = (actor.float() + 0.3 * torch.randn(B, L, V, generator=gen)).to(dtype)
        new_actor = (actor.float() + 0.2 * torch.randn(B, L, V, generator=gen)).to(dtype)
        end_scores = torch.randn(B, 1, generator=gen)
        critic = torch.randn(B, L, 1, generator=gen)
        new_critic = critic + 0.4 * torch.randn(B, L, 1, generator=gen)
        # ---- text variant: trainers/text_to_text/ppo.py:309-381 (engines stubbed) ----
        p = ref_shim.make_ppo_trainer(modality='text')
        t = ref_shim.tools()
        lp = t.gather_log_probabilities(actor[:, :-1], ids[:, 1:])
        rlp = t.gather_log_probabilities(refl[:, :-1], ids[:, 1:])
        reward = end_scores.squeeze(-1)
        old_vals = critic.squeeze(-1)[:, :-1]
        seq_mask = attn[:, 1:]
        start = prompt_len - 1
        rew = p.add_kl_divergence_regularization(reward, lp, rlp, seq_mask)
        adv, ret = p.get_advantages_and_returns(old_vals, rew, seq_mask, start)
        leaf = new_actor.clone().requires_grad_(True)
        nlp = t.gather_log_probabilities(leaf[:, :-1], ids[:, 1:])
        al = p.actor_loss_fn(nlp[:, start:], lp[:, start:], adv, seq_mask[:, start:])
        al.backward()
        cleaf = new_critic.clone().requires_grad_(True)
        nv = cleaf.squeeze(-1)[:, :-1]
        cl = p.critic_loss_fn(nv[:, start:], old_vals[:, start:], ret, seq_mask[:, start:])
        cl.backward()
        m = seq_mask[:, start:]
        metrics = {
            'actor_loss': al.detach(), 'reward_critic_loss': cl.detach(), 'reward': reward.mean(),
            'reward_with_kl_penalty': (rew[:, start:] * m).sum(-1).mean(),
            'reward_advantage': t.masked_mean(adv, m), 'reward_return': t.masked_mean(ret, m),
            'reward_value': t.masked_mean(nv[:, start:], m).detach(),
            'kl_divergence': ((lp - rlp)[:, start:] * m).sum(-1).mean(),
            'mean_generated_length': m.sum(-1).float().mean(), 'max_generated_length': m.sum(-1).float().max(),
        }
        out[f'text_{name}'] = dict(
            input_ids=ids, attention_mask=attn, start=start, actor_logits=actor, ref_logits=refl,
            new_actor_logits=new_actor, end_scores=end_scores, critic_scores=critic, new_critic_scores=new_critic,
            log_probs=lp, ref_log_probs=rlp, old_rewards=rew, advantages=adv, returns=ret, metrics=metrics,
            grad_actor_logits=leaf.grad, grad_critic_scores=cleaf.grad,
        )
    return out


def golden_layout(gen):
    """Integer pieces: move_padding_left (utils/tools.py:615-639), strip_pad, end index."""
    t = ref_shim.tools()
    from align_anything.trainers.text_image_to_text.ppo import move_padding_left as mpl_trainer

    ids = torch.randint(2, 50, (6, 17), generator=gen)
    pad = 0
    ids[0, :3] = pad
    ids[0, 14:] = pad
    ids[1, 10:] = pad
    ids[2, :5] = pad
    ids[3, :] = pad
    ids[4, 2] = pad  # interior pad only
    ids[5, :2] = pad
    ids[5, 8] = pad
    ids[5, 15:] = pad
    return dict(ids=ids, pad=pad, moved=t.move_padding_left(ids, pad), moved_trainer=mpl_trainer(ids.contiguous(), pad),
                stripped=[t.strip_pad(r, pad) for r in ids])


def golden_score_head(gen):
    """Run the reference's reward-model classes (tiny random-init configs) and record the
    tensors that enter / leave the scalar head (models/llama.py:49-101, opt.py)."""
    out = {}
    ref_shim.install()
    from transformers import LlamaConfig, OPTConfig

    from align_anything.models.llama import AccustomedLlamaRewardModel
    from align_anything.models.opt import AccustomedOPTRewardModel

    torch.manual_seed(7)
    cases = {
        'llama': (AccustomedLlamaRewardModel, LlamaConfig(vocab_size=128, hidden_size=64, intermediate_size=128,
                                                           num_hidden_layers=2, num_attention_heads=4,
                                                           num_key_value_heads=2, max_position_embeddings=64)),
        'opt': (AccustomedOPTRewardModel, OPTConfig(vocab_size=128, hidden_size=64, ffn_dim=128, num_hidden_layers=2,
                                                    num_attention_heads=4, max_position_embeddings=64,
                                                    word_embed_proj_dim=64)),
    }
    for key, (cls, cfg) in cases.items():
        for name, dtype in (('bf16', torch.bfloat16), ('f32', torch.float32)):
            try:
                model = cls(cfg).to(dtype).eval()
                ids = torch.randint(3, 128, (3, 12), generator=gen)
                attn = torch.ones(3, 12, dtype=torch.bool)
                attn[0, :4] = False
                attn[1, :1] = False
                attn[1, 9:] = False  # right pads after generation
                with torch.no_grad():
                    o = model(input_ids=ids, attention_mask=attn)
                out[f'{key}_{name}'] = dict(
                    last_hidden_state=o.last_hidden_state, weight=model.score_head.weight.detach(),
                    attention_mask=attn, scores=o.scores, end_scores=o.end_scores, end_index=o.end_index,
                    end_last_hidden_state=o.end_last_hidden_state,
                )
            except Exception as e:  # transformers 5.x vs reference >=4.50 drift: record, don't fail
                out[f'{key}_{name}_error'] = repr(e)
    return out


MM_RM_CONFIGS = {
    # tiny random-init configs of the three multimodal reward models the patch targets; the GPU test rebuilds the same
    # HF backbones from these kwargs (tests/test_gpu_parity.py::test_grafted_reward_model_forward_mm)
    'qwen2_vl': dict(
        text_config=dict(vocab_size=160, hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
                         num_key_value_heads=2, max_position_embeddings=128,
                         rope_scaling={'type': 'mrope', 'mrope_section': [2, 3, 3]}),
        vision_config=dict(depth=2, embed_dim=32, hidden_size=64, num_heads=4, patch_size=4, spatial_merge_size=2,
                           temporal_patch_size=2, in_chans=3),
        image_token_id=150, video_token_id=151, vision_start_token_id=152, vision_end_token_id=153),
    'llava': dict(
        text_config=dict(model_type='llama', vocab_size=160, hidden_size=64, intermediate_size=128, num_hidden_layers=2,
                         num_attention_heads=4, num_key_value_heads=2, max_position_embeddings=128),
        vision_config=dict(model_type='clip_vision_model', hidden_size=32, intermediate_size=64, num_hidden_layers=2,
                           num_attention_heads=4, image_size=16, patch_size=8, projection_dim=32),
        image_token_index=150, vision_feature_layer=-1, vision_feature_select_strategy='default'),
    'qwen2_audio': dict(
        text_config=dict(model_type='qwen2', vocab_size=160, hidden_size=64, intermediate_size=128, num_hidden_layers=2,
                         num_attention_heads=4, num_key_value_heads=2, max_position_embeddings=128),
        audio_config=dict(num_mel_bins=16, encoder_layers=2, encoder_attention_heads=2, encoder_ffn_dim=64, d_model=32,
                          max_source_positions=8),
        audio_token_index=150),
}


def golden_score_head_mm(gen):
    """The reference's multimodal reward models run for real on tiny random-init HF backbones
    (models/qwen2_vl.py:42-74, llava.py:33-76, qwen2_audio.py:52-110): records the state dict, the inputs (pixel values /
    grid / mel features included) and the ScoreModelOutput fields.  transformers here is 5.5, the reference pins >= 4.50:
    two constructor lines of the reference no longer resolve (`config.hidden_size` of the composite configs,
    `self.model.language_model.lm_head`), so `__init__` is restated below -- the `forward` under test is the reference's
    own, unmodified."""
    import copy

    from torch import nn
    from transformers import LlavaConfig, Qwen2AudioConfig, Qwen2VLConfig

    ref_shim.install()
    from align_anything.models.llava import AccustomedLlavaModel, AccustomedLlavaRewardModel
    from align_anything.models.qwen2_audio import AccustomedQwen2AudioRewardModel
    from align_anything.models.qwen2_vl import AccustomedQwen2VLRewardModel

    class LlavaRM(AccustomedLlavaRewardModel):  # __init__ only; forward = models/llava.py:47-76
        def __init__(self, config):
            super(AccustomedLlavaRewardModel, self).__init__(config)
            setattr(self, self.base_model_prefix, AccustomedLlavaModel(config))
            self.score_head = nn.Linear(config.text_config.hidden_size, 1, bias=False)

    out = {'configs': copy.deepcopy(MM_RM_CONFIGS)}
    torch.manual_seed(11)
    B, L = 2, 14

    def case(key, model, inputs):
        model = model.float().eval()
        with torch.no_grad():
            o = model(**inputs)
        out[key] = dict(
            state_dict={k: v.clone() for k, v in model.state_dict().items()}, inputs=inputs,
            scores=o.scores, end_scores=o.end_scores, end_index=o.end_index, last_hidden_state=o.last_hidden_state,
            end_last_hidden_state=o.end_last_hidden_state)

    # ---- Qwen2-VL: one 4x4-patch image per sample -> 4 merged image tokens
    cfg = Qwen2VLConfig(**copy.deepcopy(MM_RM_CONFIGS['qwen2_vl']))
    cfg.hidden_size = cfg.text_config.hidden_size  # transformers < 4.52 had it on the composite config (qwen2_vl.py:48)
    ids = torch.randint(3, 140, (B, L), generator=gen)
    ids[:, 3:7] = 150
    attn = torch.ones(B, L, dtype=torch.long)
    attn[1, :2] = 0
    case('qwen2_vl', AccustomedQwen2VLRewardModel(cfg), dict(
        input_ids=ids, attention_mask=attn, pixel_values=torch.randn(B * 16, 3 * 2 * 4 * 4, generator=gen),
        image_grid_thw=torch.tensor([[1, 4, 4]] * B), mm_token_type_ids=(ids == 150).long()))
    # ---- LLaVA: 16x16 image, 8x8 patches -> 4 image tokens
    cfg = LlavaConfig(**copy.deepcopy(MM_RM_CONFIGS['llava']))
    ids = torch.randint(3, 140, (B, L), generator=gen)
    ids[:, 2:6] = 150
    case('llava', LlavaRM(cfg), dict(input_ids=ids, attention_mask=attn.clone(),
                                     pixel_values=torch.randn(B, 3, 16, 16, generator=gen)))
    # ---- Qwen2-Audio: 16 mel frames -> 4 audio tokens after the encoder's stride-2 conv + pooling
    try:
        cfg = Qwen2AudioConfig(**copy.deepcopy(MM_RM_CONFIGS['qwen2_audio']))
        cfg.hidden_size = cfg.text_config.hidden_size
        ids = torch.randint(3, 140, (B, L), generator=gen)
        ids[:, 2:6] = 150
        attn2 = torch.ones(B, L, dtype=torch.long)
        attn2[1, 11:] = 0  # right pads: end_index comes from the mask the backbone returns
        case('qwen2_audio', AccustomedQwen2AudioRewardModel(cfg), dict(
            input_ids=ids, attention_mask=attn2, input_features=torch.randn(B, 16, 16, generator=gen),
            feature_attention_mask=torch.ones(B, 16, dtype=torch.long)))
    except Exception as e:  # version drift of the audio backbone: record, the test then skips this case
        out['qwen2_audio_error'] = repr(e)
    return out


def golden_sft(gen):
    """`outputs.loss` of a real HF causal LM (the quantity SupervisedTrainer.loss / ptx_step consume):
    tiny random-init LlamaForCausalLM, labels with -100 on the prompt and the pads."""
    from transformers import LlamaConfig, LlamaForCausalLM

    out = {}
    torch.manual_seed(11)
    cfg = LlamaConfig(vocab_size=1031, hidden_size=64, intermediate_size=128, num_hidden_layers=2,
                      num_attention_heads=4, num_key_value_heads=2, max_position_embeddings=64)
    for name, dtype in (('bf16', torch.bfloat16), ('f32', torch.float32)):
        model = LlamaForCausalLM(cfg).to(dtype).eval()
        ids = torch.randint(3, 1031, (3, 19), generator=gen)
        attn = torch.ones(3, 19, dtype=torch.bool)
        attn[0, 15:] = False
        attn[2, 12:] = False
        labels = ids.clone()
        labels[~attn] = -100
        labels[:, :5] = -100  # prompt tokens
        o = model(input_ids=ids, attention_mask=attn, labels=labels)
        o.logits.retain_grad()
        o.loss.backward()
        out[name] = dict(logits=o.logits.detach(), labels=labels, loss=o.loss.detach(), grad_logits=o.logits.grad)
    return out


def golden_saferlhf(gen):
    """Safe RLHF-V loss half driven through the reference class (saferlhf.py:432-481, 513-600, 772-793)."""
    import math

    out = {}
    B, W = 3, 23
    for name, dtype, vdtype in (('bf16_bf16v', torch.bfloat16, torch.bfloat16), ('bf16_f32v', torch.bfloat16, torch.float32),
                                ('f32', torch.float32, torch.float32)):
        p = ref_shim.make_ppo_trainer(modality='saferlhf')
        p.log_lambda = torch.tensor(math.log(1.7))
        lp = (-3 * torch.rand(B, W, generator=gen)).to(dtype)
        rlp = (lp.float() + 0.2 * torch.randn(B, W, generator=gen)).to(dtype)
        newlp = (lp.float() + 0.3 * torch.randn(B, W, generator=gen)).to(dtype).requires_grad_(True)
        reward, cost = torch.randn(B, generator=gen), torch.randn(B, generator=gen)
        rv, cv = torch.randn(B, W, generator=gen).to(vdtype), torch.randn(B, W, generator=gen).to(vdtype)
        nrv = (rv.float() + 0.5 * torch.randn(B, W, generator=gen)).to(vdtype).requires_grad_(True)
        ncv = (cv.float() + 0.5 * torch.randn(B, W, generator=gen)).to(vdtype).requires_grad_(True)
        mask = torch.ones(B, W, dtype=torch.bool)
        rew, cst = p.add_kl_divergence_regularization_with_cost(reward, cost, lp, rlp, mask)
        radv, rret = p.get_advantages_and_returns(rv, rew, mask, start=0)
        cadv, cret = p.get_advantages_and_returns(cv, cst, mask, start=0)
        al = p.actor_loss_fn_with_cost(newlp, lp, radv, cadv, mask)
        al.backward()
        rcl = p.critic_loss_fn(nrv, rv, rret, mask)
        rcl.backward()
        ccl = p.critic_loss_fn(ncv, cv, cret, mask)
        ccl.backward()
        out[name] = dict(log_probs=lp, ref_log_probs=rlp, new_log_probs=newlp.detach(), reward=reward, cost=cost,
                         reward_values=rv, cost_values=cv, new_reward_values=nrv.detach(), new_cost_values=ncv.detach(),
                         multiplier=p.log_lambda.exp().item(), rewards=rew, costs=cst, reward_advantages=radv,
                         reward_returns=rret, cost_advantages=cadv, cost_returns=cret, actor_loss=al.detach(),
                         reward_critic_loss=rcl.detach(), cost_critic_loss=ccl.detach(), grad_new_log_probs=newlp.grad,
                         grad_new_reward_values=nrv.grad, grad_new_cost_values=ncv.grad)
    return out


def golden_pairwise(gen):
    """SimPO / ORPO / KTO losses of the reference trainers (they subclass DPOTrainer) incl. d loss / d logits."""
    out = {}
    V, L, B, PAD = 517, 20, 3, 516
    for algo in ('simpo', 'orpo', 'kto'):
        for name, dtype in (('bf16', torch.bfloat16), ('f32', torch.float32)):
            ids, lens = synth_preference_batch(gen, B, L, V, PAD)
            for i in range(B):  # chosen / rejected share the prompt: the rows diverge inside the sequence
                ids[B + i, : L - lens[B + i]] = PAD
                shared = min(L - lens[i], L - lens[B + i])
                ids[B + i, max(shared - 4, 0):shared] = ids[i, max(shared - 4, 0):shared]
            ids[B + 1] = ids[1]  # an identical pair: skipped
            lens[B + 1] = lens[1]
            pol = (torch.randn(2 * B, L, V, generator=gen) * 2.5).to(dtype)
            ref = (pol.float() + 0.3 * torch.randn(2 * B, L, V, generator=gen)).to(dtype)
            leaf = pol.clone().requires_grad_(True)
            tr = ref_shim.make_dpo_trainer(leaf, ref, PAD, 0.1, algo)
            batch = {'input_ids': ids, 'attention_mask': ids != PAD, 'meta_info': {'response_lens': lens}}
            res = tr.loss(batch)
            res['loss'].backward()
            out[f'{algo}_{name}'] = dict(policy_logits=pol, ref_logits=ref, input_ids=ids, response_lens=lens, pad=PAD,
                                         scale_coeff=0.1, gamma=0.5, scale_better=1.0, scale_worse=1.33, kl=0.07,
                                         loss={k: v.detach() for k, v in res.items()}, grad_logits=leaf.grad)
    return out


def golden_grpo(gen):
    """The reference's GRPOTrainer.train_step run for real (trainers/text_to_text/grpo.py:258-318) with stubbed
    generation / reward model / engines: records the loss and d loss / d actor-logits."""
    ref_shim.install()
    import align_anything.trainers.text_to_text.grpo as ref_grpo

    out = {}
    B, G, Lp, K, V, pad, eos = 2, 3, 6, 11, 1031, 0, 5
    for name, dtype in (('bf16', torch.bfloat16), ('f32', torch.float32)):
        seq = torch.randint(6, V, (B * G, Lp + K), generator=gen)
        seq[0, :2] = pad
        seq[1, Lp + 4] = eos  # first eos: tokens after it are not counted
        seq[1, Lp + 7] = eos
        seq[3, Lp + 9:] = pad
        seq[4, Lp] = eos
        actor = (torch.randn(B * G, Lp + K, V, generator=gen) * 2.5).to(dtype)
        refl = (actor.float() + 0.3 * torch.randn(B * G, Lp + K, V, generator=gen)).to(dtype)
        rewards = torch.randn(B * G, generator=gen)
        leaf = actor.clone().requires_grad_(True)

        class Engine:
            def __init__(self, logits):
                self.logits = logits
                self.module = SimpleNamespace(parameters=lambda: iter([torch.zeros(1)]))

            def __call__(self, **kw):
                return SimpleNamespace(logits=self.logits)

            def train(self):
                pass

            def zero_grad(self):
                pass

            def backward(self, loss):
                loss.backward()

            def step(self):
                pass

        t = object.__new__(ref_grpo.GRPOTrainer)
        t.actor_model, t.actor_reference_model = Engine(leaf), Engine(refl)
        t.tokenizer = SimpleNamespace(pad_token_id=pad, eos_token_id=eos)
        t.beta, t.num_generations = 0.04, G
        t.generate_completions = lambda batch, seq=seq: seq
        t.compute_rewards = lambda s, pl, rewards=rewards: rewards
        saved = ref_grpo.get_all_reduce_mean
        ref_grpo.get_all_reduce_mean = lambda x: x  # no process group here; not arithmetic
        try:
            res = t.train_step({'input_ids': seq[:B, :Lp].clone()})
        finally:
            ref_grpo.get_all_reduce_mean = saved
        with torch.no_grad():
            lps = t._get_per_token_logps(Engine(actor), seq, None, K)
        out[name] = dict(sequences=seq, prompt_length=Lp, actor_logits=actor, ref_logits=refl, rewards=rewards,
                         num_generations=G, pad=pad, eos=eos, beta=0.04, loss=res['train/loss'], reward=res['train/reward'],
                         grad_logits=leaf.grad, per_token_logps=lps)
    return out


def golden_port_vs_reference(gen):
    """The reference's outputs on the seeded inputs of tests/test_oracle_vs_reference.py.  The test rebuilds those
    inputs from their seeds, so only the outputs are stored (`gen` is not used)."""
    sys.path.insert(0, os.path.dirname(OUT))
    import test_oracle_vs_reference as T

    dpo = {}
    for seed in range(4):
        for dtype in (torch.bfloat16, torch.float32):
            ids, lens, pad, pol, ref = T.dpo_inputs(seed, dtype)
            prev = None
            for modality in ('text', 'image', 'audio'):
                leaf = pol.clone().requires_grad_(True)
                tr = ref_shim.make_dpo_trainer(leaf, ref, pad, 0.1, modality)
                res = tr.loss({'input_ids': ids, 'attention_mask': ids != pad, 'meta_info': {'response_lens': lens}})
                res['loss'].backward()
                grad = leaf.grad
                if prev is not None and torch.equal(prev, grad):
                    grad = prev  # the text and image trainers agree: one storage in the file
                prev = grad
                dpo[(seed, str(dtype), modality)] = dict(loss={k: v.detach() for k, v in res.items()}, grad_logits=grad)
    ppo = {}
    for seed in range(3):
        ppo[seed] = []
        for c in T.ppo_inputs(seed):
            p = ref_shim.make_ppo_trainer(modality=c['modality'])
            s, lp, mask, vals = c['start'], c['lp'], c['mask'], c['vals']
            rew = p.add_kl_divergence_regularization(c['reward'], lp, c['rlp'], mask)
            adv, ret = p.get_advantages_and_returns(vals, rew, mask, s)
            ppo[seed].append(dict(rewards=rew, advantages=adv, returns=ret,
                                  actor_loss=p.actor_loss_fn(c['nlp'][:, s:], lp[:, s:], adv, mask[:, s:]),
                                  critic_loss=p.critic_loss_fn(c['nv'][:, s:], vals[:, s:], ret, mask[:, s:])))
    return dict(dpo=dpo, ppo=ppo, layout=ref_shim.tools().move_padding_left(T.layout_inputs(), 0))


def main():
    gen = torch.Generator().manual_seed(20260922)
    only = sys.argv[1:]
    parts = {
        'logprob': golden_logprob, 'dpo': golden_dpo, 'ppo': golden_ppo, 'ppo_step': golden_ppo_step,
        'layout': golden_layout, 'score_head': golden_score_head, 'score_head_mm': golden_score_head_mm, 'sft': golden_sft, 'grpo': golden_grpo, 'pairwise': golden_pairwise, 'saferlhf': golden_saferlhf,
        'port_vs_reference': golden_port_vs_reference,
    }
    compressed = {'port_vs_reference'}  # over 1 MB as a plain .pt; most of its gradient rows are zero
    for name, fn in parts.items():
        if only and name not in only:
            continue
        data = fn(gen)
        path = os.path.join(OUT, f'{name}.pt')
        if name in compressed:
            buf = io.BytesIO()
            torch.save(data, buf)
            path += '.gz'
            with gzip.GzipFile(path, 'wb', mtime=0) as f:
                f.write(buf.getvalue())
        else:
            torch.save(data, path)
        print(name, os.path.getsize(path) // 1024, 'KiB', [k for k in data])


if __name__ == '__main__':
    main()
