"""Graft the B200 hot path into an importable `align_anything` (the reference) in place:

    import align_anything_b200.patch as p; p.install()

swaps, without touching any reference file,
  * align_anything.utils.tools.{gather_log_probabilities, masked_mean, move_padding_left}
    (and the names re-imported by the trainer modules),
  * DPOTrainer.{compute_log_probs, loss, train_step} of the text / image / audio / video trainers,
  * PPOTrainer.{rollout, actor_loss_fn, critic_loss_fn, add_kl_divergence_regularization,
    get_advantages_and_returns, rl_step, ptx_step} of the text / image / audio / video trainers, and the
    multimodal trainers' actor_step (its post-generate bookkeeping); `reward_model_step` and the text trainer's
    actor_step (generate + mask) stay the reference's,
  * SupervisedTrainer.{loss, train_step} of the text / image / audio SFT trainers (cross-entropy from K1; opt-in
    `fused_lm_head`: from the last hidden states, no logits tile),
  * GRPOTrainer.{_get_per_token_logps, train_step} and RMTrainer.{loss, train_step} of the text trainers,
  * SimPOTrainer / ORPOTrainer / KTOTrainer.{loss, train_step} (they inherit the patched DPOTrainer.compute_log_probs),
  * SafeRLHFVTrainer.{actor_step, rollout, actor_loss_fn_with_cost, add_kl_divergence_regularization_with_cost,
    rl_step} (text+image),
  * Accustomed{Llama,OPT,Llava,Qwen2VL,Qwen2Audio}RewardModel.forward (score-head tail).
The scripts/ recipes, configs, datasets, DeepSpeed engines and the model registry are used as they
are.  `uninstall()` restores the originals.  See INTEGRATION.md.
"""
from __future__ import annotations

import importlib

from .models.reward_model import B200ScoreHeadMixin
from .trainers.text_audio_to_text.dpo import DPOTrainer as _AudioDPO
from .trainers.text_audio_to_text.ppo import PPOTrainer as _AudioPPO
from .trainers.text_image_to_text.ppo import PPOTrainer as _MMPPO
from .trainers.text_image_to_text.saferlhf import SafeRLHFVTrainer as _SafeV
from .trainers.text_to_text.dpo import DPOTrainer as _TextDPO
from .trainers.text_to_text.grpo import GRPOTrainer as _GRPO
from .trainers.text_to_text.kto import KTOTrainer as _KTO
from .trainers.text_to_text.orpo import ORPOTrainer as _ORPO
from .trainers.text_to_text.ppo import PPOTrainer as _TextPPO
from .trainers.text_to_text.rm import RMTrainer as _RM
from .trainers.text_to_text.sft import SupervisedTrainer as _SFT
from .trainers.text_to_text.simpo import SimPOTrainer as _SimPO
from .utils import tools as _tools

_saved: list[tuple[object, str, object]] = []

_TOOL_NAMES = ('gather_log_probabilities', 'masked_mean', 'move_padding_left')
_DPO_METHODS = ('compute_log_probs', 'loss', 'train_step', '_hidden_and_head')
_PPO_METHODS = ('rollout', 'actor_loss_fn', 'critic_loss_fn', 'add_kl_divergence_regularization',
                'get_advantages_and_returns', 'rl_step', 'ptx_step')
_SFT_METHODS = ('loss', 'train_step')
_GRPO_METHODS = ('_get_per_token_logps', 'step_from_rollout', 'train_step')
_RM_METHODS = ('loss', 'train_step')

_DPO_TARGETS = {
    'align_anything.trainers.text_to_text.dpo': _TextDPO,
    'align_anything.trainers.text_image_to_text.dpo': _TextDPO,
    'align_anything.trainers.text_audio_to_text.dpo': _AudioDPO,
    'align_anything.trainers.text_video_to_text.dpo': _TextDPO,
}
_PPO_TARGETS = {
    'align_anything.trainers.text_to_text.ppo': _TextPPO,
    'align_anything.trainers.text_image_to_text.ppo': _MMPPO,
    'align_anything.trainers.text_audio_to_text.ppo': _AudioPPO,
    'align_anything.trainers.text_video_to_text.ppo': _MMPPO,
}
_SFT_TARGETS = {
    'align_anything.trainers.text_to_text.sft': _SFT,
    'align_anything.trainers.text_image_to_text.sft': _SFT,
    'align_anything.trainers.text_audio_to_text.sft': _SFT,
}
_GRPO_TARGETS = {'align_anything.trainers.text_to_text.grpo': _GRPO}
_RMT_TARGETS = {'align_anything.trainers.text_to_text.rm': _RM}
_SLICED_TARGETS = {
    'align_anything.trainers.text_to_text.simpo': ('SimPOTrainer', _SimPO),
    'align_anything.trainers.text_to_text.orpo': ('ORPOTrainer', _ORPO),
    'align_anything.trainers.text_to_text.kto': ('KTOTrainer', _KTO),
}
_SAFE_TARGET = 'align_anything.trainers.text_image_to_text.saferlhf'
_SAFE_METHODS = ('actor_step', 'rollout', 'score_rollout', 'postprocess_generation', 'actor_loss_fn_with_cost', 'add_kl_divergence_regularization_with_cost', 'update_lambda', '_lambda_step',
                 'rl_step', '_actor_logits', '_tail_log_probs', 'actor_loss_fn', 'critic_loss_fn',
                 'get_advantages_and_returns')
# (module, class, end_mode, upcast_scores, mask_from_outputs, backbone_call)
_RM_TARGETS = (
    ('align_anything.models.llama', 'AccustomedLlamaRewardModel', 'mask', True, False, 'prefix'),
    ('align_anything.models.opt', 'AccustomedOPTRewardModel', 'mask', True, False, 'prefix'),
    ('align_anything.models.llava', 'AccustomedLlavaRewardModel', 'last', True, False, 'prefix'),
    ('align_anything.models.qwen2_vl', 'AccustomedQwen2VLRewardModel', 'last', False, False, 'super'),
    ('align_anything.models.qwen2_audio', 'AccustomedQwen2AudioRewardModel', 'mask', True, True, 'prefix'),
)


def graft_score_head(cls, end_mode: str, upcast: bool, from_outputs: bool, backbone_call: str = 'prefix') -> None:
    """Bind B200ScoreHeadMixin.forward and its selectors onto one reward-model class (recorded for uninstall())."""
    import inspect

    attrs = [('end_mode', end_mode), ('upcast_scores', upcast), ('mask_from_outputs', from_outputs),
             ('backbone_call', backbone_call)]
    if backbone_call == 'super':
        parent = next(b for b in cls.__mro__[1:] if 'forward' in b.__dict__)
        fn = parent.__dict__['forward']
        try:
            takes_keep = 'logits_to_keep' in inspect.signature(fn).parameters
        except (TypeError, ValueError):
            takes_keep = False
        attrs += [('_b200_super_forward', fn), ('_b200_super_kwargs', {'logits_to_keep': 1} if takes_keep else {})]
    attrs.append(('forward', B200ScoreHeadMixin.forward))
    for attr, val in attrs:
        _saved.append((cls, attr, cls.__dict__.get(attr, None)))
        setattr(cls, attr, val)


def _swap(obj, name, new):
    if not hasattr(obj, name):
        return False
    _saved.append((obj, name, obj.__dict__.get(name, getattr(obj, name))))
    setattr(obj, name, new)
    return True


def _try_import(modname):
    try:
        return importlib.import_module(modname)
    except Exception:  # optional modality (e.g. video needs `av`)
        return None


def install(trainers: bool = True, models: bool = True) -> dict[str, list[str]]:
    """Returns what was patched, keyed by module name."""
    done: dict[str, list[str]] = {}
    ref_tools = _try_import('align_anything.utils.tools')
    if ref_tools is None:
        raise ImportError('`align_anything` is not importable: nothing to patch')
    for n in _TOOL_NAMES:
        if _swap(ref_tools, n, getattr(_tools, n)):
            done.setdefault('align_anything.utils.tools', []).append(n)
    if trainers:
        for modname, src in {**_DPO_TARGETS, **_PPO_TARGETS, **_SFT_TARGETS, **_GRPO_TARGETS, **_RMT_TARGETS}.items():
            mod = _try_import(modname)
            if mod is None:
                continue
            for n in _TOOL_NAMES:  # names imported with `from ...tools import x`
                if n in mod.__dict__ and _swap(mod, n, getattr(_tools, n)):
                    done.setdefault(modname, []).append(n)
            cls = (getattr(mod, 'DPOTrainer', None) or getattr(mod, 'PPOTrainer', None)
                   or getattr(mod, 'SupervisedTrainer', None) or getattr(mod, 'GRPOTrainer', None)
                   or getattr(mod, 'RMTrainer', None))
            if cls is None:
                continue
            methods = (_DPO_METHODS if modname in _DPO_TARGETS else _PPO_METHODS if modname in _PPO_TARGETS else
                       _GRPO_METHODS if modname in _GRPO_TARGETS else _RM_METHODS if modname in _RMT_TARGETS else
                       _SFT_METHODS)
            for m in methods:
                if m in ('step_from_rollout', '_hidden_and_head') or m in cls.__dict__ or any(m in b.__dict__ for b in cls.__mro__[1:]):
                    fn = src.__dict__.get(m) or next(b.__dict__[m] for b in src.__mro__ if m in b.__dict__)
                    _saved.append((cls, m, cls.__dict__.get(m, None)))
                    setattr(cls, m, fn)
                    done.setdefault(modname, []).append(f'{cls.__name__}.{m}')
            if modname in _DPO_TARGETS:  # class attributes the grafted methods read
                for attr in ('strip_pad_tokens', 'skip_identical_pairs', 'mode', 'fused_lm_head', 'lm_head_chunk_rows'):
                    _saved.append((cls, attr, cls.__dict__.get(attr, None)))
                    setattr(cls, attr, getattr(src, attr))
            elif modname in _PPO_TARGETS or modname in _GRPO_TARGETS:
                _saved.append((cls, 'mode', cls.__dict__.get('mode', None)))
                setattr(cls, 'mode', None)
                if modname in _PPO_TARGETS:  # helpers the grafted rl_step calls + the B200-side entry points
                    helpers = ('_actor_logits', '_tail_log_probs', 'score_rollout', 'postprocess_generation')
                    if src is not _TextPPO:  # multimodal: the post-generate bookkeeping of actor_step is ours too
                        helpers += ('actor_step',)
                    for m in helpers:
                        fn = next((b.__dict__[m] for b in src.__mro__ if m in b.__dict__), None)
                        if fn is not None:
                            _saved.append((cls, m, cls.__dict__.get(m, None)))
                            setattr(cls, m, fn)
                            done.setdefault(modname, []).append(f'{cls.__name__}.{m}')
                    for attr in ('tail_logits', 'fused_lm_head', 'lm_head_chunk_rows', 'micro_batched_rollout'):
                        if hasattr(src, attr):
                            _saved.append((cls, attr, cls.__dict__.get(attr, None)))
                            setattr(cls, attr, getattr(src, attr))
            elif modname in _SFT_TARGETS:  # class attributes the grafted loss reads (its helper is a module function)
                for attr, val in (('ignore_index', -100), ('fused_lm_head', False), ('lm_head_chunk_rows', None)):
                    _saved.append((cls, attr, cls.__dict__.get(attr, None)))
                    setattr(cls, attr, val)
        for modname, (clsname, src) in _SLICED_TARGETS.items():
            mod = _try_import(modname)
            cls = getattr(mod, clsname, None) if mod is not None else None
            if cls is None:
                continue
            for m in ('loss', 'train_step', '_pair_terms', '_pack'):
                fn = next(b.__dict__[m] for b in src.__mro__ if m in b.__dict__)
                _saved.append((cls, m, cls.__dict__.get(m, None)))
                setattr(cls, m, fn)
                done.setdefault(modname, []).append(f'{clsname}.{m}')
        mod = _try_import(_SAFE_TARGET)
        cls = getattr(mod, 'SafeRLHFVTrainer', None) if mod is not None else None
        if cls is not None:
            for m in _SAFE_METHODS:
                fn = next(b.__dict__[m] for b in _SafeV.__mro__ if m in b.__dict__)
                _saved.append((cls, m, cls.__dict__.get(m, None)))
                setattr(cls, m, fn)
                done.setdefault(_SAFE_TARGET, []).append(f'SafeRLHFVTrainer.{m}')
            for attr, val in (('mode', None), ('tail_logits', False), ('fused_lm_head', False), ('lm_head_chunk_rows', None),
                              ('micro_batched_rollout', False)):
                _saved.append((cls, attr, cls.__dict__.get(attr, None)))
                setattr(cls, attr, val)
    if models:
        for modname, clsname, end_mode, upcast, from_outputs, backbone_call in _RM_TARGETS:
            mod = _try_import(modname)
            cls = getattr(mod, clsname, None) if mod is not None else None
            if cls is None:
                continue
            graft_score_head(cls, end_mode, upcast, from_outputs, backbone_call)
            done.setdefault(modname, []).append(f'{clsname}.forward')
    return done


def uninstall() -> None:
    while _saved:
        obj, name, old = _saved.pop()
        if old is None:
            try:
                delattr(obj, name)
            except AttributeError:
                pass
        else:
            setattr(obj, name, old)
