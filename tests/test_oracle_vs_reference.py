"""The oracle port against the unmodified reference on seeded random inputs, and the in-place graft
(`align_anything_b200.patch`) against the reference's real module tree.

The port tests rebuild their inputs from the seeds below and compare bit-exactly with what the reference
computed on them, stored in tests/golden/port_vs_reference.pt.gz (`python tests/golden/make_golden.py
port_vs_reference` regenerates it where the reference is importable).  The graft tests import the reference's
own packages and classes, so they run only where the reference is importable (AA_REFERENCE_ROOT)."""
import gzip
import io
import os

import pytest
import torch

from oracle import ref_port as O
from oracle import ref_shim

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'port_vs_reference.pt.gz')
needs_reference = pytest.mark.skipif(not ref_shim.available(),
                                     reason='needs the reference align-anything sources (AA_REFERENCE_ROOT)')


def _same(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    assert torch.equal(torch.nan_to_num(a.float()), torch.nan_to_num(b.float()))


@pytest.fixture(scope='module')
def reference_outputs():
    with gzip.open(GOLDEN, 'rb') as f:
        return torch.load(io.BytesIO(f.read()), weights_only=False)


def dpo_inputs(seed, dtype):
    gen = torch.Generator().manual_seed(seed)
    V, L, B, pad = 211 + seed, 14 + seed, 2 + seed % 2, 0
    lens = torch.randint(2, L // 2, (2 * B,), generator=gen).tolist()
    ids = torch.randint(1, V, (2 * B, L), generator=gen)
    for i, r in enumerate(lens):
        ids[i, : L - r - 2] = pad
    if seed % 2:
        ids[0, L - 2] = pad  # interior pad
    pol = (torch.randn(2 * B, L, V, generator=gen) * 2.5).to(dtype)
    ref = (pol.float() + 0.3 * torch.randn(2 * B, L, V, generator=gen)).to(dtype)
    return ids, lens, pad, pol, ref


def ppo_inputs(seed):
    """One dict per (dtype, value dtype, modality), in the order the reference was run."""
    gen = torch.Generator().manual_seed(100 + seed)
    B, W, start = 3, 17 + seed, 4
    cases = []
    for dtype, vdtype in ((torch.bfloat16, torch.float32), (torch.bfloat16, torch.bfloat16), (torch.float32, torch.float32)):
        for modality in ('text', 'image', 'audio'):
            lp = (-3 * torch.rand(B, W, generator=gen)).to(dtype)
            rlp = (lp.float() + 0.2 * torch.randn(B, W, generator=gen)).to(dtype)
            mask = torch.zeros(B, W, dtype=torch.bool)
            for b in range(B):
                mask[b, 1 : start + 3 + 2 * b] = True
            reward = torch.randn(B, generator=gen)
            vals = torch.randn(B, W, generator=gen).to(vdtype)
            nlp = (lp.float() + 0.3 * torch.randn(B, W, generator=gen)).to(dtype)
            nv = (vals.float() + 0.5 * torch.randn(B, W, generator=gen)).to(vdtype)
            cases.append(dict(modality=modality, start=start, lp=lp, rlp=rlp, mask=mask, reward=reward, vals=vals,
                              nlp=nlp, nv=nv))
    return cases


def layout_inputs():
    gen = torch.Generator().manual_seed(3)
    ids = torch.randint(0, 3, (32, 41), generator=gen)
    ids[:, :4] = 0
    return ids


@pytest.mark.parametrize('seed', range(4))
@pytest.mark.parametrize('dtype', [torch.bfloat16, torch.float32])
def test_dpo_port_vs_live_reference(seed, dtype, reference_outputs):
    ids, lens, pad, pol, ref = dpo_inputs(seed, dtype)
    for modality in ('text', 'image', 'audio'):
        want = reference_outputs['dpo'][(seed, str(dtype), modality)]
        got, grad = O.dpo_forward_backward(pol, ref, ids, lens, pad, 0.1, strip=(modality != 'audio'),
                                           skip_identical_pairs=(modality == 'audio'))
        for k, v in want['loss'].items():
            _same(got[k].detach(), v)
        _same(grad, want['grad_logits'])


@pytest.mark.parametrize('seed', range(3))
def test_ppo_port_vs_live_reference(seed, reference_outputs):
    hp = O.PPO_DEFAULTS
    for c, want in zip(ppo_inputs(seed), reference_outputs['ppo'][seed], strict=True):
        start, lp, mask, vals = c['start'], c['lp'], c['mask'], c['vals']
        _same(O.kl_shaped_rewards(c['reward'], lp, c['rlp'], mask, hp['kl_coeff'], hp['clip_range_score']), want['rewards'])
        a2, t2 = O.gae_advantages_and_returns(vals, want['rewards'], mask, start, hp['gamma'], hp['gae_lambda'])
        _same(a2, want['advantages'])
        _same(t2, want['returns'])
        _same(O.actor_loss(c['nlp'][:, start:], lp[:, start:], want['advantages'], mask[:, start:], hp['clip_range_ratio']),
              want['actor_loss'])
        _same(O.critic_loss(c['nv'][:, start:], vals[:, start:], want['returns'], mask[:, start:], hp['clip_range_value']),
              want['critic_loss'])


def test_layout_port_vs_live_reference(reference_outputs):
    _same(O.move_padding_left(layout_inputs(), 0), reference_outputs['layout'])


@needs_reference
def test_patch_installs_on_the_reference_tree():
    """`patch.install()` rebinds the hot-path names inside the real `align_anything` package and
    `uninstall()` restores them (no kernel is launched here: CPU container)."""
    ref_shim.install()
    import align_anything.trainers.text_to_text.dpo as ref_dpo
    import align_anything.trainers.text_to_text.ppo as ref_ppo
    import align_anything.utils.tools as ref_tools
    from align_anything_b200 import patch
    from align_anything_b200.trainers.text_to_text.dpo import DPOTrainer as B200DPO

    orig_gather = ref_tools.gather_log_probabilities
    orig_loss = ref_dpo.DPOTrainer.loss
    orig_gae = ref_ppo.PPOTrainer.get_advantages_and_returns
    orig_actor_step, orig_rm_step = ref_ppo.PPOTrainer.actor_step, ref_ppo.PPOTrainer.reward_model_step
    orig_rollout = ref_ppo.PPOTrainer.rollout
    done = patch.install()
    try:
        assert 'gather_log_probabilities' in done['align_anything.utils.tools']
        assert ref_tools.gather_log_probabilities is not orig_gather
        assert ref_dpo.gather_log_probabilities is ref_tools.gather_log_probabilities  # name imported into the trainer
        assert ref_dpo.DPOTrainer.loss is B200DPO.loss
        assert ref_ppo.PPOTrainer.get_advantages_and_returns is not orig_gae
        # the rollout half: ours on every PPO trainer; actor_step only where the reference does per-sample host work
        import align_anything.trainers.text_audio_to_text.ppo as ref_appo
        import align_anything.trainers.text_image_to_text.ppo as ref_mmppo
        from align_anything_b200.trainers.text_image_to_text.ppo import PPOTrainer as B200MMPPO
        from align_anything_b200.trainers.text_to_text.ppo import PPOTrainer as B200PPO
        assert ref_ppo.PPOTrainer.rollout is B200PPO.rollout and ref_ppo.PPOTrainer.rl_step is B200PPO.rl_step
        assert ref_ppo.PPOTrainer.actor_step is orig_actor_step and ref_ppo.PPOTrainer.reward_model_step is orig_rm_step
        assert ref_mmppo.PPOTrainer.rollout is B200MMPPO.rollout and ref_mmppo.PPOTrainer.actor_step is B200MMPPO.actor_step
        assert ref_mmppo.PPOTrainer.micro_batched_rollout is False and ref_appo.PPOTrainer.micro_batched_rollout is True
        assert ref_appo.PPOTrainer.rollout is B200MMPPO.rollout and ref_appo.PPOTrainer.actor_step is B200MMPPO.actor_step
        assert 'AccustomedLlamaRewardModel.forward' in done['align_anything.models.llama']
        import align_anything.trainers.text_audio_to_text.dpo as ref_adpo
        assert ref_adpo.DPOTrainer.skip_identical_pairs is True and ref_adpo.DPOTrainer.strip_pad_tokens is False
        import align_anything.trainers.text_to_text.kto as ref_kto
        import align_anything.trainers.text_to_text.simpo as ref_simpo
        from align_anything_b200.trainers.text_to_text.simpo import SimPOTrainer as B200SimPO
        assert ref_simpo.SimPOTrainer.loss is B200SimPO.loss
        assert 'KTOTrainer.loss' in done['align_anything.trainers.text_to_text.kto']
        assert ref_kto.KTOTrainer.compute_log_probs is B200DPO.compute_log_probs  # inherited from the patched DPO
        import align_anything.trainers.text_image_to_text.saferlhf as ref_safe
        from align_anything_b200.trainers.text_image_to_text.saferlhf import SafeRLHFVTrainer as B200Safe
        assert ref_safe.SafeRLHFVTrainer.rl_step is B200Safe.rl_step
        assert ref_safe.SafeRLHFVTrainer.rollout is B200MMPPO.rollout and ref_safe.SafeRLHFVTrainer.score_rollout is B200Safe.score_rollout
        assert ref_safe.SafeRLHFVTrainer.actor_loss_fn_with_cost is B200Safe.actor_loss_fn_with_cost
        # grafted methods fail loudly on CPU tensors: there is no fallback
        with pytest.raises(RuntimeError, match='no CPU fallback'):
            ref_tools.gather_log_probabilities(torch.randn(1, 3, 8), torch.zeros(1, 3, dtype=torch.int64))
    finally:
        patch.uninstall()
    assert ref_tools.gather_log_probabilities is orig_gather
    assert ref_dpo.DPOTrainer.loss is orig_loss
    assert ref_ppo.PPOTrainer.get_advantages_and_returns is orig_gae
    assert ref_ppo.PPOTrainer.rollout is orig_rollout


@needs_reference
def test_grafted_methods_find_their_helpers_on_the_reference_classes():
    """Every `self._helper(...)` a grafted method calls must exist on the patched reference class (the grafted bodies run
    on the reference's own trainer objects, which never saw our base classes)."""
    import ast
    import importlib
    import inspect
    import textwrap

    ref_shim.install()
    from align_anything_b200 import patch

    done = patch.install()
    try:
        checked = 0
        for modname, names in done.items():
            mod = importlib.import_module(modname)
            for name in names:
                if '.' not in name:
                    continue
                clsname, meth = name.split('.')
                cls = getattr(mod, clsname)
                fn = getattr(cls, meth)
                if not inspect.isfunction(fn):
                    continue
                tree = ast.parse(textwrap.dedent(inspect.getsource(fn)))
                for node in ast.walk(tree):
                    if (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute)
                            and isinstance(node.func.value, ast.Name) and node.func.value.id == 'self'
                            and node.func.attr.startswith('_') and not node.func.attr.startswith('__')):
                        assert hasattr(cls, node.func.attr), f'{modname}.{name} calls self.{node.func.attr}: not on the class'
                        checked += 1
        assert checked >= 8
    finally:
        patch.uninstall()


@needs_reference
@pytest.mark.parametrize('key', ['qwen2_vl', 'llava', 'qwen2_audio'])
def test_grafted_reward_model_forward_reaches_the_real_backbones(key, golden, monkeypatch):
    """ADVICE r1 (medium): the grafted forward must reach the multimodal backbones the way the reference's own forward
    does -- Qwen2-VL through `super().forward(**kwargs)` (pixel_values, image_grid_thw, M-RoPE), LLaVA / Qwen2-Audio
    through `self.model(...)`.  CPU container: the head tail is swapped for the oracle port here (the kernels need a
    GPU; tests/test_gpu_parity.py::test_grafted_reward_model_forward_mm runs the real tail on the B200), so what this
    pins is the backbone call of B200ScoreHeadMixin.forward on the REAL reference classes against the goldens the
    unmodified reference produced."""
    c = golden('score_head_mm')
    if key not in c:
        pytest.skip(c.get(key + '_error', 'no golden'))
    import copy

    from torch import nn
    from transformers import LlavaConfig, Qwen2AudioConfig, Qwen2VLConfig

    ref_shim.install()
    from align_anything_b200 import patch
    from align_anything_b200.models import reward_model as rm

    def oracle_tail(last_hidden_state, weight, attention_mask, end_mode='mask', upcast_scores=True, mode=None):
        r = O.score_head(last_hidden_state, weight, attention_mask, end_mode, upcast_scores)
        return rm.ScoreModelOutput(scores=r['scores'], end_scores=r['end_scores'], last_hidden_state=last_hidden_state,
                                   end_last_hidden_state=r['end_last_hidden_state'], end_index=r['end_index'])

    monkeypatch.setattr(rm, 'score_model_outputs', oracle_tail)
    kwargs = copy.deepcopy(c['configs'][key])
    done = patch.install(trainers=False)
    try:
        if key == 'qwen2_vl':
            from align_anything.models.qwen2_vl import AccustomedQwen2VLRewardModel as cls
            cfg = Qwen2VLConfig(**kwargs)
            cfg.hidden_size = cfg.text_config.hidden_size
            model = cls(cfg)
            assert cls.backbone_call == 'super' and cls._b200_super_forward is not None
        elif key == 'llava':
            from align_anything.models.llava import AccustomedLlavaModel, AccustomedLlavaRewardModel

            class cls(AccustomedLlavaRewardModel):  # constructor drift only (see make_golden.golden_score_head_mm)
                def __init__(self, config):
                    super(AccustomedLlavaRewardModel, self).__init__(config)
                    setattr(self, self.base_model_prefix, AccustomedLlavaModel(config))
                    self.score_head = nn.Linear(config.text_config.hidden_size, 1, bias=False)

            model = cls(LlavaConfig(**kwargs))
        else:
            from align_anything.models.qwen2_audio import AccustomedQwen2AudioRewardModel as cls
            cfg = Qwen2AudioConfig(**kwargs)
            cfg.hidden_size = cfg.text_config.hidden_size
            model = cls(cfg)
        assert cls.forward is rm.B200ScoreHeadMixin.forward
        model.load_state_dict(c[key]['state_dict'], strict=True)
        with torch.no_grad():
            o = model.float().eval()(**c[key]['inputs'])
    finally:
        patch.uninstall()
    want = c[key]
    torch.testing.assert_close(o.last_hidden_state, want['last_hidden_state'], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(o.scores, want['scores'], rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(o.end_scores, want['end_scores'], rtol=1e-5, atol=1e-6)
    assert torch.equal(o.end_index, want['end_index'])
    torch.testing.assert_close(o.end_last_hidden_state, want['end_last_hidden_state'], rtol=1e-5, atol=1e-6)
