"""CPU checks of the cross-entropy-from-hidden-states path (SupervisedTrainer / ptx_step with `fused_lm_head`): argument
validation of aa_ce_rows in the real library, and a dry run of the Python layer against a stand-in library that checks
every call against its declared ctypes signature (the `_FakeLib` of test_cpu_plumbing.py).  No kernel runs here, so no
number is checked: what is pinned is which entry points each branch reaches, the autograd wiring, the fallbacks, the
graft of the new trainer attributes and the scalar-only metric dicts."""
import ctypes
import math
import sys
import types
import warnings
from types import SimpleNamespace

import pytest
import torch

from test_cpu_plumbing import _FakeLib


def test_ce_rows_argument_errors_need_no_gpu():
    from align_anything_b200 import _lib

    lib = _lib.lib()
    buf = (ctypes.c_int64 * 8)()
    p = ctypes.cast(buf, ctypes.c_void_p).value
    q, r = p + 16, p + 32
    for B, L, V in ((0, 4, 10), (2, 0, 10), (2, 4, 0), (-1, 4, 10)):
        rc = lib.aa_ce_rows(p, B, L, L, 1, -100, V, q, r, r + 8, None, None)
        assert rc == -2 and b'bad sizes' in lib.aa_last_error(), (B, L, V, rc)
    rc = lib.aa_ce_rows(None, 2, 4, 4, 1, -100, 10, q, r, r + 8, None, None)
    assert rc == -2 and b'null pointer' in lib.aa_last_error()
    rc = lib.aa_ce_rows(p, 2, 4, 4, 1, -100, 10, q, q, r + 8, None, None)
    assert rc == -2 and b'aliased' in lib.aa_last_error()
    assert 'aa_ce_rows' in _lib.EXPORTED_SYMBOLS


@pytest.fixture
def dry(monkeypatch):
    """The stand-in library, CPU tensors accepted, and the valid-row count stubbed to `dry.n_valid` (the count would come
    back from the device)."""
    from align_anything_b200 import _lib, ops

    lib = _FakeLib(_lib._SIGS)
    lib.n_valid = 7
    monkeypatch.setattr(_lib, 'lib', lambda: lib)
    monkeypatch.setattr(_lib, 'require_cuda', lambda *t: None)
    monkeypatch.setattr(_lib, 'stream_ptr', lambda device=None: 0)
    monkeypatch.setattr(torch, 'empty', torch.zeros)
    monkeypatch.setattr(ops, '_scratch', {})
    monkeypatch.setattr(ops, '_FUSED_MIN_ROW_BYTES', 0)
    monkeypatch.setattr(ops, '_device_scratch', lambda device: ops._scratch.setdefault('cpu', {
        'status': torch.zeros(1, dtype=torch.int32), 'counter': torch.zeros(8, dtype=torch.int32)}))

    def start_count_copy(self):
        self._n = lib.n_valid

    monkeypatch.setattr(ops.CERows, '_start_count_copy', start_count_copy)
    ops._dense_plan.cache_clear()
    yield lib
    ops._dense_plan.cache_clear()


class _HiddenModel:
    """DeepSpeed-engine-shaped model that returns `hidden_states` when asked for them and `logits` otherwise, and records
    the keyword arguments of every call."""

    def __init__(self, hidden, weight, logits=None, takes_keep=True):
        self.module = self
        self.h, self.w, self.logits, self.takes_keep = hidden, weight, logits, takes_keep
        self.calls = []
        self.optimizer = SimpleNamespace(param_groups=[{'lr': 1e-6}])

    def __call__(self, **kw):
        self.calls.append({k: v for k, v in kw.items() if k not in ('input_ids', 'attention_mask')})
        if 'logits_to_keep' in kw and not self.takes_keep:
            raise TypeError("forward() got an unexpected keyword argument 'logits_to_keep'")
        if kw.get('output_hidden_states'):
            return SimpleNamespace(hidden_states=(self.h,), logits=None)
        return SimpleNamespace(logits=self.logits)

    def get_output_embeddings(self):
        return SimpleNamespace(weight=self.w)

    def backward(self, loss):
        loss.backward()

    def step(self):
        pass


def _sft_inputs(B=2, L=9, H=64, V=101):
    hidden = torch.randn(B, L, H).bfloat16().requires_grad_(True)
    weight = torch.randn(V, H).bfloat16().requires_grad_(True)
    labels = torch.randint(0, V, (B, L))
    labels[:, :3] = -100
    batch = {'input_ids': labels.clamp(min=0), 'labels': labels, 'attention_mask': torch.ones_like(labels)}
    return hidden, weight, batch


LM_HEAD_CHAIN = {'aa_ce_rows', 'aa_linear_logprob_fwd', 'aa_linear_dlogits', 'aa_linear_dhidden', 'aa_linear_dweight',
                 'aa_nll_mean'}


def test_fused_sft_step_runs_the_lm_head_chain_and_never_the_logits_kernels(dry):
    from align_anything_b200.trainers.text_to_text.sft import SupervisedTrainer

    hidden, weight, batch = _sft_inputs()
    model = _HiddenModel(hidden, weight)
    tr = SupervisedTrainer(None, model)
    tr.fused_lm_head = True
    out = tr.train_step(batch)
    assert set(out) == {'train/loss', 'train/lr'} and all(isinstance(v, float) for v in out.values())
    assert model.calls == [{'output_hidden_states': True, 'logits_to_keep': 1}]
    assert LM_HEAD_CHAIN <= set(dry.calls), LM_HEAD_CHAIN - set(dry.calls)
    assert dry.calls.index('aa_ce_rows') < dry.calls.index('aa_linear_logprob_fwd')
    assert not {'aa_logprob_ce_fused', 'aa_logprob_fwd', 'aa_logprob_bwd'} & set(dry.calls)
    assert hidden.grad is not None and hidden.grad.shape == hidden.shape
    assert weight.grad is not None and weight.grad.shape == weight.shape


def test_fused_sft_with_no_valid_row_launches_no_lm_head_kernel(dry):
    from align_anything_b200.trainers.text_to_text.sft import SupervisedTrainer

    dry.n_valid = 0
    hidden, weight, batch = _sft_inputs()
    tr = SupervisedTrainer(None, _HiddenModel(hidden, weight))
    tr.fused_lm_head = True
    loss = tr.loss(batch)['loss']
    assert math.isnan(float(loss.detach()))
    loss.backward()
    assert 'aa_ce_rows' in dry.calls and not [c for c in dry.calls if c.startswith('aa_linear_')]
    assert torch.count_nonzero(hidden.grad) == 0 and torch.count_nonzero(weight.grad) == 0


def test_default_sft_path_is_unchanged(dry):
    from align_anything_b200.trainers.text_to_text.sft import SupervisedTrainer

    hidden, weight, batch = _sft_inputs()
    logits = torch.randn(2, 9, 101).bfloat16().requires_grad_(True)
    model = _HiddenModel(hidden, weight, logits=logits)
    assert SupervisedTrainer.fused_lm_head is False and SupervisedTrainer.lm_head_chunk_rows is None
    out = SupervisedTrainer(None, model).train_step(batch)
    assert isinstance(out['train/loss'], float)
    assert model.calls == [{}]
    assert 'aa_logprob_ce_fused' in dry.calls and 'aa_ce_rows' not in dry.calls


def test_forward_without_logits_to_keep_falls_back_to_the_logits_path(dry):
    from align_anything_b200.trainers.text_to_text.sft import SupervisedTrainer

    hidden, weight, batch = _sft_inputs()
    logits = torch.randn(2, 9, 101).bfloat16().requires_grad_(True)
    model = _HiddenModel(hidden, weight, logits=logits, takes_keep=False)
    tr = SupervisedTrainer(None, model)
    tr.fused_lm_head = True
    with pytest.warns(RuntimeWarning, match='logits_to_keep'):
        tr.train_step(batch)
    assert tr.fused_lm_head is False  # switched off for this trainer: later steps go straight to the logits
    assert 'aa_logprob_ce_fused' in dry.calls and logits.grad is not None
    assert not [c for c in dry.calls if c.startswith('aa_linear_')]
    with warnings.catch_warnings():
        warnings.simplefilter('error')
        tr.train_step(batch)


def test_hidden_states_that_do_not_line_up_with_the_labels_fall_back(dry):
    from align_anything_b200.trainers.text_to_text.sft import SupervisedTrainer

    hidden, weight, batch = _sft_inputs()
    spliced = torch.randn(2, 13, 64).bfloat16()  # e.g. image embeddings spliced in inside the forward
    logits = torch.randn(2, 9, 101).bfloat16().requires_grad_(True)
    tr = SupervisedTrainer(None, _HiddenModel(spliced, weight, logits=logits))
    tr.fused_lm_head = True
    with pytest.warns(RuntimeWarning, match='do not line up'):
        tr.train_step(batch)
    assert 'aa_logprob_ce_fused' in dry.calls and logits.grad is not None
    assert not [c for c in dry.calls if c.startswith('aa_linear_')]


@pytest.mark.parametrize('fused', [False, True])
def test_multimodal_ptx_step_dry_run(dry, fused):
    from align_anything_b200.trainers.text_image_to_text.ppo import PPOTrainer

    hidden, weight, batch = _sft_inputs()
    logits = torch.randn(2, 9, 101).bfloat16().requires_grad_(True)
    model = _HiddenModel(hidden, weight, logits=logits)
    t = object.__new__(PPOTrainer)
    t.infer_batch = lambda b: {k: v for k, v in b.items() if k != 'meta_info'}
    t.actor_model, t.ptx_coeff, t.fused_lm_head = model, 16.0, fused
    out = t.ptx_step(batch)
    assert set(out) == {'train/ptx_loss'} and isinstance(out['train/ptx_loss'], float)
    if fused:
        assert model.calls == [{'output_hidden_states': True, 'logits_to_keep': 1}]
        assert LM_HEAD_CHAIN <= set(dry.calls) and 'aa_logprob_ce_fused' not in dry.calls
        assert hidden.grad is not None and weight.grad is not None
    else:
        assert model.calls == [{}] and 'aa_ce_rows' not in dry.calls and logits.grad is not None


def test_text_ppo_trainer_gains_no_switch():
    from align_anything_b200.trainers.text_to_text.ppo import PPOTrainer

    assert not hasattr(PPOTrainer, 'fused_lm_head')


_SFT_MODULES = ('text_to_text', 'text_image_to_text', 'text_audio_to_text')


@pytest.fixture
def sft_reference_tree(monkeypatch):
    """The reference's module paths of the three SFT trainers, with a SupervisedTrainer that has the reference's own
    loss / train_step (stand-ins) and none of the new attributes."""
    names = ['align_anything', 'align_anything.utils', 'align_anything.utils.tools', 'align_anything.trainers']
    for m in _SFT_MODULES:
        names += [f'align_anything.trainers.{m}', f'align_anything.trainers.{m}.sft']
    mods = {}
    for name in names:
        mod = types.ModuleType(name)
        mod.__path__ = []
        mods[name] = mod
        monkeypatch.setitem(sys.modules, name, mod)
    tools = mods['align_anything.utils.tools']
    tools.gather_log_probabilities = tools.masked_mean = tools.move_padding_left = lambda *a, **k: None
    for m in _SFT_MODULES:
        def loss(self, sft_batch):
            raise AssertionError('not grafted')

        cls = type('SupervisedTrainer', (), {'loss': loss, 'train_step': loss})
        mods[f'align_anything.trainers.{m}.sft'].SupervisedTrainer = cls
    return {m: mods[f'align_anything.trainers.{m}.sft'].SupervisedTrainer for m in _SFT_MODULES}


def test_patch_installs_and_restores_the_sft_attributes(sft_reference_tree):
    from align_anything_b200 import patch
    from align_anything_b200.trainers.text_to_text.sft import SupervisedTrainer as Ours

    before = {m: dict(cls.__dict__) for m, cls in sft_reference_tree.items()}
    done = patch.install(models=False)
    try:
        for m, cls in sft_reference_tree.items():
            assert {'SupervisedTrainer.loss', 'SupervisedTrainer.train_step'} <= set(done[f'align_anything.trainers.{m}.sft'])
            assert cls.loss is Ours.loss and cls.train_step is Ours.train_step
            assert cls.fused_lm_head is False and cls.lm_head_chunk_rows is None and cls.ignore_index == -100
    finally:
        patch.uninstall()
    for m, cls in sft_reference_tree.items():
        assert dict(cls.__dict__) == before[m]
        assert not hasattr(cls, 'fused_lm_head') and not hasattr(cls, 'lm_head_chunk_rows')
