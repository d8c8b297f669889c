"""The shim directory stands in for the reference's top-level modules, so its unmodified model_trainer.py builds the B200
modules.  What the reference asks of those modules is stored in tests/golden/reference_trainer.json (written by
`oracle/make_golden.py reference_trainer` from the reference itself): the names its files import from them, the
constructor calls `VideoTransformer.__init__` (model_trainer.py:40-104) makes, and the parameter surface of the trainer
built from the reference's own modules.  Here those imports resolve through the shim, the recorded calls build the B200
modules, and a forward + backward runs (kernel table = CPU emulation)."""
import importlib
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, 'videotransformer_pytorch_b200', 'shim')
SHIM_MODULES = ('transformer', 'video_transformer', 'mixup', 'mask_generator')
TRAINER_CFG = dict(objective='supervised', arch='timesformer', pretrain_pth=None, weights_from='imagenet', img_size=32,
                   num_frames=2, attention_type='divided_space_time', num_class=5, eval_metrics='finetune', mixup=False)


@pytest.fixture
def reference_trainer():
    with open(os.path.join(ROOT, 'tests', 'golden', 'reference_trainer.json')) as fh:
        return json.load(fh)


@pytest.fixture
def shim_modules():
    saved_path = list(sys.path)
    saved_mods = {k: sys.modules.pop(k, None) for k in SHIM_MODULES}
    sys.path.insert(0, SHIM)
    try:
        yield {k: importlib.import_module(k) for k in SHIM_MODULES}
    finally:
        sys.path[:] = saved_path
        for k, v in saved_mods.items():
            sys.modules.pop(k, None)
            if v is not None:
                sys.modules[k] = v


def test_reference_trainer_builds_b200_modules_through_the_shim(reference_trainer, shim_modules, emu):
    import videotransformer_pytorch_b200 as pkg
    ref = reference_trainer
    assert ref['cfg'] == TRAINER_CFG
    # every name the reference imports from a shimmed module resolves, and the trainer's five are the package's classes
    for mod, names in ref['imports'].items():
        for name in names:
            assert hasattr(shim_modules[mod], name), (mod, name)
    vt, tr = shim_modules['video_transformer'], shim_modules['transformer']
    assert vt.TimeSformer is pkg.TimeSformer and vt.ViViT is pkg.ViViT and vt.MaskFeat is pkg.MaskFeat
    assert tr.ClassificationHead is pkg.ClassificationHead and shim_modules['mixup'].Mixup is pkg.Mixup
    assert set(ref['imports']['video_transformer']) >= {'TimeSformer', 'ViViT', 'MaskFeat'}
    assert 'ClassificationHead' in ref['imports']['transformer'] and 'Mixup' in ref['imports']['mixup']
    # the constructor calls the reference trainer makes for this configuration, through the shim
    built = {}
    for name, args, kwargs in ref['constructions']:
        built[name] = getattr(vt if hasattr(vt, name) else tr, name)(*args, **kwargs)
    assert sorted(built) == ['ClassificationHead', 'TimeSformer']
    trainer = torch.nn.Module()
    trainer.model, trainer.cls_head = built['TimeSformer'], built['ClassificationHead']
    assert isinstance(trainer.model, pkg.TimeSformer) and isinstance(trainer.cls_head, pkg.ClassificationHead)
    assert sorted(ref['no_weight_decay_keywords']) == sorted(trainer.model.no_weight_decay_keywords())
    # the parameter surface the reference's optimizer grouping walks (optimizer.py:49), name for name and shape for shape
    assert [[n, list(p.shape)] for n, p in trainer.named_parameters()] == ref['named_parameters']
    names = [n for n, _ in trainer.named_parameters()]
    assert 'model.transformer_layers.layers.0.attentions.0.temporal_fc.weight' in names and 'cls_head.cls_head.weight' in names
    # the reference's training_step core (model_trainer.py:204-208) on a tiny clip; embed_dims 768 is fixed by the ctor
    x = torch.randn(2, 2, 3, 32, 32)
    y = torch.tensor([1, 3])
    preds = trainer.cls_head(trainer.model(x))
    loss = torch.nn.CrossEntropyLoss()(preds, y)
    loss.backward()
    assert preds.shape == (2, 5) and torch.isfinite(loss)
    assert all(p.grad is not None for p in trainer.model.parameters())
