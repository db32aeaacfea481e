"""hawkeye_b200.data — the mirror of the reference's dataset package (dataset/dataset.py, transforms.py:14-73, sampler.py) — on a
generated image folder: item format, the deterministic eval preset, class-balanced batches; and item-for-item / batch-for-batch
equality with what the reference's own classes produced on the same folder (tests/golden/make_golden_compat.py)."""
import os

import numpy as np
import pytest
import torch

import detgen
from hawkeye_b200 import data as D


@pytest.fixture(scope='module')
def folder(tmp_path_factory):
    root = str(tmp_path_factory.mktemp('imgs'))
    return root, detgen.image_folder(root)


def test_dataset_items_and_eval_preset(folder):
    root, meta = folder
    ds = D.FGDataset(root, meta, transform=D.ClassificationPresetEval(crop_size=32, resize_size=36), return_id=True)
    assert len(ds) == 24
    it = ds[5]
    assert set(it) == {'img', 'label', 'id'} and it['id'] == 5 and int(it['label']) == 1
    assert it['img'].shape == (3, 32, 32) and it['img'].dtype == torch.float32
    assert torch.equal(ds[5]['img'], it['img'])                               # deterministic
    tr = D.FGDataset(root, meta, transform=D.ClassificationPresetTrain(crop_size=32, auto_augment_policy='ta_wide',
                                                                      random_erase_prob=0.1))
    assert tr[0]['img'].shape == (3, 32, 32)


def test_balanced_batches(folder):
    root, meta = folder
    ds = D.FGDataset(root, meta)
    np.random.seed(3)
    s = D.BalancedBatchSampler(ds, n_classes=2, n_samples=3)
    batches = list(s)
    assert len(s) == 4 and 1 <= len(batches) <= 4
    labels = np.array(ds.images['label'])
    for b in batches:
        assert len(b) == 6
        cls, cnt = np.unique(labels[b], return_counts=True)
        assert len(cls) == 2 and (cnt == 3).all()                               # what MAMCLoss needs


def test_matches_reference_classes(folder):
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_compat.npz'))
    root, meta = folder
    ours = D.FGDataset(root, meta, transform=D.ClassificationPresetEval(crop_size=32, resize_size=36))
    assert len(ours) == int(G['data_len'])
    for j, i in enumerate((0, 7, 23)):
        a = ours[i]
        assert int(a['label']) == int(G['data_eval_labels'][j])
        assert torch.equal(a['img'], torch.from_numpy(G['data_eval_imgs'][j]))
    # train preset: same transform pipeline => same draws from the same torch / python RNG state
    import random
    to = D.ClassificationPresetTrain(32, auto_augment_policy='ta_wide', random_erase_prob=0.1)
    img = D.default_loader(os.path.join(root, 'c1/img_5.png'))
    torch.manual_seed(11); random.seed(11)
    x = to(img)
    assert torch.equal(x, torch.from_numpy(G['data_train_img']))
    # sampler: same numpy call order => same batches
    np.random.seed(5)
    b1 = [list(map(int, b)) for b in D.BalancedBatchSampler(ours, 2, 3)]
    assert b1 == G['data_sampler_batches'].tolist() and len(b1) > 0
