"""Golden fixtures for checkpoint and dataset compatibility with the UNMODIFIED reference.
Run where the reference tree is importable:  python tests/golden/make_golden_compat.py  -> tests/golden/reference_compat.npz

  <name>_state_json   the reference model's state_dict layout, in order: [[key, shape, dtype], ...] (BCNN stage 2, MPN);
                      a .pth file written by the reference holds exactly these tensors (train.py:375)
  data_*              dataset/dataset.FGDataset, dataset/transforms and dataset/sampler on detgen.image_folder(): eval-preset
                      items 0, 7, 23; the train preset on c1/img_5.png after torch / python seeds 11; BalancedBatchSampler(2, 3)
                      batches after numpy seed 5"""
import importlib
import json
import os
import random
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, 'tests'))
from oracle import ref_harness as rh  # noqa: E402
import detgen  # noqa: E402

CHECKPOINT_MODELS = {'BCNN': dict(stage=2, num_classes=200),
                     'MPN': dict(iter_num=5, is_sqrt=True, is_vec=True, input_dim=2048, dimension_reduction=256,
                                 num_classes=200)}
DATA_ITEMS = (0, 7, 23)


def _json_bytes(obj):
    return np.frombuffer(json.dumps(obj).encode(), dtype=np.uint8)


def main():
    rh.load_reference()
    from model.registry import MODEL
    out = {}
    for name, kw in CHECKPOINT_MODELS.items():
        sd = MODEL.get(name)(rh.cfg(name=name, **kw)).state_dict()
        out[f'{name}_state_json'] = _json_bytes([[k, list(v.shape), str(v.dtype)] for k, v in sd.items()])

    root = rh.find_reference_root()
    if root not in sys.path:
        sys.path.insert(0, root)
    rd, rt, rs = (importlib.import_module(m) for m in ('dataset.dataset', 'dataset.transforms', 'dataset.sampler'))
    with tempfile.TemporaryDirectory() as folder:
        meta = detgen.image_folder(folder)
        ref = rd.FGDataset(folder, meta, transform=rt.ClassificationPresetEval(crop_size=32, resize_size=36))
        out['data_len'] = np.int64(len(ref))
        out['data_eval_labels'] = np.array([int(ref[i]['label']) for i in DATA_ITEMS], dtype=np.int64)
        out['data_eval_imgs'] = np.stack([ref[i]['img'].numpy() for i in DATA_ITEMS])
        tr = rt.ClassificationPresetTrain(32, auto_augment_policy='ta_wide', random_erase_prob=0.1)
        img = rd.default_loader(os.path.join(folder, 'c1/img_5.png'))
        torch.manual_seed(11)
        random.seed(11)
        out['data_train_img'] = tr(img).numpy()
        np.random.seed(5)
        out['data_sampler_batches'] = np.array([list(map(int, b)) for b in rs.BalancedBatchSampler(ref, 2, 3)],
                                               dtype=np.int64)
    path = os.path.join(HERE, 'reference_compat.npz')
    np.savez_compressed(path, **out)
    print('wrote', len(out), 'arrays;', os.path.getsize(path) / 1e6, 'MB')


if __name__ == '__main__':
    main()
