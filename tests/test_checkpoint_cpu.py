"""Checkpoint wire format (SURVEY 8(f) N4; reference train.py:369-395, test.py:64-76): a .pth written by the UNMODIFIED
reference loads into the native classes key for key, and one written by hawkeye_b200.Trainer.save_model's code path loads into the
reference.  The reference's state_dict layout (keys in order, shapes, dtypes) is stored in tests/golden/reference_compat.npz by
tests/golden/make_golden_compat.py; a reference file is that layout filled with seeded values."""
import json
import os
import sys

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
G = np.load(os.path.join(REPO, 'tests', 'golden', 'reference_compat.npz'))


class Cfg(dict):
    __getattr__ = dict.__getitem__


def _reference_state(name, seed=1):
    """A state_dict with the reference model's layout: what the reference's torch.save(model.state_dict()) writes."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k, shape, dtype in json.loads(G[f'{name}_state_json'].tobytes()):
        dt = getattr(torch, dtype.split('.')[1])
        out[k] = torch.randn(shape, generator=g).to(dt) if dt.is_floating_point else torch.randint(0, 100, shape, generator=g, dtype=dt)
    return out


@pytest.mark.parametrize('name,kw', [('BCNN', dict(stage=2, num_classes=200)),
                                     ('MPN', dict(iter_num=5, is_sqrt=True, is_vec=True, input_dim=2048,
                                                  dimension_reduction=256, num_classes=200))])
def test_reference_checkpoint_round_trip(name, kw, tmp_path, monkeypatch):
    monkeypatch.setenv('HAWKEYE_ALLOW_RANDOM_INIT', '1')
    import hawkeye_b200 as hb
    from hawkeye_b200.utils import load_state_dict
    a = _reference_state(name)
    path = str(tmp_path / f'{name}_epoch_1.pth')
    torch.save(a, path)                                                       # exactly train.py:375
    ours = hb.MODEL.get(name)(Cfg(name=name, **kw))
    load_state_dict(ours, torch.load(path, map_location='cpu'))               # hawkeye_b200.test.Tester.get_model
    b = ours.state_dict()
    assert list(a.keys()) == list(b.keys())
    assert all(torch.equal(a[k], b[k]) for k in a)
    # DataParallel-prefixed files (the reference saves self.model.state_dict() of the wrapped module, train.py:375)
    torch.save({'module.' + k: v for k, v in a.items()}, path)
    ours2 = hb.MODEL.get(name)(Cfg(name=name, **kw))
    load_state_dict(ours2, torch.load(path, map_location='cpu'))
    assert all(torch.equal(a[k], ours2.state_dict()[k]) for k in a)
    # and back: our file carries exactly the tensors a strict load into the reference (test.py:74-75) requires
    torch.save({k: v.detach().cpu().clone() for k, v in ours.state_dict().items()}, path)     # Trainer.save_model
    c = torch.load(path, map_location='cpu')
    assert list(c.keys()) == list(a.keys())
    assert all(c[k].shape == a[k].shape and c[k].dtype == a[k].dtype and torch.equal(c[k], a[k]) for k in a)
