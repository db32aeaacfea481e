"""Deterministic tensors shared by the golden-fixture generator and the tests.

numpy's legacy RandomState stream is stable across numpy versions, so the GPU box can
regenerate bit-identical inputs/weights without the fixture having to carry them.
"""
import numpy as np
import torch


def det(shape, seed, scale=1.0, positive=False):
    rs = np.random.RandomState(seed)
    a = rs.standard_normal(size=tuple(shape)).astype(np.float32)
    if positive:
        a = np.abs(a)
    return torch.from_numpy(a * np.float32(scale))


def det_uniform(shape, seed):
    rs = np.random.RandomState(seed)
    return torch.from_numpy(rs.random_sample(size=tuple(shape)).astype(np.float32))


def tf32_rna(t):
    """Round an fp32 tensor to the nearest TF32-representable value (ties away from zero, like cvt.rna.tf32.f32)."""
    u = t.contiguous().view(torch.int32)
    r = ((u + 0x1000) & ~0x1FFF)          # add half an ulp of the 13 dropped bits to the magnitude bits, then truncate
    return r.view(torch.float32)


def det_labels(n, num_classes, seed):
    return torch.from_numpy(np.random.RandomState(seed).randint(0, num_classes, size=n).astype(np.int64))


def vgg_bcnn_state(cfg, num_classes, seed=100, feat_dim=None, head_in=None):
    """state_dict-shaped weights for a VGG-'D'-style backbone + Linear head, kaiming-like scales."""
    state, idx, cin = {}, 0, 3
    for v in cfg:
        if v == 'M':
            idx += 1
            continue
        state[f'backbone.{idx}.weight'] = det((v, cin, 3, 3), seed + idx, (2.0 / (v * 9)) ** 0.5)
        state[f'backbone.{idx}.bias'] = det((v,), seed + 1000 + idx, 0.01)
        cin = v
        idx += 2
    head_in = head_in if head_in is not None else cin * cin
    state['classifier.weight'] = det((num_classes, head_in), seed + 5000, (2.0 / head_in) ** 0.5)
    state['classifier.bias'] = det((num_classes,), seed + 5001, 0.01)
    return state


def state_like(module, seed=7):
    """Deterministic state_dict for ANY module (same keys/shapes => same values): per-key seed = crc32(key).
    conv/linear weights ~ kaiming-scaled normals, BN weight ~ 1 + 0.1 n, biases ~ 0.1 n, running stats untouched."""
    import zlib
    out = {}
    for k, v in module.state_dict().items():
        ks = seed + (zlib.crc32(k.encode()) & 0x7fffffff)
        if k.endswith('num_batches_tracked') or k.endswith('running_mean') or k.endswith('running_var'):
            out[k] = v.clone()
        elif v.dim() >= 2:
            fan = v[0].numel()
            out[k] = det(v.shape, ks, (2.0 / fan) ** 0.5)
        elif k.endswith('weight'):
            out[k] = 1.0 + det(v.shape, ks, 0.1)
        else:
            out[k] = det(v.shape, ks, 0.1)
    return out


def image_folder(root):
    """24 random RGB PNGs of growing size in 4 class folders under ``root`` plus the ``<label> <path>`` list the dataset
    reads; returns the list's path."""
    import os
    from PIL import Image
    rng = np.random.RandomState(0)
    lines = []
    for i in range(24):
        arr = rng.randint(0, 256, size=(40 + i, 50 + 2 * i, 3), dtype=np.uint8)
        name = f'c{i % 4}/img_{i}.png'
        os.makedirs(os.path.join(root, f'c{i % 4}'), exist_ok=True)
        Image.fromarray(arr).save(os.path.join(root, name))
        lines.append(f'{i % 4} {name}')
    meta = os.path.join(root, 'train.txt')
    open(meta, 'w').write('\n'.join(lines) + '\n')
    return meta
