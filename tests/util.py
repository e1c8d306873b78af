"""Shared helpers for the parity tests."""
import os
import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
_cache = {}


def golden(name):
    """The arrays of one fixture; a fixture over 1 MB is stored in parts name.npz, name.1.npz, ... (make_golden.save)."""
    if name not in _cache:
        d, path, i = {}, os.path.join(GOLDEN, name + '.npz'), 0
        while True:
            with np.load(path) as z:
                d.update({k: z[k] for k in z.files})
            i += 1
            path = os.path.join(GOLDEN, '%s.%d.npz' % (name, i))
            if not os.path.exists(path):
                break
        _cache[name] = d
    return _cache[name]


def T(a, device='cpu'):
    return torch.from_numpy(np.asarray(a)).to(device)


def rel_err(a, b):
    """max |a-b| / max(|b|_inf, tiny): the '1e-4 relative in fp32' bar of BASELINE.json is read as
    error relative to the tensor's scale (per-element relative error is meaningless at zero crossings)."""
    a = torch.as_tensor(a, dtype=torch.float64).cpu()
    b = torch.as_tensor(b, dtype=torch.float64).cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(b.abs().max().item(), 1e-30)
    return (a - b).abs().max().item() / scale


def assert_close(a, b, tol=1e-4, what=''):
    e = rel_err(a, b)
    assert e <= tol, f'{what}: rel err {e:.3e} > {tol:.1e}'


def key_with_stride(d, prefix):
    """Golden grads of big tensors are stored as flat[::stride] under 'name@stride'."""
    for k in d:
        if k == prefix:
            return k, None
        if k.startswith(prefix + '@'):
            return k, int(k.split('@')[1])
    raise KeyError(prefix)


def pick(g, stride):
    return g if stride is None else g.flatten()[::stride]


def assert_close_robust(a, b, tol=1e-4, max_outlier_frac=2e-4, what=''):
    """Full-size variant: the gradient of a bilinear sample is discontinuous where a coordinate lands on
    an integer pixel, so 1-ulp coordinate differences flip a handful of pixels' gradients - the oracle
    run on CPU and on GPU disagree with EACH OTHER at ~1e-4 of the level-0 pixels (gpurun diag_masks
    log, profiles/r01_parity_notes.md).  Require <= tol everywhere except a vanishing fraction."""
    a = torch.as_tensor(a, dtype=torch.float64).cpu()
    b = torch.as_tensor(b, dtype=torch.float64).cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    scale = max(b.abs().max().item(), 1e-30)
    err = (a - b).abs() / scale
    n_bad = int((err > tol).sum().item())
    allowed = max(2, int(max_outlier_frac * err.numel()))
    assert n_bad <= allowed, f'{what}: {n_bad} of {err.numel()} elements exceed {tol:.1e} (max {err.max().item():.2e}), allowed {allowed}'
