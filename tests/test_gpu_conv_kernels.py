"""Kernel-level GPU tests: the CUDA-core (backend 0) and tensor-core (tcgen05, conv_mma2.cu; 1 = bf16x3, 2 = tf32x3 with
2 K-chains, 5 = fp16x3 with 1 chain, 6 = fp16x3 with 2 chains) Conv1d kernels against a float64 torch reference of the
same op.  (Backends 3 and 4 are the same kernels as 1 and 2.)"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _ref(x, w, b, dil, slope, resid):
    import torch
    import torch.nn.functional as F
    xt = torch.from_numpy(x).double()
    if slope:
        xt = F.leaky_relu(xt, slope)
    y = F.conv1d(xt, torch.from_numpy(w).double(), None if b is None else torch.from_numpy(b).double(),
                 dilation=dil, padding=dil * (w.shape[2] - 1) // 2)
    if resid is not None:
        y = y + torch.from_numpy(resid).double()
    return y.numpy()


CASES = [  # (B, ci, co, k, dil, L)   every generator resblock shape of the medium / high presets + odd lengths
    (2, 32, 32, 3, 1, 300), (1, 32, 32, 7, 12, 1000), (2, 64, 64, 5, 6, 517), (1, 64, 64, 11, 5, 400),
    (1, 128, 128, 7, 3, 260), (1, 128, 128, 3, 2, 129), (1, 256, 256, 3, 1, 200), (1, 256, 256, 11, 1, 140),
    (3, 32, 32, 5, 2, 7),
    # flow / text-encoder shapes (output rows tiled across CTAs when > 256), ragged tile ends
    (2, 192, 384, 5, 1, 519), (1, 192, 768, 3, 1, 259), (1, 768, 192, 3, 1, 259), (2, 96, 192, 1, 1, 600),
    (1, 192, 96, 1, 1, 333), (1, 48, 96, 1, 1, 150), (1, 192, 576, 1, 1, 259), (1, 96, 48, 1, 1, 257),
    (1, 192, 256, 7, 1, 519),
    # enough tiles for every SM to walk several tiles of the persistent tensor-core kernel
    (4, 32, 32, 7, 12, 40000), (2, 64, 64, 5, 6, 45001), (2, 128, 128, 7, 3, 20003), (2, 192, 384, 5, 1, 6001),
    (1, 192, 768, 3, 1, 5000), (2, 256, 256, 3, 1, 9999),
]


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("backend", [0, 1, 2, 5, 6])
def test_conv1d_kernels(lib_built, backend, case):
    from piper_b200 import engine
    B, ci, co, k, dil, L = case
    rng = np.random.default_rng(hash(case) % (2 ** 31))
    x = rng.standard_normal((B, ci, L)).astype(np.float32) * 2
    w = (rng.standard_normal((co, ci, k)) / np.sqrt(ci * k)).astype(np.float32)
    b = rng.standard_normal(co).astype(np.float32)
    resid = rng.standard_normal((B, co, L)).astype(np.float32)
    ref = _ref(x, w, b, dil, 0.1, resid)
    y = engine.debug_conv1d(backend, x, w, b, dil, 0.1, resid)
    err = np.abs(y - ref).max()
    # fp32 FFMA / tf32x3 / fp16x3: accumulation-order noise; bf16x3: ~2^-16 relative per product on O(1) outputs
    tol = 3e-4 if backend else 1e-4      # tensor-core fp32 accumulation truncates (RZ): error grows ~linearly with K
    assert err <= tol, err
    y2 = engine.debug_conv1d(backend, x, w, None, dil, 0.0, None)
    assert np.abs(y2 - _ref(x, w, None, dil, 0.0, None)).max() <= tol
