"""GPU: every sampled predictor of mpvae on an empty batch returns its usual result type with zero rows, each field's
trailing shape and dtype as for a non-empty batch, and does so without a library launch, a host synchronisation or a
noise offset."""
import pytest
import torch

from oracle import probit_elbo_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

S, L, Z, C = 6, 40, 5, 3
W = (L + 31) // 32
f32, f64, i32 = torch.float32, torch.float64, torch.int32

# name -> (result type name or None for a bare tensor, [(shape, dtype) of each field])
EXPECTED = {
    "predict": (None, [((0, L), f32)]),
    "predict_conditional": ("ConditionalPrediction", [((0, L), f32), ((0,), f32), ((0,), f32)]),
    "predict_conditional_ghk": ("ConditionalPrediction", [((0, L), f32), ((0,), f32), ((0,), f32)]),
    "sample_labels": (None, [((0, S, W), i32)]),
    "predict_sets": ("SetPrediction", [((0, L), torch.bool), ((0,), f64), ((0,), i32)]),
    "score_sets": ("SetScores", [((0, C), f64), ((0, C), f64)]),
    "predict_mode": ("ModePrediction", [((0, L), torch.bool), ((0,), f64), ((0,), f64), ((0,), i32), ((0,), i32)]),
}


def _call(name, fx, r, args):
    from mpvae_b200 import mpvae
    if name in ("predict_conditional", "predict_conditional_ghk"):
        return getattr(mpvae, name)(fx, r, torch.full((0, L), -1, dtype=torch.int8, device=DEV), args)
    if name == "score_sets":
        return mpvae.score_sets(fx, r, torch.zeros(0, C, W, dtype=torch.int32, device=DEV), args)
    return getattr(mpvae, name)(fx, r, args)


@pytest.mark.parametrize("name", sorted(EXPECTED))
def test_empty_batch(name):
    from mpvae_b200 import _lib, mpvae
    fx = torch.empty(0, L, device=DEV)
    r = torch.randn(L, Z, dtype=torch.float64, device=DEV)
    args = orc.make_args(L, Z, n_test_sample=S, mode="test", noise_seed=3)     # no noise_offset: a call would take one
    mpvae.set_noise_seed(11, offset=5)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    torch.cuda.set_sync_debug_mode("error")
    try:
        with torch.no_grad():
            res = _call(name, fx, r, args)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert _lib.launch_count() == n0
    assert mpvae._state["offset"] == 5
    kind, fields = EXPECTED[name]
    if kind is None:
        assert type(res) is torch.Tensor
        res = (res,)
    else:
        assert type(res) is getattr(mpvae, kind)
    assert [(tuple(t.shape), t.dtype) for t in res] == fields
    assert all(t.device == torch.device(DEV) for t in res)
