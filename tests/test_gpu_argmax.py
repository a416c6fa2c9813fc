"""GPU parity: scores -> label map (argmax front end) against numpy argmax, bit-exact."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _ref(scores, axis):
    # numpy argmax: first maximal element, NaN counts as maximal
    return np.argmax(scores.astype(np.float32), axis=axis).astype(np.uint8)


def _labels_and_kernel(scores, **kw):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import _lib, suite
    with _lib.kernel_profile() as prof:
        got = suite.labels_from_scores(scores, **kw)
        torch.cuda.synchronize()
    assert len(prof.kernels) == 1, prof.kernels
    return got.cpu().numpy(), next(iter(prof.kernels))


@pytest.mark.parametrize("dtype", ["float32", "float16", "bfloat16"])
@pytest.mark.parametrize("shape", [(3, 8, 32, 64), (2, 11, 17, 23), (1, 4, 496, 512), (5, 1, 8, 8), (2, 200, 6, 10),
                                   # K not a multiple of the planes kernel's 4-plane batch, and K = 256, on planes
                                   (2, 3, 16, 32), (2, 5, 8, 48), (1, 7, 16, 16), (2, 9, 32, 32), (1, 13, 8, 64),
                                   (1, 256, 16, 16)])
def test_argmax_planes_and_generic(cuda, dtype, shape):
    """Class-major scores take the planes kernel when the plane holds whole 32-byte vectors (8 float32 or 16 16-bit
    scores; fresh tensors are aligned), the generic kernel otherwise; channels-last scores always take the generic one."""
    import torch
    g = torch.Generator().manual_seed(hash((dtype, shape)) % 2**31)
    x = torch.randn(shape, generator=g)
    x = (x * 4).round() / 4                       # many exact ties, also after rounding to 16 bits
    x = x.to(getattr(torch, dtype))
    vpt = 8 if dtype == "float32" else 16
    got, kern = _labels_and_kernel(x.to(cuda))
    assert kern == ("argmax_planes_kernel" if shape[2] * shape[3] % vpt == 0 else "argmax_generic_kernel")
    ref = _ref(x.float().numpy(), 1)
    np.testing.assert_array_equal(got, ref)
    xl = x.permute(0, 2, 3, 1).contiguous()
    got, kern = _labels_and_kernel(xl.to(cuda), channels_last=True)
    assert kern == "argmax_generic_kernel"
    np.testing.assert_array_equal(got, ref)


def test_argmax_nan_and_inf(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite
    x = torch.zeros((1, 5, 4, 8))
    x[0, 3, 0, 0] = float("nan")
    x[0, 1, 0, 1] = float("inf")
    x[0, :, 0, 2] = float("-inf")
    x[0, 2, 0, 3] = float("nan"); x[0, 4, 0, 3] = float("nan")
    x[0, 4, 1, :] = 1e-30
    got = suite.labels_from_scores(x.to(cuda)).cpu().numpy()
    np.testing.assert_array_equal(got, _ref(x.numpy(), 1))
    assert got[0, 0, 0] == 3 and got[0, 0, 1] == 1 and got[0, 0, 2] == 0 and got[0, 0, 3] == 2


def test_evaluate_scores_matches_evaluate_on_labels(cuda):
    import torch
    from retinal_oct_image_segmentation_via_deep_learning_b200 import suite, synth
    yt, yp = synth.layered_pair(2, 64, 128, 6, seed=9, noise=0.01)
    onehot = np.eye(6, dtype=np.float32)[yp].transpose(0, 3, 1, 2) * 3.0 - 1.0       # scores whose argmax is yp
    a = suite.evaluate(torch.from_numpy(yt).to(cuda), torch.from_numpy(yp).to(cuda), 6).integers()
    b = suite.evaluate_scores(torch.from_numpy(yt).to(cuda), torch.from_numpy(np.ascontiguousarray(onehot)).to(cuda)).integers()
    for key in a:
        np.testing.assert_array_equal(a[key], b[key], err_msg=key)
