"""GPU parity: boundary rows -> label maps (octm_labels_from_boundaries) against the oracle, bit-exact."""
import numpy as np
import pytest
import torch

from oracle import labelmap_oracle as lo
from retinal_oct_image_segmentation_via_deep_learning_b200 import suite, synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,h,w,kb", [(3, 60, 48, 4), (2, 496, 512, 7), (2, 33, 50, 3), (1, 17, 7, 15), (2, 40, 1032, 9)]
                         # V = 4 strips (w % 4 == 0) and byte columns at small and ragged widths, 0 to 15 boundaries
                         + [(2, 37, w, kb) for w in (1, 3, 4, 8, 513, 2048) for kb in (0, 1, 15)])
def test_int_boundaries(cuda, n, h, w, kb):
    rng = np.random.default_rng(n * 1000 + w)
    b = rng.integers(-3, h + 4, size=(n, kb, w)).astype(np.int32)           # unsorted, partly outside [0, H]
    got = suite.labels_from_boundaries(torch.from_numpy(b).to(cuda), h).cpu().numpy()
    assert np.array_equal(got, lo.labels_from_boundaries(b, h))


def test_float_boundaries_with_nan(cuda):
    rng = np.random.default_rng(4)
    b = rng.uniform(-2, 70, size=(4, 6, 96)).astype(np.float32)
    b[:, :, ::7] = np.round(b[:, :, ::7])                                  # exact integers: y == b counts
    b[1, 2, 10:30] = np.nan
    b[2, :, 40:44] = np.nan
    got = suite.labels_from_boundaries(torch.from_numpy(b).to(cuda), 64).cpu().numpy()
    assert np.array_equal(got, lo.labels_from_boundaries(b, 64))


def test_round_trip_with_the_label_pass(cuda):
    yt, yp = synth.layered_pair(6, 128, 256, 6, seed=21)
    a, b = torch.from_numpy(yt).to(cuda), torch.from_numpy(yp).to(cuda)
    lp = suite.label_pass(a, b, 6, boundaries=True)
    assert torch.equal(suite.labels_from_boundaries(lp.bnd_true, 128), a)
    assert torch.equal(suite.labels_from_boundaries(lp.bnd_pred.to(torch.float32) - 0.5, 128), b)


def test_zero_boundaries_and_errors(cuda):
    z = suite.labels_from_boundaries(torch.empty((2, 0, 16), dtype=torch.int32, device=cuda), 8)
    assert z.shape == (2, 8, 16) and int(z.sum()) == 0
    with pytest.raises(ValueError):
        suite.labels_from_boundaries(torch.zeros((1, 16, 8), dtype=torch.int32, device=cuda), 8)
    with pytest.raises(TypeError):
        suite.labels_from_boundaries(np.zeros((1, 2, 8), np.int32), 8)
