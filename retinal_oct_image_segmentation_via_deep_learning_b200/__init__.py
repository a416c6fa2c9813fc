"""B200-native evaluation-metric suite for retinal OCT segmentation label maps.

Drop-in (same module and function names) for ``Metrics/`` of
ZhangHH233/Retinal_OCT_Image_Segmentation_via_Deep_Learning, plus batched device-resident entry
points.  All label arithmetic runs in hand-written sm_100a kernels (``liboctm.so``, C ABI in
``include/octm.h``); there is no CPU fallback.

    from retinal_oct_image_segmentation_via_deep_learning_b200 import evaluate
    res = evaluate(y_true_cuda_u8, y_pred_cuda_u8, num_classes=8)
    res.metrics()["dice_coefficient"]        # float64 [N, K]

    # reference-style: put the drop-in directory on sys.path, exactly like the reference's Metrics/
    import sys; sys.path.insert(0, METRICS_DIR)
    import Region_based_metrics as R; R.dice_coefficient(mask_true, mask_pred)
"""
import os as _os

METRICS_DIR = _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "Metrics")

_LAZY = {"evaluate", "label_pass", "contour_pass", "confusion", "boundary_error", "validate_labels", "SuiteResult",
         "surface_dice", "components"}


def __getattr__(name):          # keep `import package.synth` free of torch / the CUDA library
    if name in _LAZY:
        from . import suite
        return getattr(suite, name)
    raise AttributeError(name)
