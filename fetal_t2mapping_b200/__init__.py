"""fetal_t2mapping_b200: the per-voxel T2 relaxation fit of fetal_t2mapping on B200 (sm_100a).

Only the hot path lives here (SURVEY.md section 8): ``fit_voxel`` driven over the masked voxels
plus ``compute_residuals`` (run_t2mapping.py:120-312, :411-461; utils/t2map_utils.py:62-89),
behind the C ABI of ``include/t2fit.h`` (``csrc/libt2fit.so``, hand-written CUDA).  Everything
else of the reference (DICOM->BIDS, registration, segmentation, NIfTI I/O, plots) stays in the
reference.  There is no CPU implementation of the fit in this package.
"""
from .presets import preset, set_fit_params                                           # noqa: F401
from .api import (BootstrapMaps, BootstrapResult, FitResult, compute_residuals,      # noqa: F401
                  device_info, fit_voxels_batch, init, mask_indices_device, parameter_stderr, parametric_bootstrap,
                  pinned_array, shutdown, t2_interval, t2map_volume, work_model)

from .roi import phantom_roi_table, roi_stats, save_phantom_csv, set_phantom_gt        # noqa: F401
from .loader import VolumeMaps, t2map_series                                          # noqa: F401

__version__ = "0.2.0"
