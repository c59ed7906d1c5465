"""passiveradar_b200 -- B200-native (sm_100a) core for the passive-radar hot path.

Drop-in operators with the reference's call signatures (Max-Manning/passiveRadar):

    from passiveradar_b200 import fast_xambg, LS_Filter, NLMS_filter, block_NLMS

and a device-resident frame pipeline for streams of CPI frames
(``passiveradar_b200.frames.FramePipeline``).  All arithmetic runs in
``libprcore.so`` (hand-written CUDA, C ABI in ``include/prcore.h``); importing
this package never imports the CPU oracle and never falls back to the CPU.
"""
from .range_doppler_processing import fast_xambg, direct_xambg            # noqa: F401
from .clutter_removal import (LS_Filter, NLMS_filter, block_NLMS,            # noqa: F401
                              LS_Filter_Toeplitz, LS_Filter_Multiple)
from .signal_utils import deinterleave_IQ, frequency_shift, resample, frontend            # noqa: F401
from .signal_utils import xcorr, find_channel_offset, offset_compensation            # noqa: F401
from .target_detection import CFAR_2D            # noqa: F401

__all__ = ["fast_xambg", "direct_xambg", "LS_Filter", "NLMS_filter", "block_NLMS", "LS_Filter_Toeplitz",
           "LS_Filter_Multiple", "deinterleave_IQ", "frequency_shift", "resample", "frontend", "CFAR_2D",
           "xcorr", "find_channel_offset", "offset_compensation"]
__version__ = "0.1.0"


def install(reference_package: str = "passiveRadar"):
    """Swap the hot-path functions of an importable copy of the reference for the GPU ones.

    ``main.py`` binds ``find_channel_offset``, ``fast_xambg``, ``LS_Filter_Multiple`` and ``NLMS_filter`` with
    ``from passiveRadar... import ...`` (main.py:10-14); calling ``install()`` before ``main.py`` is
    imported/run makes those names resolve to this package while config, I/O and the dask graph stay
    the reference's own code::

        python -c "import passiveradar_b200 as p, runpy; p.install(); runpy.run_path('main.py', run_name='__main__')" --config PRconfig.yaml

    Returns the list of ``module.attribute`` names that were replaced.
    """
    import importlib
    replaced = []
    table = {
        "range_doppler_processing": {"fast_xambg": fast_xambg, "direct_xambg": direct_xambg},
        "signal_utils": {"deinterleave_IQ": deinterleave_IQ, "frequency_shift": frequency_shift, "resample": resample,
                         "find_channel_offset": find_channel_offset, "offset_compensation": offset_compensation},
        "target_detection": {"CFAR_2D": CFAR_2D},
        "clutter_removal": {"LS_Filter": LS_Filter, "NLMS_filter": NLMS_filter,
                            "LS_Filter_Toeplitz": LS_Filter_Toeplitz, "LS_Filter_Multiple": LS_Filter_Multiple},
    }
    for modname, attrs in table.items():
        try:
            mod = importlib.import_module(f"{reference_package}.{modname}")
        except Exception:          # e.g. the reference's target_detection needs np.float (NumPy < 1.24)
            if modname in ("range_doppler_processing", "clutter_removal"):
                raise
            continue
        for name, fn in attrs.items():
            setattr(mod, name, fn)
            replaced.append(f"{reference_package}.{modname}.{name}")
        if modname == "clutter_removal" and not hasattr(mod, "block_NLMS"):
            mod.block_NLMS = block_NLMS
            replaced.append(f"{reference_package}.{modname}.block_NLMS")
    return replaced
