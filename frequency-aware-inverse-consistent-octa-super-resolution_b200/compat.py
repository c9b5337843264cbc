"""Make the reference's import names resolve to this package.

    import b200wave.compat; b200wave.compat.install()
    from pytorch_wavelets import DWTForward, DWTInverse      # -> b200wave.DWTForward / DWTInverse
    import pytorch_wavelets.dwt.lowlevel as lowlevel          # -> b200wave.dwt.lowlevel
    import ssim; ssim.SSIM()                                  # -> b200wave.ssim

so that ``model.py`` (``from pytorch_wavelets import DWTForward, DWTInverse``, model.py:4) and ``train.py``
(``import ssim``-style use at train.py:97) of the reference run unmodified on the CUDA path.  The 2-D and 1-D DWT
surfaces are provided (SWT / DTCWT / scattering are out of scope, SURVEY.md section 2); asking for anything else
raises AttributeError instead of silently falling back.
"""
import importlib
import sys
import types


def install(force=False):
    import b200wave
    from b200wave.dwt import lowlevel, transform1d, transform2d
    ssim_mod = importlib.import_module("b200wave.ssim")

    if not force:
        for name in ("pytorch_wavelets", "ssim"):
            mod = sys.modules.get(name)
            if mod is not None and not getattr(mod, "__b200wave_alias__", False):
                raise RuntimeError("module %r is already imported from %s; call install(force=True) to shadow it"
                                   % (name, getattr(mod, "__file__", "?")))

    pw = types.ModuleType("pytorch_wavelets")
    pw.__b200wave_alias__ = True
    pw.__version__ = "1.3.0+b200wave." + b200wave.__version__
    pw.__path__ = []
    for name in ("DWTForward", "DWTInverse", "DWT", "IDWT", "DWT2D", "IDWT2D", "DWT1DForward", "DWT1DInverse", "DWT1D",
                 "IDWT1D", "SWTForward"):
        setattr(pw, name, getattr(b200wave, name))
    dwt = types.ModuleType("pytorch_wavelets.dwt")
    dwt.__b200wave_alias__ = True
    dwt.__path__ = []
    dwt.lowlevel = lowlevel
    dwt.transform2d = transform2d
    dwt.transform1d = transform1d
    pw.dwt = dwt
    sys.modules["pytorch_wavelets"] = pw
    sys.modules["pytorch_wavelets.dwt"] = dwt
    sys.modules["pytorch_wavelets.dwt.lowlevel"] = lowlevel
    sys.modules["pytorch_wavelets.dwt.transform2d"] = transform2d
    sys.modules["pytorch_wavelets.dwt.transform1d"] = transform1d
    ssim_mod.__b200wave_alias__ = True
    sys.modules["ssim"] = ssim_mod
    return pw


def patch_utils(utils_module):
    """Point ``utils.high_pass`` / ``utils.low_pass`` of an already imported reference ``utils`` module
    (``utils.py:93-117``; called at ``train.py:173-213``) at the batched CUDA implementation in ``b200wave.freq``.
    Everything else in that module is left alone."""
    from b200wave import freq
    utils_module.high_pass = freq.high_pass
    utils_module.low_pass = freq.low_pass
    return utils_module


def patch_model(model_module):
    """Swap ``FS_DiscriminatorA.filter_wavelet`` / ``FS_DiscriminatorB.filter_wavelet`` of an already imported
    reference ``model`` module (``model.py:166-179, 222-235``) for the fused analysis-kernel epilogue in
    ``b200wave.fsd``.  The methods keep reading ``self.DWT2`` (its tap buffers and mode) and ``self.cs``, so the
    discriminators' constructors, state dicts and ``forward`` are untouched.  ``model.TVLoss`` and
    ``model.phase_consistency_loss`` (``model.py:17-58``) are replaced by the fused versions in ``b200wave.losses``."""
    from b200wave import fsd

    def make(variant):
        def filter_wavelet(self, x, norm=True):
            d = self.DWT2
            taps = fsd.module_taps(x, (d.h0_col, d.h1_col, d.h0_row, d.h1_row))
            return fsd.filter_wavelet(x, self.cs, norm, variant, taps, d.mode)
        return filter_wavelet

    model_module.FS_DiscriminatorA.filter_wavelet = make("A")
    model_module.FS_DiscriminatorB.filter_wavelet = make("B")
    # the reduction-style losses beside the path (model.py:17-58, constructed at train.py:94,98)
    from b200wave import losses
    model_module.TVLoss = losses.TVLoss
    model_module.phase_consistency_loss = losses.phase_consistency_loss
    return model_module
