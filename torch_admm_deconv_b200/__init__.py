"""B200-native drop-in for the ADMM-TV deconvolution path of georgegrosu1/torch-admm-deconv.

    reference                                    this package
    admmtor.eops.deconv.fft_admm_tv         ->   torch_admm_deconv_b200.eops.deconv.fft_admm_tv
    admmtor.elayers.admmdeconv.ADMMDeconv   ->   torch_admm_deconv_b200.elayers.admmdeconv.ADMMDeconv
    admmtor.modelbuild.blocks.MultiADMM, admmtor.modelbuild.deconver.Deconvs, admmtor.elayers.admmfusion.ADMMFusion
                                            ->   torch_admm_deconv_b200.elayers.multiadmm.{MultiADMM, Deconvs, ADMMFusion}
    a whole reference model (DivergentRestorer ...)  ->  torch_admm_deconv_b200.use_b200_admm(model)

The arithmetic runs in hand-written sm_100a CUDA kernels reached through the C ABI of
include/admm_b200.h; there is no CPU or PyTorch fallback.
"""
from .eops.deconv import fft_admm_tv, fft_admm_tv_f64, identity, soft_thresh, block_thresh, pixelnorm, hard_thresh, torch_abs2
from .elayers.admmdeconv import ADMMDeconv
from .elayers.multiadmm import MultiADMM, Deconvs, ADMMFusion
from .dropin import use_b200_admm

__all__ = ["fft_admm_tv", "fft_admm_tv_f64", "ADMMDeconv", "MultiADMM", "Deconvs", "ADMMFusion", "use_b200_admm", "identity", "soft_thresh", "block_thresh", "pixelnorm", "hard_thresh",
           "torch_abs2"]
__version__ = "0.2.0"
