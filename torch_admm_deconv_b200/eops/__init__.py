from .deconv import (fft_admm_tv, fft_admm_tv_f64, soft_thresh, block_thresh, pixelnorm, hard_thresh, torch_abs2, identity,
                     conv_circular)

__all__ = ["fft_admm_tv", "fft_admm_tv_f64", "soft_thresh", "block_thresh", "pixelnorm", "hard_thresh", "torch_abs2", "identity",
           "conv_circular"]
