"""ganspace_b200 -- B200-native activation-sampling + incremental-PCA hot path of GANSpace.

Drop-in surfaces (same names, arguments and error behaviour as the reference's modules):
    ganspace_b200.config.Config
    ganspace_b200.estimators.get_estimator / IPCAEstimator
    ganspace_b200.models.get_model / get_instrumented_model / BaseModel / StyleGAN / StyleGAN2 / BigGAN
    ganspace_b200.decomposition.get_or_compute / get_random_dirs / SEED_*
Compute runs only through the C-ABI CUDA library (include/ganspace_b200.h); there is no CPU fallback.
"""
__version__ = "0.1.0"
