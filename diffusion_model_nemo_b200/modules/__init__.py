"""Export surface of the sampling hot path: the class / function names a Hydra `_target_: diffusion_model_nemo.modules.X` refers to
resolve here as `_target_: diffusion_model_nemo_b200.modules.X` (SURVEY.md section 8b).  The table below is the whole public API,
grouped by the submodule that implements it."""
import importlib

_API = {
    "unet": ("Unet", "WaveGradUNet"),
    "diffusion_process": (
        "AbstractDiffusionProcess", "LinearSchedule", "QuadraticSchedule", "SigmoidSchedule", "CosineSchedule",
        "linear_beta_schedule", "quadratic_beta_schedule", "sigmoid_beta_schedule", "cosine_beta_schedule",
    ),
    "gaussian_diffusion": ("GaussianDiffusion",),
    "learned_gaussian_diffusion": ("LearnedGaussianDiffusion",),
    "generalized_gaussian_diffusion": ("GeneralizedGaussianDiffusion",),
    "dpm_solver_diffusion": ("DPMSolverDiffusion",),
    "wavegrad_diffusion": ("WaveGradDiffusion",),
    "sde": (
        "SDE", "VPSDE", "VESDE", "PredictorCorrectorSampler", "ProbabilityFlowSampler", "DPMSolverSampler", "LikelihoodEstimate", "resolve_score_function",
        "Predictor", "NonePredictor", "EulerMaruyamaPredictor", "AncestralSamplingPredictor", "ReverseDiffusionPredictor",
        "register_predictor", "get_predictor",
        "Corrector", "NoneCorrector", "LangevinCorrector", "AnnealedLangevinDynamics", "register_corrector", "get_corrector",
    ),
}

__all__ = []
for _mod, _names in _API.items():
    _m = importlib.import_module(f"{__name__}.{_mod}")
    for _n in _names:
        globals()[_n] = getattr(_m, _n)
        __all__.append(_n)
del _mod, _names, _m, _n
