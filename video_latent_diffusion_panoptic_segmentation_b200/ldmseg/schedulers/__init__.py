from .ddim_scheduler import DDIMNoiseScheduler, DDIMNoiseSchedulerOutput
from .dpm_solver import DPMSolverMultistepScheduler, DPMSolverMultistepSchedulerOutput

__all__ = ["DDIMNoiseScheduler", "DDIMNoiseSchedulerOutput", "DPMSolverMultistepScheduler",
           "DPMSolverMultistepSchedulerOutput"]
