from .ddim_scheduler import DDIMNoiseScheduler, DDIMNoiseSchedulerOutput
from .dpm_solver import DPMSolverMultistepScheduler, DPMSolverMultistepSchedulerOutput
from .unipc import UniPCMultistepScheduler, UniPCMultistepSchedulerOutput

__all__ = ["DDIMNoiseScheduler", "DDIMNoiseSchedulerOutput", "DPMSolverMultistepScheduler",
           "DPMSolverMultistepSchedulerOutput", "UniPCMultistepScheduler", "UniPCMultistepSchedulerOutput"]
