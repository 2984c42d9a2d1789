"""Which CUDA kernels a call launched, read from a torch.profiler trace."""
import torch


def kernels_launched(fn, match):
    """Names of the CUDA kernels `fn` launches whose name contains `match` (profiler trace)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if match in e.name]
