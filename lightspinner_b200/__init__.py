"""lightspinner_b200 -- B200-native MALI hot path for Lightspinner (formal solution + Gamma + statistical equilibrium).

    from lightspinner_b200 import Context, piecewise_linear_1d      # drop-ins for rh_method.Context / formal_solver
    from lightspinner_b200 import MaliEngine                        # batched columns on one GPU
    from lightspinner_b200 import NgOptions                         # opt-in Ng acceleration (ng=NgOptions())
    from lightspinner_b200 import RayDepthData                      # what compute_rays_depth returns
    from lightspinner_b200 import RadiativeRates                    # what compute_rates returns
    from lightspinner_b200 import ResponseFunction                  # what MaliEngine.compute_response returns

The compute lives in csrc/ (hand-written CUDA for sm_100a behind the C ABI of include/mali_b200.h); there is no CPU
fallback.  Importing the package does not touch the GPU; constructing a Context / MaliEngine does.
"""

__all__ = ['Context', 'BatchContext', 'piecewise_linear_1d', 'IPsi', 'UV', 'MaliEngine', 'NgOptions', 'RayDepthData',
           'RadiativeRates', 'ResponseFunction']


def __getattr__(name):
    if name in ('Context', 'BatchContext', 'piecewise_linear_1d', 'IPsi', 'UV'):
        from . import context
        return getattr(context, name)
    if name in ('MaliEngine', 'RayDepthData', 'RadiativeRates'):
        from . import engine
        return getattr(engine, name)
    if name == 'ResponseFunction':
        from .response import ResponseFunction
        return ResponseFunction
    if name == 'NgOptions':
        from .ng import NgOptions
        return NgOptions
    raise AttributeError(name)
