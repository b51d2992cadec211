"""Options of the opt-in Ng acceleration of the population iteration (Auer 1987; include/mali_b200.h, mali_iterate_ng).

    from lightspinner_b200 import BatchContext, NgOptions
    batch = BatchContext(columns, ng=NgOptions())          # order 2, delay 3, period 3

Per column and active atom, the last order + 2 solved population vectors are kept; once more than `delay` solves have
been done, every `period`-th solve is followed by a least-squares extrapolation from them.  (2, 3, 3) is the measured
default: on CaII+H/FALC it converges in 32 iterations instead of 79, while (2, 2, 2) did not converge within 400
(DESIGN.md section 4).  The reference has no Ng acceleration, so with it on the iteration counts differ from the
reference's; the fixed point is the same.
"""
from dataclasses import dataclass


@dataclass(frozen=True)
class NgOptions:
    order: int = 2
    delay: int = 3
    period: int = 3

    def __post_init__(self):
        for k in ('order', 'delay', 'period'):
            v = getattr(self, k)
            if isinstance(v, bool) or not isinstance(v, int):
                raise ValueError('NgOptions.%s must be an int, got %r' % (k, v))
        if not 1 <= self.order <= 3:
            raise ValueError('NgOptions.order must be 1, 2 or 3, got %d' % self.order)
        if self.delay < 0:
            raise ValueError('NgOptions.delay must be >= 0, got %d' % self.delay)
        if self.period < 1:
            raise ValueError('NgOptions.period must be >= 1, got %d' % self.period)

    def due(self, nse):
        """Whether an extrapolation follows the nse-th solve since the last reset."""
        return nse > self.delay and nse >= self.order + 2 and (nse - self.delay) % self.period == 0
