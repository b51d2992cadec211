"""Stand-in for compute-sanitizer's racecheck on the TMA-ring protocol: the CHECKED build of the library (-DMALI_CHECK,
lightspinner_b200/_lib/libmali_b200_check.so, built next to the stock library by build()) makes every lane compare,
at every depth step, what arrived through the ring -- heights, populations, background field, line-profile row -- with a direct global load of the
same element of (tile, depth k), and raise status bit 2 (value 4) on any mismatch.  A ring stage refilled before its
last reader was done, or read before its copy landed, cannot pass this: the stage would hold another depth's record.
Run on every fixture shape (82 / 81 / 512 depths, 3 / 5 / 10 rays), both arithmetic modes, the per-call entry point and
the device loop; results must also stay bit-identical to the stock build's."""
import os

import numpy as np
import pytest
import torch

from helpers import drop_depth, load_golden
from lightspinner_b200.build import CHECK_LIB as LIB

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('arith', ['exact', 'contracted'])
@pytest.mark.parametrize('name', ['c1_falc_ca', 'c2_falc_cah', 'c1v_jitter_ca3', 'stress_r10_d512', 'c1_odd'])
def test_ring_delivers_the_right_record_at_every_step(name, arith):
    assert os.path.isfile(LIB), 'checked build missing: __graft_entry__.build() makes it'
    from lightspinner_b200.engine import MaliEngine
    p, _ = load_golden('c1_falc_ca' if name == 'c1_odd' else name)
    if name == 'c1_odd':
        p = drop_depth(p, 40)               # 81 depth points: the last ring group holds a single step
    ncol = 3
    chk = MaliEngine(p, ncol, library=LIB, arith=arith)
    ref = MaliEngine(p, ncol, arith=arith)
    for e in (chk, ref):
        e.upload([p] * ncol)
        for it in range(1, 6):
            e.formal_sol_gamma_matrices()
            if it > 3:
                e.stat_equil()
        e.reset_iteration_state()
        e.iterate_async(6)
        torch.cuda.synchronize()
    status = chk.t_status.cpu().numpy()
    assert not (status & 4).any(), 'a ring stage held the wrong record (status %s)' % status
    assert np.array_equal(chk.t_pops.cpu().numpy(), ref.t_pops.cpu().numpy())
    assert np.array_equal(chk.t_I.cpu().numpy(), ref.t_I.cpu().numpy())
    chk.close()
    ref.close()
