"""CPU: state.set_hp_grid flattens an hp dict in the key order of default_hyperparams(), which must be the flat layout
of the C ABI (include/mscope_b200.h, enum msb_family) that the checker's flat_hp writes."""
import numpy as np
import pytest

import common_b200 as cb
from common_b200.state import flat_hp
from oracle_lib import Oracle


@pytest.mark.parametrize("desc", [cb.bb, cb.bbnc, cb.bnb, cb.gp, cb.nich, cb.dd(7), cb.dm(5), cb.niw(1), cb.niw(3)],
                         ids=lambda d: d().name() + str(d()._param() or ""))
def test_flat_hp_is_the_abi_layout(desc):
    rng = np.random.default_rng(0)
    hp = {k: rng.uniform(0.5, 3.0, np.shape(v)) if np.ndim(v) else float(rng.uniform(0.5, 3.0))
          for k, v in desc().default_hyperparams().items()}
    assert np.array_equal(flat_hp(desc(), hp), Oracle.flat_hp(desc, hp))
    assert np.array_equal(flat_hp(desc(), desc().default_hyperparams()), Oracle.flat_hp(desc))
