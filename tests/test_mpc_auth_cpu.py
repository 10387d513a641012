"""`collaborative.auth_share_table`: authenticated additive shares in Python integers."""
import numpy as np

from renegade_b200 import collaborative as co
from renegade_b200.fields import SCALAR_FIELD_MODULUS as R, limbs_to_scalars, scalars_to_limbs


def _sums(tables):
    return [sum(col) % R for col in zip(*[limbs_to_scalars(t) for t in tables])]


def test_auth_share_table_sums_to_values_and_macs():
    vals = [0, 1, 2, R - 1, 2**200 + 17]
    keys = scalars_to_limbs([11, R - 4, 123456789])
    alpha = (11 + R - 4 + 123456789) % R
    shares, macs = co.auth_share_table(scalars_to_limbs(vals), 3, keys, seed=5)
    assert len(shares) == len(macs) == 3
    assert all(s.shape == (len(vals), 4) and s.dtype == np.uint64 for s in shares + macs)
    assert _sums(shares) == vals
    assert _sums(macs) == [alpha * v % R for v in vals]


def test_auth_share_table_shares_look_random():
    shares, _ = co.auth_share_table(scalars_to_limbs([7] * 4), 2, scalars_to_limbs([1, 2]), seed=9)
    assert len(set(limbs_to_scalars(shares[0]))) == 4
