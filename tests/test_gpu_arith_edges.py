"""sm_100a field and point arithmetic of every group at extreme operands, through the C ABI's test hooks: the device
build of each group's translation unit (its out-of-line multipliers, constant-bank modulus, dedicated squaring and
fused sums of products, as that unit enables them) against big-integer arithmetic on the raw Montgomery limbs
(opcases.check_field_edges) and the oracle's point formulas (opcases.check_point_edges)."""
import pytest

from oracle import oracle as O
from tests import opcases

pytestmark = pytest.mark.gpu


def _runner(g):
    import gnark_crypto_b200  # noqa: F401
    from importlib import import_module

    mx = import_module("gnark-crypto_b200.multiexp")

    def run(op, a, b, out_words):
        return mx.test_op(g, op, a, b, out_words)

    return run


@pytest.mark.parametrize("g", list(O.GROUPS))
def test_field_edges_device(g):
    """every extreme value against every other (all rotations of the extreme list) plus 20k random operands"""
    opcases.check_field_edges(O.GROUPS[g], _runner(g), n_random=20000)


@pytest.mark.parametrize("g", list(O.GROUPS))
def test_point_edges_device(g):
    opcases.check_point_edges(O.GROUPS[g], _runner(g))
