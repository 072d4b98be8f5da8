"""The permutation argument's recalled constants, re-derived: the coset representatives k = (1, K1, K2, K3) = (1, 7, 13, 17) of
dusk-plonk 0.8 permutation/constants.rs must put the four wires in distinct cosets of every evaluation domain up to 2^32 --
k_i / k_j outside the subgroup of order 2^32 (which contains every smaller domain) for i != j -- or the identity permutation
k_w * w^i would not be injective and the copy constraints would not bind."""
from itertools import combinations

from oracle import pymodel as pm
from tests import permutation_model as perm
from tests.programs import Q


def test_coset_constants_lie_in_distinct_cosets():
    assert perm.PERM_K == (1, 7, 13, 17)
    for a, b in combinations(perm.PERM_K, 2):
        ratio = a * pow(b, Q - 2, Q) % Q
        assert pow(ratio, 1 << pm.TWO_ADICITY, Q) != 1, (a, b)


def test_identity_positions_are_distinct_on_a_small_domain():
    """The same property, element by element, on the domain of 2^6 points: the 4 x 64 identities k_w * w^i are pairwise distinct."""
    g = pm.group_gen(6)
    ids = {k * pow(g, i, Q) % Q for k in perm.PERM_K for i in range(64)}
    assert len(ids) == 4 * 64
