"""The generic gate check whose selector products q_r*b + q_o*c + q_4*d run on the tensor cores (kernels.cuh k_check_tc), against
big-int verdicts: range_check segments with random bounds (their values enter the row template as selector constants), random
witnesses and random faults, at instance counts that are not a multiple of the 128-instance block.  Run on the B200 box with
`pytest -m gpu`."""
import random

import pytest

import plonk_gadgets_b200 as pg
from tests.fault_cases import eval_rows
from tests.programs import Q

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("seed", [1, 2])
def test_random_bounds_and_faults_vs_big_ints(oracle, seed):
    import torch
    assert torch.cuda.is_available(), "this test needs the B200"
    rng = random.Random(seed)
    n = torch.cuda.get_device_properties(0).multi_processor_count * 320 + rng.choice([77, 1, 127])   # the one-thread-per-instance kernel
    lo = rng.randrange(2 ** rng.randrange(1, 200))
    hi = lo + rng.randrange(2, 2 ** rng.randrange(8, 96))
    wit = [rng.choice([lo, hi - 1, hi, lo + rng.randrange(hi - lo), rng.randrange(Q)]) for _ in range(n)]
    c = pg.StandardComposer(device=0, check_mode=pg.CHECK_GENERIC)
    w = c.add_input(oracle.from_ints(wit))
    y = pg.range_check(c, oracle.from_ints([lo]), oracle.from_ints([hi]), w)
    assert oracle.to_ints(y.values(0, 64)) == [1 if lo <= v < hi else 0 for v in wit[:64]]
    base_row = 3
    rows_per = (c.circuit_size() - base_row) // n
    assert base_row + rows_per * n == c.circuit_size()
    c.check_stats(reset=True)
    assert c.check_circuit_satisfied() == (0, None)
    assert c.check_stats(reset=True)["instance_generic"][1] >= rows_per * n
    # faults: the witness or the result of each chosen instance changed by a random amount (block ends, the partial last block,
    # random instances); only the instance's own rows read either variable
    chosen = sorted({0, 127, 128, n - 1, n - 2, n - (n % 128)} | {rng.randrange(n) for _ in range(12)})
    w_ids, y_ids = w.ids(), y.ids()
    undo, exp = [], []
    for i in chosen:
        var = int(rng.choice([w_ids, y_ids])[i])
        old = c.variables(var, 1)[0].copy()
        c.poke_variable(var, oracle.from_ints([(oracle.to_ints(old[None])[0] + rng.choice([1, Q - 1, rng.randrange(1, Q)])) % Q])[0])
        undo.append((var, old))
    for i in chosen:
        r0 = base_row + rows_per * i
        exp += [r0 + r for r in eval_rows(oracle, c.rows(r0, rows_per, want=("w_val", "sel", "pi")))]
    exp = sorted(set(exp))
    assert exp
    assert c.check_circuit_satisfied() == (len(exp), exp[0])
    assert c.check_stats(reset=True)["instance_generic"][1] >= rows_per * n
    for var, old in reversed(undo):
        c.poke_variable(var, old)
    assert c.check_circuit_satisfied() == (0, None)
    c.close()
