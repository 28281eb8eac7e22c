"""CPU, needs the original project's sources (ref_harness.REFERENCE_ROOT): the seeded random scenarios of test_fuzz_gpu.py,
restricted to what the reference can express (its hard-coded 1000-step cap, no shared learner), run through the LIVE
reference classes (oracle/ref_harness.py, randomness injected) and through the C oracle — traces and final tables must
agree bit for bit. Together with test_fuzz_gpu.py (CUDA == oracle on the same generator) this extends reference parity
from the fixed fixtures to option combinations no fixture has."""
import numpy as np
import pytest

import multiagent_rlrm_b200 as P
import oracle as O
from ref_harness import REFERENCE_MISSING, reference_available

from test_fuzz_gpu import random_scenario

pytestmark = [pytest.mark.reference,
              pytest.mark.skipif(not reference_available(), reason=REFERENCE_MISSING)]

SEEDS = list(range(0, 128, 4))


@pytest.mark.parametrize("seed,n,T", [(s, 2, 220) for s in SEEDS] + [(s, 1, 3000) for s in range(1, 128, 16)])
def test_random_scenario_oracle_equals_live_reference(seed, n, T):
    import ref_harness as H

    sc, _opts = random_scenario(seed)
    sc.max_steps, sc.shared_q = 1000, False
    ref = H.run_reference(sc.to_dict(), n, T, np.float32, pre_resets=1)
    c = P.compile_scenario(sc)
    o = O.Oracle(c, n, "f32")
    o.reset(); o.reset()
    tr = O.unpack_trace(o.train(0, T, learn=True, trace=True), n, c.n_agents)
    info = f"seed {seed}: {sc.env}/{sc.map_name} A={len(sc.starts)} {sc.algo} lr={sc.learning_rate} rsh={sc.use_rsh}"
    for k in ("action", "cell", "q", "term", "trunc"):
        assert np.array_equal(tr[k], ref[k].astype(np.int32)), f"{info}: {k}"
    q_ref = ref["q_final"]
    assert np.array_equal(o.q.reshape(-1), np.asarray(q_ref).reshape(-1)), f"{info}: final Q tables"
    if "e_final" in ref and ref["e_final"] is not None and sc.algo == "qlambda":
        assert np.array_equal(o.e.reshape(-1), np.asarray(ref["e_final"]).reshape(-1)), f"{info}: final traces"
