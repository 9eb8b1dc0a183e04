"""The block count StreamScheduler.replay(handoff=) checks against the Handoff capacity before anything runs: gated_block_count must
equal the length of the gated plan, for the whole recording and summed over any split into windows.  No GPU."""
import random

import pytest

from freeze_omni_b200.scheduler import IPU_CONT, IPU_START, gated_block_count, plan_gated_replay


@pytest.mark.parametrize("H,O", [(10, 6), (4, 4), (3, 0), (0, 0), (5, 1)])
def test_gated_block_count_is_the_plan_length(H, O):
    rng = random.Random(100 * H + O)
    for _ in range(50):
        statuses = [rng.choice([None, None, IPU_START, IPU_CONT, "other"]) for _ in range(rng.randint(0, 60))]
        n = gated_block_count(statuses, O)
        assert n == len(plan_gated_replay(statuses, H, O).blocks)
        cuts = sorted(rng.sample(range(len(statuses) + 1), min(3, len(statuses) + 1)))
        parts = [statuses[a:b] for a, b in zip([0] + cuts, cuts + [len(statuses)])]
        assert sum(len(plan_gated_replay(p, H, O).blocks) for p in parts) == n
