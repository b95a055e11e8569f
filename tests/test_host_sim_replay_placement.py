"""The display-loop super-block makes room in its queue of deferred TIA writes in one of two places, chosen per kernel flavour
(csrc/pong_superblocks.cuh, REPLAY_AT_TOP): the CTA-synchronous flavours replay at the top of an iteration, the one-warp flavour
where writes are queued.  tests/host_sim runs the one-warp choice; these builds force the other one, with the normal queue and
with nine slots (early replays at every other event), and must match the oracle frame for frame."""
import pytest

from test_host_sim import _build_variant, _run_fast_against_oracle


@pytest.mark.parametrize("slots", [24, 9])
def test_replay_at_top_of_iteration_matches_oracle(slots):
    L, sim = _build_variant(f"replaytop{slots}", "-DA26_SB_REPLAY_AT_TOP=true", f"-DA26_SB_MAX_EVENTS={slots}")
    _run_fast_against_oracle(L, sim, 400, seed=8)
