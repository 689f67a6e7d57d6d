"""ReplayBuffer (row a18) against the reference's own class (phc/learning/replay_buffer.py) on CPU with the same seed: circular
store, the pre-fill `% head` rule, the permutation refresh.  tests/golden/replay.npz holds what the reference class stored and
sampled (tests/golden/make_golden.py:gen_replay)."""
import torch

from tests.helpers import load

STORE_SIZES = [8, 8, 8, 20, 13, 50, 3]          # partial fill, wrap-around, a full-size store
SAMPLE_SIZES = (5, 17, 30)                      # crosses the permutation refresh several times


def test_store_and_sample_match_the_reference():
    from phc_b200.learning.amp_agent import ReplayBuffer
    g = load("replay.npz")
    size = int(g["size"])
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(5)                    # the reference buffer drew its permutations from this generator state
        ours = ReplayBuffer(size, g["rows0"].shape[1], "cpu")
        for step, n in enumerate(STORE_SIZES):
            rows = g[f"rows{step}"]
            assert rows.shape[0] == n
            ours.store(rows)
            assert ours.get_total_count() == int(g[f"total{step}"]) and ours.get_buffer_size() == size
            assert torch.equal(ours.data, g[f"data{step}"]), f"store {step}"
            for k in SAMPLE_SIZES:
                idx = ours.sample_indices(k)
                assert torch.equal(ours.data[idx], g[f"sample{step}_{k}"]), f"sample {k} after store {step}"
