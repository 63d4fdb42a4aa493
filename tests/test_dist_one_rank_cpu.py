"""CPU: a process on its own is the one-rank case of the sharded rollout block (cmbpo_b200.dist.Ranks()).  Its
gathers return its own vector without a process group, and the batch-wide rules over one rank are identities, so
the one-GPU block runs the code of the sharded block."""
import numpy as np
import torch.distributed as dist

from cmbpo_b200.dist import Ranks, cap_split, rank_order_sum


def test_one_rank_gather_needs_no_process_group():
    assert not (dist.is_available() and dist.is_initialized())
    r = Ranks()
    assert (r.group, r.rank, r.world, r.root, r.sharded) == (None, 0, 1, 0, False)
    for vec in (np.array([7], np.int64), np.arange(10, dtype=np.int64), np.linspace(-1.0, 2.0, 12).reshape(6, 2)):
        g = r.gather(vec, device="cpu")
        assert g.shape == (1,) + vec.shape and g.dtype == vec.dtype
        assert g.tobytes() == vec.tobytes()


def test_rules_over_one_rank_are_identities():
    rng = np.random.default_rng(0)
    for _ in range(200):
        row = rng.standard_normal(int(rng.integers(1, 40))) * 10.0 ** rng.integers(-5, 16)
        assert rank_order_sum(Ranks().gather(row)).tobytes() == row.tobytes()
        h = rng.integers(0, 1000, int(rng.integers(1, 40)))
        assert rank_order_sum(h[None]).tobytes() == h.tobytes()
        survivors = int(rng.integers(0, 1000))
        for n in {0, survivors, int(rng.integers(0, survivors + 1))}:        # the sampler caps n <= survivors
            assert cap_split(n, [survivors]) == [n]
