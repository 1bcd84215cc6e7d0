"""CPU checks of the multi-valued-field configuration (AutoIntConfig.bag_size): every refusal happens before a device,
a library call or a process-group call is needed."""
import pytest

from util import ROOT  # noqa: F401  (puts the repository on sys.path)


def _cfg(**kw):
    from recommendsystem_b200.autoint import AutoIntConfig
    return AutoIntConfig(**{"num_fields": 4, "rows_per_field": 10, "batch": 8, **kw})


def test_bag_sizes_per_field():
    assert _cfg().bags() == [1, 1, 1, 1]
    assert _cfg(bag_size=3).bags() == [3, 3, 3, 3]
    assert _cfg(bag_size=(1, 8, 2, 1)).bags() == [1, 8, 2, 1]


@pytest.mark.parametrize("bag_size", [(1, 2, 3), (1, 2, 3, 4, 5), 0, (1, 0, 2, 1), (1, -2, 1, 1)])
def test_bad_bag_size_raises(bag_size):
    from recommendsystem_b200.autoint import AutoIntTrainer
    with pytest.raises(ValueError, match="bag_size"):
        _cfg(bag_size=bag_size).bags()
    with pytest.raises(ValueError, match="bag_size"):
        AutoIntTrainer(_cfg(bag_size=bag_size), device="cpu")


def test_slot_count_must_fit_32_bit_positions():
    from recommendsystem_b200.autoint import AutoIntTrainer
    with pytest.raises(ValueError, match="32-bit"):
        AutoIntTrainer(_cfg(batch=2 ** 25, bag_size=(16, 16, 16, 16)), device="cpu")      # B * S = 2^31


def test_sharded_trainer_refuses_bags_before_any_collective(monkeypatch):
    import torch.distributed as dist
    from recommendsystem_b200 import sharded

    def no_collective(*a, **k):
        raise AssertionError("process-group call before the bag refusal")
    for name in ("get_world_size", "get_rank", "new_group", "all_gather", "all_reduce", "barrier", "broadcast"):
        monkeypatch.setattr(dist, name, no_collective)
    monkeypatch.setattr(sharded, "Exchange", no_collective)
    with pytest.raises(ValueError, match="row-sharded bag fields are not built"):
        sharded.ShardedAutoIntTrainer(_cfg(bag_size=(1, 2, 1, 1)), device="cpu")
