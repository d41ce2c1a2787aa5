"""CPU test: the argument rules of the CAFM memory pool (stage.check_state_args) shared by forward(), forward_from_bank() and
forward_host(): state / resume / state_slots go together on the host path, one entry per clip, distinct slots inside the pool,
the pool's row capacity equal to the configuration's kmax, and no device-path use of a pool with host calls in flight."""
import pytest
import torch


def _pool(slots=5, kmax=30):
    from tscd_b200 import stage
    return stage.CAFMState(slots, kmax, 256, device="cpu")


def test_valid_arguments_pass():
    from tscd_b200.stage import check_state_args
    pool = _pool()
    check_state_args(3, 30)                                                   # stateless
    check_state_args(3, 30, pool, [0, 1, 1], [4, 0, 2], host=True)
    check_state_args(3, 30, pool, torch.tensor([0, 1, 0]), torch.tensor([2, 3, 4], dtype=torch.int32))
    check_state_args(5, 30, pool)                                             # device path: a dense state of B slots
    check_state_args(3, 30, pool, None, [1, 2, 3])


@pytest.mark.parametrize("host", [False, True])
def test_slots_or_flags_without_state(host):
    from tscd_b200.stage import check_state_args
    with pytest.raises(RuntimeError, match="without state"):
        check_state_args(3, 30, None, None, [0, 1, 2], host=host)
    if host:
        with pytest.raises(RuntimeError, match="without state"):
            check_state_args(3, 30, None, [0, 0, 0], None, host=True)


def test_host_state_needs_flags_and_slots():
    from tscd_b200.stage import check_state_args
    pool = _pool()
    for resume, slots in ((None, [0, 1, 2]), ([0, 0, 0], None), (None, None)):
        with pytest.raises(RuntimeError, match="needs resume and state_slots"):
            check_state_args(3, 30, pool, resume, slots, host=True)


@pytest.mark.parametrize("host", [False, True])
def test_lengths_must_be_B(host):
    from tscd_b200.stage import check_state_args
    pool = _pool()
    with pytest.raises(RuntimeError, match="resume has 2 entries for 3 clips"):
        check_state_args(3, 30, pool, [0, 1], [0, 1, 2], host=host)
    with pytest.raises(RuntimeError, match="state_slots has 4 entries for 3 clips"):
        check_state_args(3, 30, pool, [0, 1, 0], [0, 1, 2, 3], host=host)


@pytest.mark.parametrize("host", [False, True])
def test_duplicate_and_out_of_range_slots(host):
    from tscd_b200.stage import check_state_args
    pool = _pool(5)
    with pytest.raises(RuntimeError, match="duplicate state slot"):
        check_state_args(3, 30, pool, [0, 0, 0], [1, 3, 1], host=host)
    with pytest.raises(RuntimeError, match=r"outside \[0, 5\)"):
        check_state_args(3, 30, pool, [0, 0, 0], [0, 5, 1], host=host)
    with pytest.raises(RuntimeError, match=r"outside \[0, 5\)"):
        check_state_args(3, 30, pool, [0, 0, 0], [-1, 2, 1], host=host)


@pytest.mark.parametrize("host", [False, True])
def test_kmax_mismatch_names_expected(host):
    from tscd_b200.stage import check_state_args
    pool = _pool(5, kmax=40)
    with pytest.raises(RuntimeError, match="kmax = 30"):
        check_state_args(3, 30, pool, [0, 0, 0], [0, 1, 2], host=host)


def test_device_path_refuses_pool_with_host_calls_in_flight():
    from tscd_b200.stage import check_state_args
    pool = _pool()
    pool._host_in_flight = 2
    with pytest.raises(RuntimeError, match="in flight"):
        check_state_args(3, 30, pool, None, [0, 1, 2])
    check_state_args(3, 30, pool, [0, 0, 0], [0, 1, 2], host=True)          # more host calls are fine: they are ordered
    pool._host_in_flight = 0
    check_state_args(3, 30, pool, None, [0, 1, 2])


def test_host_path_takes_host_side_flags_and_slots():
    """forward_host copies the flags and the slot map with the call: device tensors are refused with a clear message."""
    from tscd_b200.stage import check_state_args
    pool = _pool()
    dev = torch.zeros(3, dtype=torch.int32, device="meta")
    with pytest.raises(RuntimeError, match="must be host-side"):
        check_state_args(3, 30, pool, [0, 0, 0], dev, host=True)
    with pytest.raises(RuntimeError, match="must be host-side"):
        check_state_args(3, 30, pool, dev, [0, 1, 2], host=True)
    check_state_args(3, 30, pool, torch.zeros(3, dtype=torch.int32), torch.tensor([0, 1, 2]), host=True)
