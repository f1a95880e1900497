"""Which text a context keeps resident after each kind of call, on the CPU logic emulator (tests/emu; NOT the product):
on one device and on a device group of three logical shards.  The same cases run on the B200 in
test_resident_index_gpu.py; resident_cases.py describes them."""
import pytest

from device_entry_cases import HostMem
from resident_cases import CALLS, SETUPS, SHARD_MIN, check_call


@pytest.mark.parametrize("name", sorted(CALLS))
@pytest.mark.parametrize("setup", sorted(SETUPS))
@pytest.mark.parametrize("group", [False, True], ids=["single", "group"])
def test_call_then_search_with_resident_index(group, setup, name, monkeypatch):
    import emu
    from deltaq_b200._native import Context
    if group:
        monkeypatch.setenv("DQ_SHARD_MIN", SHARD_MIN)
    with Context(device=[0, 0, 0] if group else None, lib=emu.library()) as ctx:
        check_call(ctx, HostMem(), setup, name, monkeypatch)
