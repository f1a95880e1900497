"""Which text a context keeps resident after each kind of call, on the B200: on one GPU and on a device group of three
logical shards of it, with device buffers as torch CUDA tensors.  The same cases run on the emulator in
test_emu_resident_index.py; resident_cases.py describes them."""
import pytest

from device_entry_cases import CudaMem
from resident_cases import CALLS, SETUPS, SHARD_MIN, check_call

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mem():
    return CudaMem()


@pytest.mark.parametrize("name", sorted(CALLS))
@pytest.mark.parametrize("setup", sorted(SETUPS))
@pytest.mark.parametrize("group", [False, True], ids=["single", "group"])
def test_call_then_search_with_resident_index(mem, group, setup, name, monkeypatch):
    from deltaq_b200._native import Context
    if group:
        monkeypatch.setenv("DQ_SHARD_MIN", SHARD_MIN)
    with Context(device=[0, 0, 0] if group else 0) as ctx:
        check_call(ctx, mem, setup, name, monkeypatch)
