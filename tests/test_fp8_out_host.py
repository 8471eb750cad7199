"""Host-side part of the e4m3fn matmul output: the sharded linear refuses it."""
import pytest
import torch

from fp8_sharded import ShardedScaledMM


@pytest.mark.parametrize("odt", [torch.float8_e4m3fn, torch.float8_e5m2])
@pytest.mark.parametrize("mode", ["allgather", "push", "peers", "multicast", "auto"])
def test_sharded_refuses_fp8_out(odt, mode):
    """FP8 results are not exchanged between ranks: every entry point raises before any launch or collective."""
    W = torch.zeros(64, 32, dtype=torch.uint8)
    lin = ShardedScaledMM(W, torch.ones(1))
    x = torch.zeros(4, 32, dtype=torch.uint8)
    with pytest.raises(ValueError, match="out_dtype"):
        lin(x, torch.ones(1), out_dtype=odt, mode=mode)
    for fwd in (lin.forward_push, lin.forward_peers, lin.forward_multicast):
        with pytest.raises(ValueError, match="out_dtype"):
            fwd(x, torch.ones(1), out_dtype=odt)
