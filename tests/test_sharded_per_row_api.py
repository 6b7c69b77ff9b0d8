"""CPU tests of the speaker-sharded per-utterance API: the three C entry points load with the header's arity, refuse a
NULL grad_rows (and the peer entry point a NULL row_scale or a bad rank count) before anything is launched, and the
Python layer refuses an unknown reduction before any device or process-group call -- all without a GPU."""
import ctypes as C

import pytest
import torch

SHAPE, ARG = -1, -3              # GE2E_ERR_SHAPE, GE2E_ERR_ARGUMENT
NEW = {"ge2e_b200_bwd_rows_per_row": "ge2e_b200_bwd_rows",
       "ge2e_b200_bwd_finalize_per_row_typed": "ge2e_b200_bwd_finalize_typed",
       "ge2e_b200_bwd_rows_peers_per_row": None}


@pytest.fixture(scope="module")
def h():
    from speaker_embedding_ge2e_loss_b200 import _lib, build
    build.build()   # nvcc cross-compiles sm_100a without a GPU
    return _lib.lib()


def owners(n):
    return (C.c_void_p * n)(*([1 << 12] * n))


def test_sharded_per_row_symbols_load_through_prototypes(h):
    from speaker_embedding_ge2e_loss_b200 import _lib
    for name, scalar in NEW.items():
        fn = getattr(h, name)
        assert fn.restype is _lib.PROTOTYPES[name][0] and fn.argtypes == _lib.PROTOTYPES[name][1]
        if scalar is not None:      # grad_rows in place of grad_out, every other parameter as the scalar entry point
            assert _lib.PROTOTYPES[name][1] == _lib.PROTOTYPES[scalar][1]
    assert len(_lib.PROTOTYPES["ge2e_b200_bwd_rows_peers_per_row"][1]) == 24


@pytest.mark.parametrize("variant,precision", [(0, 0), (1, 0), (0, 1), (0, 2), (0, 3)])
def test_null_grad_rows_is_an_argument_error(h, variant, precision):
    # every other pointer is a non-null dummy: the call must return before touching any of them
    assert h.ge2e_b200_bwd_rows_per_row(1, 1, 1, 1, 1, 1, 1, 128, 256, 128, 8, 256, 1, 1, 1e-6, variant, precision,
                                        None, 1, 1, 1, 1, 1 << 20, None) == ARG
    assert h.ge2e_b200_bwd_finalize_per_row_typed(1, 0, None, 1, 1, 1, 1, 1, 1, 128, 8, 256, 1, 1, 1e-6, variant,
                                                  None, 1, 0, None) == ARG
    assert h.ge2e_b200_bwd_rows_peers_per_row(1, 1, 1, 1, 1, 1, 128, 256, 128, 8, 256, 1, 1, 1e-6, variant, precision,
                                              None, 1, 1, owners(2), 2, 1, 1 << 20, None) == ARG


def test_peer_entry_point_host_refusals(h):
    args = lambda **o: (1, 1, 1, 1, 1, o.get("row_scale", 1), o.get("n_local", 128), 256, 0, 8, 256, 1, 1, 1e-6, 0, 1,
                        1, 1, 1, owners(8), o.get("n_ranks", 2), 1, 1 << 20, None)
    f = h.ge2e_b200_bwd_rows_peers_per_row
    assert f(*args(row_scale=None)) == ARG                  # the forward must have prepared dE_hat
    assert f(*args(n_ranks=1)) == SHAPE
    assert f(*args(n_ranks=9)) == SHAPE
    assert f(*args(n_local=64)) == SHAPE                    # n_local * n_ranks != n_total


@pytest.mark.parametrize("reduction", ["avg", "", None, "mean", "SUM"])
def test_unknown_reduction_raises_before_any_group_call(reduction):
    import torch.distributed as dist

    from speaker_embedding_ge2e_loss_b200 import ShardedGE2EPlan
    from speaker_embedding_ge2e_loss_b200.sharded import sharded_ge2e_loss
    assert not dist.is_initialized()        # a group call would raise something other than the ValueError below
    E = torch.zeros(4, 8, 16)
    w, b = torch.tensor(10.0), torch.tensor(-5.0)
    with pytest.raises(ValueError, match="reduction"):
        sharded_ge2e_loss(E, w, b, reduction=reduction)
    with pytest.raises(ValueError, match="reduction"):
        ShardedGE2EPlan(4, 8, 0, 8, 16, device="cpu", reduction=reduction)


def test_reduction_is_keyword_only():
    from speaker_embedding_ge2e_loss_b200.sharded import sharded_ge2e_loss
    with pytest.raises(TypeError):
        sharded_ge2e_loss(torch.zeros(4, 8, 16), torch.tensor(10.0), torch.tensor(-5.0), 1e-6, "softmax", "fp32", None,
                          None, "none")
