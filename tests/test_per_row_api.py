"""CPU tests of the per-utterance loss API (reduction="none" / "mean"): the two C entry points load, refuse a NULL
per_row / grad_rows with GE2E_ERR_ARGUMENT before anything is launched, and the Python layer rejects a bad
reduction before touching a device -- all without a GPU."""
import pytest
import torch

ARG = -3                         # GE2E_ERR_ARGUMENT
NEW = ("ge2e_b200_forward_per_row_typed", "ge2e_b200_backward_per_row_typed")


@pytest.fixture(scope="module")
def h():
    from speaker_embedding_ge2e_loss_b200 import _lib, build
    build.build()   # nvcc cross-compiles sm_100a without a GPU
    return _lib.lib()


def test_per_row_symbols_load_through_prototypes(h):
    from speaker_embedding_ge2e_loss_b200 import _lib
    for name in NEW:
        assert name in _lib.PROTOTYPES
        fn = getattr(h, name)
        assert fn.restype is _lib.PROTOTYPES[name][0] and fn.argtypes == _lib.PROTOTYPES[name][1]
    # same arguments as the scalar entry points, plus per_row (forward); grad_rows in place of grad_out (backward)
    assert len(_lib.PROTOTYPES[NEW[0]][1]) == len(_lib.PROTOTYPES["ge2e_b200_forward_typed"][1]) + 1
    assert _lib.PROTOTYPES[NEW[1]][1] == _lib.PROTOTYPES["ge2e_b200_backward_typed"][1]


@pytest.mark.parametrize("variant,precision", [(0, 0), (1, 0), (0, 1), (0, 2), (0, 3)])
def test_null_per_row_is_an_argument_error(h, variant, precision):
    # every other pointer is a non-null dummy: the call must return before touching any of them
    assert h.ge2e_b200_forward_per_row_typed(1, 0, None, 4, 8, 256, 1, 1, 1e-6, variant, precision, 1, 1, 1, 1, 1, 1,
                                             1, 1, 1, None, 1, 1 << 20, None) == ARG


@pytest.mark.parametrize("variant,precision", [(0, 0), (1, 0), (0, 1), (0, 2), (0, 3)])
def test_null_grad_rows_is_an_argument_error(h, variant, precision):
    assert h.ge2e_b200_backward_per_row_typed(1, 0, None, 1, 1, 1, 1, 1, 1, 1, 4, 8, 256, 1, 1, 1e-6, variant,
                                              precision, None, 1, 1, 1, 1, 0, 1, 1 << 20, None) == ARG


@pytest.mark.parametrize("reduction", ["avg", "", None, "SUM"])
def test_unknown_reduction_raises(reduction):
    from speaker_embedding_ge2e_loss_b200 import GE2ELoss, ge2e_loss
    E = torch.zeros(4, 8, 16)
    w, b = torch.tensor(10.0), torch.tensor(-5.0)
    with pytest.raises(ValueError, match="reduction"):
        ge2e_loss(E, w, b, reduction=reduction)
    with pytest.raises(ValueError, match="reduction"):
        GE2ELoss(reduction=reduction, device="cpu")


def test_reduction_is_keyword_only():
    from speaker_embedding_ge2e_loss_b200 import ge2e_loss
    E = torch.zeros(4, 8, 16)
    with pytest.raises(TypeError):
        ge2e_loss(E, torch.tensor(10.0), torch.tensor(-5.0), 1e-6, "softmax", "fp32", None, 0, "none")


def test_none_with_process_group_raises():
    from speaker_embedding_ge2e_loss_b200 import GE2ELoss
    with pytest.raises(ValueError, match="process_group"):
        GE2ELoss(reduction="none", process_group=object(), device="cpu")
