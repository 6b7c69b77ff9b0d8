"""CPU tests of the element-type arguments of the _typed entry points (enum ge2e_dtype): unknown codes, and a dE type
that is neither fp32 nor E's own, are refused with GE2E_ERR_ARGUMENT before anything is launched, so these run
without a GPU."""
import pytest

ARG = -3                         # GE2E_ERR_ARGUMENT
F32, BF16, F16 = 0, 1, 2
BAD_PAIRS = [(3, F32), (-1, F32), (BF16, F16), (F16, BF16), (F32, BF16), (F32, F16), (BF16, 7)]


@pytest.fixture(scope="module")
def h():
    from speaker_embedding_ge2e_loss_b200 import _lib, build
    build.build()   # nvcc cross-compiles sm_100a without a GPU
    assert (_lib.DT_F32, _lib.DT_BF16, _lib.DT_F16) == (F32, BF16, F16)
    return _lib.lib()


def test_version_bumped(h):
    assert h.ge2e_b200_version() >= 101


@pytest.mark.parametrize("e_dt", [3, -1, 100])
def test_e_only_entry_points_refuse_unknown_codes(h, e_dt):
    # pointers are non-null dummies: the call must return before touching them
    assert h.ge2e_b200_prep_typed(1, e_dt, None, 4, 8, 256, 0, 1, 1, 1, 1, None) == ARG
    assert h.ge2e_b200_forward_typed(1, e_dt, None, 4, 8, 256, 1, 1, 1e-6, 0, 0, 1, 1, 1, 1, None, 1, 1, None, None,
                                     None, 0, None) == ARG


@pytest.mark.parametrize("e_dt,de_dt", BAD_PAIRS)
def test_dE_entry_points_refuse_bad_pairs(h, e_dt, de_dt):
    assert h.ge2e_b200_bwd_finalize_typed(1, e_dt, None, 1, 1, 1, 1, 1, None, 4, 8, 256, 1, 1, 1e-6, 0, 1, 1, de_dt,
                                          None) == ARG
    assert h.ge2e_b200_backward_typed(1, e_dt, None, 1, 1, 1, 1, None, 1, None, 4, 8, 256, 1, 1, 1e-6, 0, 0, 1, 1, 1, 1,
                                      1, de_dt, None, 0, None) == ARG
    assert h.ge2e_b200_forward_backward_typed(1, e_dt, None, 4, 8, 256, 1, 1, 1e-6, 0, 0, 1, 1, 1, 1, 1, None, 1, 1, 1,
                                              1, 1, 1, de_dt, None, 0, None) == ARG


@pytest.mark.parametrize("de_dt", [3, -1])
def test_scale_grads_refuses_unknown_codes(h, de_dt):
    assert h.ge2e_b200_scale_grads_typed(1, 1, de_dt, 16, 1, 1, 1, None) == ARG


def test_plane_alignment_is_per_element_type():
    from speaker_embedding_ge2e_loss_b200 import _lib
    assert _lib.planes_need_copy(8, _lib.FP32_SPLIT)                 # fp32: 16 bytes
    assert not _lib.planes_need_copy(8, _lib.FP32_SPLIT, 2)          # bf16 / fp16: 8 bytes
    assert _lib.planes_need_copy(4, _lib.F16, 2)
    assert not _lib.planes_need_copy(4, _lib.TF32, 2)                # only the plane precisions need it
