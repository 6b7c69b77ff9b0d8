"""CPU tests of the contrast loss's peer-memory entry points: both load with the header's arity and refuse NULL pointers,
a bad rank count, a bad shape and the fp16-plane precisions before any device call -- all without a GPU (every pointer
is a dummy the call must never touch)."""
import ctypes as C

import pytest

OK, SHAPE, UNSUPPORTED, ARG = 0, -1, -2, -3
NAMES = ("ge2e_b200_contrast_bwd_rows_peers", "ge2e_b200_contrast_bwd_rows_peers_per_row")


@pytest.fixture(scope="module")
def h():
    from speaker_embedding_ge2e_loss_b200 import _lib, build
    build.build()   # nvcc cross-compiles sm_100a without a GPU
    return _lib.lib()


def owners(n, p=1 << 12):
    return (C.c_void_p * n)(*([p] * n))


def args(**o):
    """e_hat, c_hat_all, cos_diag, row_stat, row_kstar, n_local, n_total, spk_offset, M, D, w, b, eps, precision,
    grad, dE_hat, dwdb_accum, dC_owner_host, n_ranks, stream; base: 2 ranks of 128 speakers, TF32."""
    n_ranks = o.get("n_ranks", 2)
    return (1, 1, 1, 1, o.get("row_kstar", 1), o.get("n_local", 128), 256, 0, o.get("M", 8), o.get("D", 256), 1, 1,
            1e-6, o.get("precision", 1), o.get("grad", 1), 1, o.get("dwdb", 1),
            o.get("owners", owners(max(n_ranks, 1))), n_ranks, None)


def test_contrast_peer_symbols_load_through_prototypes(h):
    from speaker_embedding_ge2e_loss_b200 import _lib
    for name in NAMES:
        fn = getattr(h, name)
        assert fn.restype is _lib.PROTOTYPES[name][0] and fn.argtypes == _lib.PROTOTYPES[name][1]
        assert len(_lib.PROTOTYPES[name][1]) == 20
    # grad_rows in place of grad_out, every other parameter as the scalar entry point
    assert _lib.PROTOTYPES[NAMES[0]][1] == _lib.PROTOTYPES[NAMES[1]][1]


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("over,code", [
    (dict(grad=None), ARG), (dict(row_kstar=None), ARG), (dict(dwdb=None), ARG), (dict(owners=None), ARG),
    (dict(n_ranks=1), SHAPE), (dict(n_ranks=9), SHAPE), (dict(n_local=64), SHAPE), (dict(M=1), SHAPE),
    (dict(precision=2), UNSUPPORTED), (dict(precision=3), UNSUPPORTED), (dict(precision=7), ARG),
    (dict(owners=(C.c_void_p * 2)(1 << 12, None)), ARG),
    (dict(owners=owners(2, (1 << 12) + 4)), ARG),              # D % 4 == 0: the vector reductions need 16 bytes
    (dict(owners=owners(2, (1 << 12) + 2), D=66), ARG),        # scalar reductions: 4 bytes
])
def test_host_refusals_return_before_any_device_call(h, name, over, code):
    assert getattr(h, name)(*args(**over)) == code
