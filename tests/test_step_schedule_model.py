"""Host model behind the step kernel's pass-2 schedule (no GPU): pass 2 of a cluster waits per utterance tile for
that tile's row sums instead of at a grid barrier, and walks its range so that late tiles come last."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def pkg():
    from speaker_embedding_ge2e_loss_b200 import build
    build.build()   # nvcc cross-compiles sm_100a without a GPU
    import speaker_embedding_ge2e_loss_b200 as p
    return p

SHAPES = [(10240, 1024), (131072, 8192), (16384, 8192), (4096, 2048), (2100, 300), (256, 8192), (300 * 7, 300),
          (65536, 256), (1024, 1024), (10000, 1000), (1290, 129)]


def _model(h, u_local, n_total, cg, max_cl):
    de = (C.c_int * (max_cl + 1))()
    dc = (C.c_int * (max_cl + 1))()
    part = (C.c_int * 2)()
    units = (C.c_int * 4)()
    nc = h.ge2e_b200_debug_step_schedule(u_local, n_total, cg, max_cl, de, dc, part, units)
    rot = (C.c_int * max_cl)()
    fin = (C.c_double * max_cl)()
    model = (C.c_double * 2)()
    assert h.ge2e_b200_debug_step_model(u_local, n_total, cg, max_cl, rot, fin, model) == nc
    return nc, list(de)[:nc + 1], list(dc)[:nc + 1], list(units), list(rot)[:nc], list(fin)[:nc], list(model)


@pytest.mark.parametrize("u_local,n_total", SHAPES)
@pytest.mark.parametrize("cg,max_cl", [(2, 74), (1, 148), (2, 8), (1, 3)])
def test_pass2_walk_covers_its_range_once(pkg, u_local, n_total, cg, max_cl):
    nc, de, dc, units, rot, fin, model = _model(pkg.lib(), u_local, n_total, cg, max_cl)
    ogc, stc = units[2], units[3]
    seen = []
    for c in range(nc):
        a, b = dc[c], dc[c + 1]
        n = b - a
        if rot[c]:
            assert 0 < rot[c] < n and a // stc == (b - 1) // stc, "a rotated range lies in one owner group"
        order = [a + (i + rot[c]) % n for i in range(n)] if n else []
        assert sorted(order) == list(range(a, b))
        seen += order
    assert sorted(seen) == list(range(ogc * stc))


@pytest.mark.parametrize("u_local,n_total", SHAPES)
@pytest.mark.parametrize("cg,max_cl", [(2, 74), (1, 148), (2, 8), (1, 3)])
def test_model_never_worse_than_the_barrier(pkg, u_local, n_total, cg, max_cl):
    nc, de, dc, units, rot, fin, model = _model(pkg.lib(), u_local, n_total, cg, max_cl)
    x, barrier = model
    assert max(fin) <= barrier + 1e-9, (max(fin), barrier)


def test_cfg3_makespan_near_the_average(pkg):
    """cfg3 (N = 1024, M = 10) on 74 CTA pairs: 320 + 320 units, 8.65 per cluster on average; the barrier version
    finished at 8 + 5 = 13."""
    nc, de, dc, units, rot, fin, model = _model(pkg.lib(), 10240, 1024, 2, 74)
    x, barrier = model
    total = units[0] * units[1] + units[2] * units[3]
    assert nc == 74 and total == 640
    assert max(fin) <= total / nc + x + 1, (max(fin), x)
    assert barrier >= 13


def test_model_refuses_bad_arguments(pkg):
    h = pkg.lib()
    rot = (C.c_int * 8)()
    fin = (C.c_double * 8)()
    model = (C.c_double * 2)()
    assert h.ge2e_b200_debug_step_model(0, 1024, 2, 8, rot, fin, model) < 0
    assert h.ge2e_b200_debug_step_model(10240, 1024, 3, 8, rot, fin, model) < 0
    assert h.ge2e_b200_debug_step_model(10240, 1024, 2, 8, None, fin, model) < 0
