"""Step kernel without a grid barrier: pass 2 waits per utterance tile for that tile's row sums, and the CTA that
completes a tile closes its rows.  The per-tile counters must be zero again after every call (a replayed graph
never sees last step's counts) and every step of a captured graph must equal an eager step on the same batch."""
import pytest
import torch

from oracle import ge2e_oracle as orc
from oracle import ge2e_oracle_torch as orct

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SHAPES = [(1024, 10, 256), (1000, 10, 256), (129, 10, 256)]   # cfg3, a partial last utterance tile, smallest TC shape


@pytest.fixture(scope="module")
def pkg():
    import speaker_embedding_ge2e_loss_b200 as p
    p.lib()
    assert torch.cuda.is_available()
    return p


def trel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def bookkeeping(plan, N, M):
    """workspace header (step counters) and the per-utterance-tile counters behind it"""
    ot = -(-N * M // 128)
    return plan._ws[:256 + 4 * ot]


@pytest.mark.parametrize("N,M,D", SHAPES)
def test_workspace_counters_left_zero(pkg, N, M, D):
    plan = pkg.GE2EPlan(N, M, D, "softmax", "tf32", device=DEV)
    assert plan.path == 1
    E = torch.tensor(orc.make_embeddings(N, M, D, seed=3, kind="clustered"), device=DEV)
    w, b = torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV)
    plan.step(E, w, b)
    torch.cuda.synchronize()
    assert int(bookkeeping(plan, N, M).count_nonzero()) == 0
    g = plan.capture(E, w, b, steps=20)
    g.replay()
    torch.cuda.synchronize()
    assert int(bookkeeping(plan, N, M).count_nonzero()) == 0


@pytest.mark.parametrize("N,M,D", SHAPES)
def test_captured_steps_match_eager_and_oracle(pkg, N, M, D):
    nb, steps = 4, 20
    batches = [torch.tensor(orc.make_embeddings(N, M, D, seed=40 + i, kind="clustered" if i % 2 else "random"),
                            device=DEV) for i in range(nb)]
    w, b = torch.tensor(10.0, device=DEV), torch.tensor(-5.0, device=DEV)
    plan = pkg.GE2EPlan(N, M, D, "softmax", "tf32", device=DEV)
    eager = []
    for E in batches:
        plan.step(E, w, b)
        torch.cuda.synchronize()
        eager.append((plan._accum[:3].clone(), plan.dE.clone()))
    scal = torch.zeros(steps, 3, device=DEV)
    dEs = torch.zeros(steps, N, M, D, device=DEV)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        for k in range(steps):
            plan.step(batches[k % nb], w, b)
            scal[k].copy_(plan._accum[:3])
            dEs[k].copy_(plan.dE)
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    for k in range(steps):
        ref_s, ref_dE = eager[k % nb]
        got = scal[k].double().cpu()
        ref = ref_s.double().cpu()
        assert abs(got[0] - ref[0]) <= 1e-5 * max(1.0, abs(ref[0])), (k, got, ref)
        assert abs(got[1] - ref[1]) <= 1e-4 * max(1.0, abs(ref[1])), (k, got, ref)
        assert abs(got[2] - ref[2]) <= 1e-4 * max(1.0, abs(ref[2])), (k, got, ref)
        assert trel(dEs[k], ref_dE) <= 1e-4, k
    for i, E in enumerate(batches):
        ref = orct.forward_backward(E, 10.0, -5.0, 1e-6, "softmax")
        s = scal[i].double().cpu()
        assert abs(s[0] - ref["loss"]) <= 2e-3 * max(1.0, abs(ref["loss"]))
        assert trel(dEs[i].reshape(-1), ref["dE"].reshape(-1)) <= 2e-3
        assert abs(s[1] - ref["dw"]) <= 2e-3 * max(1.0, abs(ref["dw"]))
        assert abs(s[2] - ref["db"]) <= 1e-5 * N * M
