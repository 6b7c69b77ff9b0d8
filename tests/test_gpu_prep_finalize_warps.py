"""The register-resident prep / finalize kernels at D = 256 run two warps per speaker, two speakers per block:
with an odd speaker count the last block holds one speaker and one pair of warps that return at once.  Every
operand precision those kernels write (fp32, TF32-rounded, split fp16 planes, one fp16 plane), the contrast
variant, and the fused row index, against the float64 oracles."""
import pytest
import torch

from oracle import ge2e_oracle as orc
from test_gpu_edges import DEV, TOL, check, pkg, reference, run_and_check, run_unperm  # noqa: F401

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("N,precision,path", [(7, "fp32", 0), (129, "tf32", 1), (129, "fp32", 2), (129, "f16", 3)])
def test_odd_speaker_count(pkg, N, precision, path):
    plan = run_and_check(pkg, N, 10, 256, precision=precision)
    assert plan.path == path and not plan.single_kernel


# The contrast loss takes a hard arg-max over the negatives: on these clustered speakers TF32 / fp16 operands move
# it for some rows (dE then differs from float64 by ~2e-2 on any build), so the variant is checked in fp32.
@pytest.mark.parametrize("N", [7, 129])
def test_odd_speaker_count_contrast(pkg, N):
    plan = run_and_check(pkg, N, 10, 256, precision="fp32", variant="contrast")
    assert plan.path == 0 and not plan.single_kernel


@pytest.mark.parametrize("N,precision", [(7, "fp32"), (129, "tf32")])
def test_odd_speaker_count_unperm(pkg, N, precision):
    E_np = orc.make_embeddings(N, 10, 256, seed=N, kind="clustered")
    E = torch.tensor(E_np, device=DEV)
    got = run_unperm(pkg, E, 10.0, -5.0, precision, "softmax")
    check(got, reference(E_np, 10.0, -5.0, "softmax"), N * 10, TOL[precision])
