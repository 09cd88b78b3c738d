"""Image objective of the training step (Trainer.calc_dr_loss): this repo's L1Loss / IouLoss against the reference's
own classes (tests/golden/reference/dr_loss.npz, minted by tests/golden/make_golden_dr_loss.py), the C ABI mirror of
the fused op, and its argument checks."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from dss_b200 import _lib
from dss_b200.training import IouLoss, L1Loss, dr_image_loss
from dss_b200.training.losses import eps_denom
from tests.golden.make_golden_dr_loss import calc_dr_loss

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference", "dr_loss.npz")
CASES = ["binary", "soft", "empty_views", "no_overlap", "exact"]


def golden(name):
    z = np.load(GOLDEN)
    return {k.split("/", 1)[1]: z[k] for k in z.files if k.startswith(name + "/")}


def restated(case):
    """calc_dr_loss in float64 on this repo's L1Loss and IouLoss: (terms, d loss / d image)"""
    lr, ls, iw = case["weights"]
    assert iw == 0.01
    return calc_dr_loss(L1Loss, IouLoss, case["image"], case["img"], case["mask"], lr, ls)


@pytest.mark.parametrize("name", CASES)
def test_repo_losses_reproduce_the_reference_objective(name):
    case = golden(name)
    terms, grad = restated(case)
    np.testing.assert_allclose(terms, case["terms"], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(grad, case["grad"], rtol=1e-12, atol=1e-12 * np.abs(case["grad"]).max())


def test_golden_covers_the_edge_cases():
    image, mask = golden("empty_views")["image"], golden("empty_views")["mask"]
    assert mask[0].sum() == 0 and image[1, ..., 3].sum() == 0            # empty GT, empty prediction
    assert 0 < mask[3].sum() < 1e-17 and image[3, ..., 3].sum() == 0    # union below eps_denom's clamp
    nov = golden("no_overlap")
    assert ((nov["mask"][:, 0] != 0) & (nov["image"][..., 3] != 0)).sum() == 0 and nov["terms"][1] == 0
    assert (nov["grad"][..., :3] == 0).all()
    ex = golden("exact")
    assert (np.moveaxis(ex["img"], 1, -1) == ex["image"][..., :3]).any()
    soft = golden("soft")["mask"]
    assert ((soft > 0) & (soft < 1)).any()


def test_iou_loss_semantics():
    """IouLoss(reduction, channel_dim) of losses.py:498-514: per batch element over dims 1.., then the reduction."""
    g = torch.Generator().manual_seed(3)
    a, b = torch.rand(4, 5, 6, generator=g, dtype=torch.float64), torch.rand(4, 5, 6, generator=g, dtype=torch.float64)
    want = 1 - (a * b).sum((1, 2)) / (a + b - a * b).sum((1, 2))
    torch.testing.assert_close(IouLoss(reduction="none", channel_dim=None)(a, b), want)
    torch.testing.assert_close(IouLoss(reduction="mean", channel_dim=None)(a, b), want.mean())
    torch.testing.assert_close(IouLoss()(a, b), want.sum())      # default channel_dim=-1 sums the (N,) result first
    z = torch.zeros(2, 3, dtype=torch.float64)
    assert torch.equal(IouLoss(reduction="none", channel_dim=None)(z, z), 1 - z.sum(1) / eps_denom(z.sum(1)))


def test_dr_loss_args_struct_layout_matches_c():
    """compile a tiny C program against the header and compare sizeof/offsetof with the ctypes mirror."""
    fields = [f[0] for f in _lib.DrLossArgs._fields_]
    body = "".join('printf("%s %%zu\\n", offsetof(dss_dr_loss_args, %s));\n' % (f, f) for f in fields)
    src = ('#include <stddef.h>\n#include <stdio.h>\n#include "dss_b200.h"\nint main(){'
           'printf("size %%zu\\n", sizeof(dss_dr_loss_args));\n'
           'printf("blocks %%d\\n", DSS_DR_LOSS_BLOCKS_PER_VIEW);\nprintf("num_sums %%d\\n", DSS_DR_LOSS_NUM_SUMS);\n'
           '%s return 0;}' % body)
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "t.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "t")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        out = dict(l.split() for l in subprocess.check_output([exe], text=True).strip().splitlines())
    assert int(out["size"]) == C.sizeof(_lib.DrLossArgs)
    assert int(out["blocks"]) == _lib.DR_LOSS_BLOCKS_PER_VIEW and int(out["num_sums"]) == _lib.DR_LOSS_NUM_SUMS
    for f in fields:
        assert int(out[f]) == getattr(_lib.DrLossArgs, f).offset, f


def test_dr_image_loss_refuses_cpu_tensors():
    case = golden("binary")
    image, img, mask = (torch.from_numpy(case[k]) for k in ("image", "img", "mask"))
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        dr_image_loss(image, img, mask)
