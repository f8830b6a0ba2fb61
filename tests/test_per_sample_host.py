"""Host logic of the per-sample fused losses (reduction="none"): argument validation, the C header constant and the
ctypes table.  No CUDA compute: every refusal below happens before a launch (the inputs are CPU tensors, which a
launch would reject with a different error)."""
import os
import re
import subprocess

import pytest
import torch

from diffnet_b200 import DiffNet2DFEM, DiffNet3DFEM, ops
from diffnet_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "diffnet_fem.h")


def test_consts_accepts_none_and_rejects_unknown():
    assert ops._consts(1.0, 1.0, 1.0, "none").reduction == L.DN_REDUCE_NONE
    assert ops._consts(1.0, 1.0, 1.0, "mean").reduction == 0
    assert ops._consts(1.0, 1.0, 1.0, "sum").reduction == 1
    for bad in ("avg", "None", None, 2):
        with pytest.raises(L.DiffNetFEMError, match="reduction"):
            ops._consts(1.0, 1.0, 1.0, bad)


def test_reduce_none_matches_the_header(tmp_path):
    src = tmp_path / "none.c"
    src.write_text('#include <stdio.h>\n#include "diffnet_fem.h"\nint main(){printf("%d\\n", DN_REDUCE_NONE); return 0;}\n')
    exe = tmp_path / "none"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    assert int(subprocess.run([str(exe)], capture_output=True, text=True).stdout) == L.DN_REDUCE_NONE


def test_new_exports_have_prototypes():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for name in ("dn_scale_per_sample_f32", "dn_fem_residual_reduce_2d_f32", "dn_fem_residual_reduce_3d_f32"):
        assert re.search(rf"\b{name}\s*\(", text), name
        assert name in L.PROTOTYPES, name
    # the reduce variants are the residual signature plus one int
    assert L.PROTOTYPES["dn_fem_residual_reduce_2d_f32"][1][:-1] == L.PROTOTYPES["dn_fem_residual_2d_f32"][1]


def _cpu_inputs(nsd):
    shape = (2, 1, 8, 8) if nsd == 2 else (2, 1, 6, 6, 6)
    return torch.randn(shape), (DiffNet2DFEM(None, domain_size=8) if nsd == 2 else DiffNet3DFEM(None, domain_size=6))


@pytest.mark.parametrize("nsd", [2, 3])
def test_none_refuses_what_splits_a_sample_before_any_launch(nsd):
    u, fem = _cpu_inputs(nsd)
    geom = fem.geometry
    cases = [
        lambda: ops.fem_energy(geom, u, reduction="none", z_own=(1, 3)),
        lambda: ops.fem_energy(geom, u, reduction="none", mean_count=10.0),
        lambda: ops.energy_raw(geom, u, reduction="none", z_own=(1, 3)),
        lambda: ops.energy_raw(geom, u, reduction="none", mean_count=10.0),
        lambda: ops.PreparedEnergy(geom, u, reduction="none", mean_count=10.0),
        lambda: ops.PreparedEnergy(geom, u, reduction="none", link=L.dn_slab_link()),
        lambda: ops.energy_input_grads_raw(geom, u, f=u, reduction="none", mean_count=10.0, want_f=True),
    ]
    for i, call in enumerate(cases):
        with pytest.raises(L.DiffNetFEMError, match="reduction='none'"):
            call()


def test_residual_reduction_validated_before_any_launch():
    u, fem = _cpu_inputs(2)
    for bad in ("mean", "avg"):
        with pytest.raises(L.DiffNetFEMError, match="residual reduction"):
            fem.residual_loss(u, reduction=bad)
        with pytest.raises(L.DiffNetFEMError, match="residual reduction"):
            ops.residual_raw(fem.geometry, u, reduction=bad)


def test_per_sample_gradient_views():
    """reduction="none" asks for a gradient per sample of a field shared by the batch: _per_sample materialises it."""
    t = torch.randn(1, 5, 7)
    assert ops._per_sample(t, 4) is t
    e = ops._per_sample(t, 4, expand=True)
    assert e.shape == (4, 5, 7) and e.is_contiguous() and torch.equal(e[3], t[0])
