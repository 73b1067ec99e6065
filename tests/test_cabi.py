"""CPU: the C-ABI library builds for sm_100a, loads, and exports every symbol include/bcosk.h declares.
No compute call is made here (there is no GPU); product entry points must refuse to run without one."""
import ctypes
import re

import pytest
import torch

from bcos_b200 import _lib as L


def test_library_exports_every_declared_symbol(bcosk_lib):
    with open(L.HEADER) as fh:
        src = fh.read()
    declared = set(re.findall(r"\b(bcosk_[a-z0-9_]+)\s*\(", src))
    declared.discard("bcosk_igemm_params")
    assert len(declared) >= 16
    for name in sorted(declared):
        assert hasattr(bcosk_lib, name), f"libbcosk.so lacks {name}"
    assert bcosk_lib.bcosk_version() >= 100


def test_struct_layout_matches_header(bcosk_lib):
    assert bcosk_lib.bcosk_sizeof_igemm_params() == ctypes.sizeof(L.IgemmParams)
    names = [f[0] for f in L.IgemmParams._fields_]
    for must in ("a", "b", "y", "inv_norm", "tap_off_w", "seg_a_choff", "mask2", "os_q"):
        assert must in names


def test_bad_arguments_are_rejected_without_touching_a_device(bcosk_lib):
    p = L.IgemmParams()
    rc = bcosk_lib.bcosk_igemm(ctypes.byref(p), None)
    assert rc == L.BCOSK_EINVAL
    assert b"null" in bcosk_lib.bcosk_last_error()
    assert bcosk_lib.bcosk_igemm(None, None) == L.BCOSK_EINVAL


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only check")
def test_product_fails_loudly_without_gpu(bcosk_lib):
    from bcos_b200.engine import ResNetPlan
    from bcos_b200.models import resnet_state_shapes
    from bcos_b200.utils import synth
    with pytest.raises(L.BcoskError):
        L.require_device()
    plan = ResNetPlan("resnet18", synth.synth_state_dict(resnet_state_shapes("resnet18")), 1, device="cpu", image_size=32)
    with pytest.raises(L.BcoskError):
        plan.explain(torch.zeros(1, 6, 32, 32))


def test_odd_image_sizes_are_rejected_before_any_launch(bcosk_lib):
    """The space-to-depth kernels (input_prep_s2d, contrib_map_s2d) cover the image in 2x2 blocks with float2 stores: an odd
    height or width must be refused on the host (host buffers stand in for the operands; nothing may touch them)."""
    f6 = (ctypes.c_float * 6)(*([1.0] * 6))
    x = torch.zeros(6 * 9 * 9)
    u8 = torch.zeros(3 * 9 * 9, dtype=torch.uint8)
    g = torch.zeros(5 * 5 * 32)
    cmap = torch.zeros(9 * 9)
    p = ctypes.c_void_p
    for h, w in ((9, 8), (8, 9), (9, 9), (1, 2)):
        for fn, src in ((bcosk_lib.bcosk_contrib_map_s2d, x), (bcosk_lib.bcosk_contrib_map_s2d_u8, u8)):
            rc = fn(p(g.data_ptr()), p(src.data_ptr()), 1, h, w, 32, f6, ctypes.c_float(1.0), p(cmap.data_ptr()), None, None)
            assert rc == L.BCOSK_EINVAL, (h, w, rc)
            assert b"even" in bcosk_lib.bcosk_last_error()
        rc = bcosk_lib.bcosk_input_prep_s2d(p(x.data_ptr()), 1, h, w, f6, f6, p(g.data_ptr()), 32, 1, L.DTYPE_CODE["fp16"], None, 0, 0, None)
        assert rc == L.BCOSK_EINVAL, (h, w, rc)
    assert torch.equal(cmap, torch.zeros_like(cmap)) and torch.equal(g, torch.zeros_like(g))


def test_gap_logits_rejects_empty_shapes(bcosk_lib):
    buf = torch.zeros(16)
    p = ctypes.c_void_p(buf.data_ptr())
    for nb, npix, ncls in ((0, 49, 10), (1, 0, 10), (1, 49, 0)):
        rc = bcosk_lib.bcosk_gap_logits(p, nb, npix, ncls, ctypes.c_float(1.0), ctypes.c_float(0.0), p, None, None)
        assert rc == L.BCOSK_EINVAL, (nb, npix, ncls, rc)


@pytest.mark.parametrize("bad", [-1, 10, 1 << 20])
def test_explain_targets_rejects_out_of_range_class_before_launch(bcosk_lib, bad):
    """explain_targets copies the class indices to the seed kernel, which reads the classifier's weight row of each: an index
    outside [0, ncls) is refused with ValueError before any launch (the plan here lives on the host and could launch nothing)."""
    from bcos_b200.engine import ResNetPlan
    from bcos_b200.models import resnet_state_shapes
    from bcos_b200.utils import synth
    plan = ResNetPlan("resnet18", synth.synth_state_dict(resnet_state_shapes("resnet18", num_classes=10)), 2, device="cpu",
                      image_size=32)
    with pytest.raises(ValueError, match="targets"):
        plan.explain_targets(None, torch.tensor([[0, bad]]))
    with pytest.raises(ValueError, match="targets"):
        plan.explain_targets(None, torch.tensor([bad, 3]))
