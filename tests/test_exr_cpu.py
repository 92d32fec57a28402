"""LinearEXRExport mirror: node surface == reference, file naming rules, and the self-contained OpenEXR / Radiance
writers (files read back with OpenCV's OpenEXR codec where it is available)."""
import os

os.environ.setdefault("OPENCV_IO_ENABLE_OPENEXR", "1")      # must be set before cv2 is imported

import numpy as np
import pytest
import torch

from oracle.ref_loader import reference_available
from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS
from vae_decode_hdr_b200.linear_exr_export import (LinearEXRExport, highest_version, write_exr_scanlines,
                                                   write_radiance_hdr)

try:
    import cv2
except Exception:      # pragma: no cover
    cv2 = None


def test_node_surface_equals_reference():
    cls = NODE_CLASS_MAPPINGS["LinearEXRExport"]
    assert cls is LinearEXRExport
    assert (cls.RETURN_TYPES, cls.RETURN_NAMES, cls.FUNCTION, cls.CATEGORY, cls.OUTPUT_NODE) == \
        (("STRING",), ("filepath",), "export_linear_exr", "image", True)


@pytest.mark.skipif(not reference_available(), reason="unmodified reference source not present (HDRVAE_REFERENCE_ROOT)")
def test_node_surface_equals_reference_tree():
    """Same INPUT_TYPES and export_linear_exr() parameters as the unmodified reference class."""
    import importlib.util, inspect, sys, types
    from oracle.ref_loader import REFERENCE_ROOT
    cls = NODE_CLASS_MAPPINGS["LinearEXRExport"]
    for name in ("pyexr", "imageio", "imageio.v3", "folder_paths"):
        sys.modules.setdefault(name, types.ModuleType(name))
    spec = importlib.util.spec_from_file_location("_ref_linear_exr_export",
                                                  os.path.join(REFERENCE_ROOT, "linear_exr_export.py"))
    mod = importlib.util.module_from_spec(spec)
    try:
        spec.loader.exec_module(mod)
    except Exception as e:      # the reference needs cv2 at import time
        pytest.skip(f"reference exporter not importable here: {e}")
    ref = mod.LinearEXRExport
    assert cls.INPUT_TYPES() == ref.INPUT_TYPES()
    assert list(inspect.signature(cls.export_linear_exr).parameters) == list(inspect.signature(ref.export_linear_exr).parameters)


@pytest.mark.skipif(cv2 is None, reason="cv2 not importable")
@pytest.mark.parametrize("dtype", [np.float16, np.float32])
@pytest.mark.parametrize("compression", ["none", "zip"])
def test_exr_writer_reads_back_exactly(tmp_path, dtype, compression):
    rng = np.random.default_rng(3)
    img = (rng.standard_normal((37, 53, 3)) * 4).astype(np.float32)
    img[0, 0] = [70000.0, -70000.0, 1e-9]                       # half overflow -> +-inf, underflow -> 0
    planes = np.ascontiguousarray(img[..., ::-1].transpose(0, 2, 1)).astype(dtype)     # [H, (B,G,R), W]
    path = str(tmp_path / "t.exr")
    write_exr_scanlines(path, planes, compression)
    back = cv2.imread(path, cv2.IMREAD_UNCHANGED)
    if back is None:
        pytest.skip("this OpenCV build has no OpenEXR codec")
    assert back.shape == (37, 53, 3)
    assert np.array_equal(back[..., ::-1], img.astype(dtype).astype(np.float32))


@pytest.mark.skipif(cv2 is None, reason="cv2 not importable")
def test_radiance_writer_reads_back(tmp_path):
    rng = np.random.default_rng(4)
    img = np.abs(rng.standard_normal((9, 11, 3)) * 3).astype(np.float32)
    path = str(tmp_path / "t.hdr")
    write_radiance_hdr(path, img)
    back = cv2.imread(path, cv2.IMREAD_UNCHANGED)
    assert back is not None and back.shape == (9, 11, 3)
    assert np.abs(back[..., ::-1] - img).max() <= img.max() / 128.0      # 8-bit shared-exponent mantissas


def test_filename_rules(tmp_path, monkeypatch):
    """versioning scans for `<prefix>_vN*` (linear_exr_export.py:43-78), batches get `_frame_%0Nd` (:297-299), a
    prefix with a path separator adds sub-folders (:280-287), failures come back as 'ERROR: ...' (:366-369)."""
    # the reference treats any output_path starting with "/" as a sub-folder of ComfyUI's output directory (:268-273), so
    # an absolute path cannot be passed on Linux: use a path relative to the working directory, as SURVEY.md §8f notes
    monkeypatch.chdir(tmp_path)
    d = tmp_path / "out"
    d.mkdir()
    for n in ("shot_v001.exr", "shot_v012_frame_1001.exr", "shot_v3.json", "other_v099.exr"):
        (d / n).write_bytes(b"")
    assert highest_version(str(d), "shot") == 12
    node = LinearEXRExport()
    img = torch.rand(2, 4, 5, 3) * 3
    (p,) = node.export_linear_exr(img, "sub/shot", output_path="out", start_frame=1001, frame_pad=4, versioning=True,
                                  format="exr", bit_depth="32bit", compression="zip", save_workflow=True,
                                  prompt={"a": 1})
    assert os.path.abspath(p) == str(d / "sub" / "shot_v001_frame_1002.exr") and os.path.isfile(p)
    assert os.path.isfile(str(d / "sub" / "shot_v001_frame_1001.exr")) and os.path.isfile(str(d / "sub" / "shot_v001_frame_1001.json"))
    (p2,) = node.export_linear_exr(img[0], "single", output_path="out", versioning=False, format="hdr")
    assert os.path.abspath(p2) == str(d / "single.hdr") and os.path.getsize(p2) > 4 * 5 * 4
    (err,) = node.export_linear_exr(torch.zeros(1, 4, 5, 2), "bad", output_path="out", format="exr")
    assert err.startswith("ERROR: ")
    if not torch.cuda.is_available():      # the half pack is a GPU kernel: without a device the node reports, not falls back
        (err,) = node.export_linear_exr(img, "h", output_path="out", format="exr", bit_depth="16bit")
        assert err.startswith("ERROR: ") and "GPU" in err
