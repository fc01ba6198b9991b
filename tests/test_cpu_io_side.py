"""CPU: frame I/O side (SURVEY 8 row f.3): the oracle restatement of MultiRestrictSize + MultiToTensor + _save_mask against the
fixture produced by the REAL reference (oracle/gen_golden.py --only io), the product's size rule / palette / mask writer."""
import io
import os

import numpy as np
import pytest
import torch

from oracle import io_side as IO


@pytest.fixture(scope="module")
def fx(golden_dir):
    return torch.load(os.path.join(golden_dir, "io_side.pt"))


def test_oracle_preprocess_vs_reference_fixture(fx):
    img = fx["img"].numpy()
    for name, c in fx["cases"].items():
        kw, k = c["kw"], 0
        for sc in kw["multi_scale"]:
            for fl in ((False, True) if kw["flip"] else (False,)):
                mine = IO.preprocess(img, kw["max_short_edge"], kw["max_long_edge"], sc, kw["align_corners"], 16, fl)
                assert tuple(mine.shape) == tuple(c["ref"][k].shape), name
                assert (mine - c["ref"][k]).abs().max().item() < 2e-5, name      # fp32 summation order of cv2's SIMD passes
                k += 1


def test_cubic_restatement_vs_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (61, 83, 3)).astype(np.float32)
    for (Ho, Wo) in ((97, 129), (33, 49), (61, 100)):
        ref = cv2.resize(img, dsize=(Wo, Ho), interpolation=cv2.INTER_CUBIC)
        assert np.abs(ref - IO.resize_cubic(img, Ho, Wo)).max() < 1e-3               # on a 0..255 scale


def test_product_size_rule_and_palette_match_the_restatement():
    from aot_benchmark_b200.io_side import FramePreprocessor, davis_palette
    assert davis_palette() == IO.davis_palette()
    for args in ((None, 800, True), (480, 800 * 1.3, False), (None, 1040, False)):
        fp = FramePreprocessor(args[0], args[1], False, [1.0], args[2], device="cpu")
        for (h, w) in ((480, 854), (720, 1280), (1080, 1920), (360, 640), (854, 480)):
            for sc in (1.0, 1.3, 0.75):
                assert fp.target_size(h, w, sc) == IO.restrict_size(h, w, args[0], args[1], sc, args[2], 16)


def test_async_mask_writer_png_equals_reference(fx, tmp_path):
    """AsyncMaskWriter on CPU tensors (no device needed for the host half): same pixels and palette as the reference's
    _save_mask output stored in the fixture, with and without the id remap."""
    from PIL import Image
    from aot_benchmark_b200.io_side import AsyncMaskWriter
    wr = AsyncMaskWriter(workers=2, ring=2)
    mask = fx["mask"]
    wr.save(mask.float().view(1, 1, *mask.shape), str(tmp_path / "a.png"))
    wr.save(mask.float(), str(tmp_path / "b.png"), squeeze_idx=fx["squeeze_idx"])
    wr.save(mask.float(), str(tmp_path / "c.png"))                                    # ring wrap-around
    wr.close()
    for mine, ref in (("a.png", "png_plain"), ("b.png", "png_squeezed"), ("c.png", "png_plain")):
        a, b = Image.open(tmp_path / mine), Image.open(io.BytesIO(fx[ref]))
        assert a.mode == b.mode == "P"
        assert np.array_equal(np.array(a), np.array(b))
        assert a.getpalette() == b.getpalette()


def test_palette_equals_the_reference_table(golden_dir):
    from oracle.fixtures import load_reference_contract
    assert IO.davis_palette() == load_reference_contract(golden_dir)["palette"]
