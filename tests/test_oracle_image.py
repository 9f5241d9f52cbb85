"""Output side (main.cpp:100-102 mean, Image/Image.cpp:14-55 write_ppm / write_pfm): the oracle's restatement against files
the reference's own sp::write produced (tests/golden/image_pack.npz, made by tests/golden/make_golden_image.py)."""
import numpy as np

from conftest import GOLDEN


def golden():
    z = np.load(GOLDEN / "image_pack.npz")
    return z["sums"], int(z["spp"]), z["pfm"], z["ppm"]


def test_oracle_pfm_payload_is_the_reference_file(oracle_port):
    sums, spp, pfm, _ = golden()
    assert oracle_port.pack_image(sums, spp, 0).tobytes() == pfm.tobytes()


def test_oracle_ppm_numbers_are_the_reference_file(oracle_port):
    """Exact: the oracle calls the same libm powf as the reference's std::pow(float, float).  Numbers above 65535 (radiance
    beyond ~5e5) saturate in the uint16 the packed format uses; the file itself prints them in full."""
    sums, spp, _, ppm = golden()
    got = oracle_port.pack_image(sums, spp, 1).astype(np.int64)
    assert np.array_equal(got, np.minimum(ppm, 65535))
    assert (ppm > 255).any() and (ppm > 65535).any() and (ppm == 0).any()


def test_oracle_image_on_live_reference(oracle_port, tmp_path):
    import pytest
    from oracle import ref
    import imagecases
    if not ref.available():
        pytest.skip("reference library not built (needs the reference sources: SP_REFERENCE, or a checkout named reference beside the repository)")
    sums, spp = imagecases.sums(seed=5, w=33, h=17, spp=64)
    ref.write_image(sums, spp, tmp_path / "a.pfm")
    ref.write_image(sums, spp, tmp_path / "a.ppm")
    assert oracle_port.pack_image(sums, spp, 0).tobytes() == imagecases.read_pfm_payload(tmp_path / "a.pfm").tobytes()
    assert np.array_equal(oracle_port.pack_image(sums, spp, 1).astype(np.int64),
                          np.minimum(imagecases.read_ppm_numbers(tmp_path / "a.ppm"), 65535))
