"""Feature buffers without a GPU: the host model's Philox against the Random123 known answers, the PFM writer, and the
frame program's --aov option."""
import subprocess

import numpy as np
import pytest

import aov_model as am
from test_frames_and_checkpoints import RENDER_BIN


def test_model_philox_matches_the_random123_known_answers():
    # the three vectors test_philox_known_answers checks the GPU's Philox4x32-10 against: (counter[4], key[2]) -> out[4]
    kat = [([0, 0, 0, 0, 0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
           ([0xffffffff] * 6, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
           ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, 0xa4093822, 0x299f31d0], [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])]
    for inp, want in kat:
        assert [int(w) for w in am.philox4x32_10(*inp)] == want


def test_model_variates_stay_in_range():
    x = np.array([0, 1, 0xFF, 0x100, 0xFFFFFFFF], dtype=np.uint32)
    u = am.u01(x)
    assert u.dtype == np.float32 and u[0] == 0 and u[3] == np.float32(2.0**-24) and u[4] < 1
    g = am.gen_range(x, 0.25, 0.5)
    assert g.dtype == np.float32 and (g >= np.float32(0.25)).all() and (g < np.float32(0.5)).all()


@pytest.mark.parametrize("channels", [3, 1])
def test_write_pfm_round_trip(vb, tmp_path, channels):
    H, W = 5, 7
    rng = np.random.default_rng(3)
    plane = rng.standard_normal((H, W, channels) if channels == 3 else (H, W)).astype(np.float32)
    plane.flat[0] = np.inf  # depth of a pixel no sample hit
    path = tmp_path / "p.pfm"
    vb.write_pfm(str(path), plane)
    raw = path.read_bytes()
    header = (b"PF" if channels == 3 else b"Pf") + b"\n7 5\n-1.0\n"
    assert raw.startswith(header)  # negative scale: little-endian
    body = np.frombuffer(raw[len(header):], dtype="<f4")
    assert body.size == plane.size
    # rows bottom-to-top in the file, the planes' own order: row 0 first, nothing flipped
    assert np.array_equal(body.view(np.uint32), plane.reshape(-1).view(np.uint32))
    assert np.array_equal(body.reshape(plane.shape)[0], plane[0])


def test_write_pfm_refuses_bad_arguments(vb, tmp_path):
    with pytest.raises(ValueError):
        vb.write_pfm(str(tmp_path / "x.pfm"), np.zeros((4, 4, 2), dtype=np.float32))
    with pytest.raises(vb.VecchioError):
        vb.write_pfm(str(tmp_path / "no_such_dir" / "x.pfm"), np.zeros((4, 4), dtype=np.float32))


@pytest.mark.parametrize("args", [["--aov"], ["--aov", "0"], ["--aov", "65537"], ["--aov", "x"]])
def test_program_refuses_aov_without_a_sample_count(args):
    r = subprocess.run([RENDER_BIN, *args], capture_output=True, text=True)
    assert r.returncode == 2 and "--aov needs" in r.stderr, r.stderr


def test_program_documents_aov():
    r = subprocess.run([RENDER_BIN, "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--aov N" in r.stdout and "albedo_NNNN.pfm" in r.stdout
