"""The host side of environment lighting (no GPU): the rt_environment struct of the ABI and the mirror's PFM reader,
which loads the maps of `rtow_b200 --env`."""
import ctypes as C

import numpy as np
import pytest

from raytracingoneweekendapplication_b200 import capi


def test_environment_struct_size(built):
    lib = capi.load()
    assert lib.rt_struct_size(17) == C.sizeof(capi.rt_environment) == 88
    assert "rt_set_environment" in capi.EXPORTED_SYMBOLS


def _write_pfm(path, rgb, little):
    """An independent PFM writer: the scale's sign names the byte order, rows are stored bottom-up."""
    h, w, _ = rgb.shape
    dt = np.dtype("<f4" if little else ">f4")
    with open(path, "wb") as f:
        f.write(f"PF\n{w} {h}\n{-1.0 if little else 1.0}\n".encode())
        f.write(np.ascontiguousarray(rgb[::-1]).astype(dt).tobytes())


def _read_pfm(path):
    s = capi.load_scenes()
    w, h = C.c_int(), C.c_int()
    assert s.rtsc_read_pfm(str(path).encode(), C.byref(w), C.byref(h), None, 0) == 2
    out = np.empty((h.value, w.value, 3), dtype=np.float32)
    assert s.rtsc_read_pfm(str(path).encode(), C.byref(w), C.byref(h), out.ctypes.data, out.size) == 0
    return out


@pytest.mark.parametrize("little", [True, False])
def test_read_pfm_is_bit_exact(built, tmp_path, little):
    rng = np.random.default_rng(7)
    rgb = (rng.standard_normal((5, 7, 3)) * 1e3).astype(np.float32)
    rgb[0, 0] = [0.0, np.float32(1e-40), np.float32(3.4e38)]  # a denormal and a value near the top of the range
    rgb[4, 6] = [-0.0, 1.0, np.inf]
    p = tmp_path / "m.pfm"
    _write_pfm(p, rgb, little)
    got = _read_pfm(p)
    assert np.array_equal(got.view(np.uint32), rgb.view(np.uint32))


def test_read_pfm_refuses_other_files(built, tmp_path):
    s = capi.load_scenes()
    w, h = C.c_int(), C.c_int()
    bad = {"grey.pfm": b"Pf\n2 2\n-1.0\n" + bytes(16), "short.pfm": b"PF\n4 4\n-1.0\n" + bytes(40),
           "zero.pfm": b"PF\n0 4\n-1.0\n", "text.pfm": b"P3\n1 1\n255\n0 0 0\n"}
    for name, data in bad.items():
        (tmp_path / name).write_bytes(data)
        assert s.rtsc_read_pfm(str(tmp_path / name).encode(), C.byref(w), C.byref(h), None, 0) == 1, name
    assert s.rtsc_read_pfm(str(tmp_path / "missing.pfm").encode(), C.byref(w), C.byref(h), None, 0) == 1
