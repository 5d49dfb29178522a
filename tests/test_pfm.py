"""The Portable Float Map writer of the host library (rtnw_host_write_pfm, rtnw.write_pfm): the files the driver's --aov
writes.  CPU only."""
import numpy as np
import pytest


def read_pfm(path):
    """(header lines, float32 array of shape (ny, nx[, 3]) in file order: the first row of the file is row 0)"""
    raw = open(path, "rb").read()
    lines, at = [], 0
    for _ in range(3):
        end = raw.index(b"\n", at)
        lines.append(raw[at:end].decode())
        at = end + 1
    nx, ny = map(int, lines[1].split())
    channels = 3 if lines[0] == "PF" else 1
    data = np.frombuffer(raw[at:], dtype="<f4")
    assert data.size == nx * ny * channels
    return lines, data.reshape((ny, nx, 3) if channels == 3 else (ny, nx))


@pytest.mark.parametrize("shape, magic", [((3, 4, 3), "PF"), ((3, 4), "Pf")])
def test_pfm_is_byte_exact_with_the_bottom_row_first(rtnw, tmp_path, shape, magic):
    a = (np.arange(np.prod(shape), dtype=np.float32) * np.float32(0.37) - 1.5).reshape(shape)
    a.flat[5] = np.float32(1e-30)
    path = tmp_path / "img.pfm"
    rtnw.write_pfm(path, a)
    want = f"{magic}\n4 3\n-1.0\n".encode() + a.astype("<f4").tobytes()  # row 0 (the library's j = 0, the bottom) first
    assert path.read_bytes() == want
    lines, back = read_pfm(path)
    assert lines == [magic, "4 3", "-1.0"]
    assert np.array_equal(back.view(np.uint32), a.view(np.uint32))


def test_pfm_refuses_other_channel_counts(rtnw, tmp_path):
    with pytest.raises(rtnw.RtnwError) as e:
        rtnw.write_pfm(tmp_path / "two.pfm", np.zeros((2, 2, 2), np.float32))
    assert e.value.code == rtnw.RTNW_ERR_INVALID
    assert not (tmp_path / "two.pfm").exists()
