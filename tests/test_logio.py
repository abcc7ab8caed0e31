"""Host side of the replay driver (SURVEY 8f N1): the reference's text-log formats (A.7) and the bounded IMU buffer of
FILTER::SetImuData (filter.cpp:50-54).  CPU only."""
import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("imu", "image", "corners", "fusion")


def test_writer_reproduces_logged_lines():
    """the first lines of all eight bundled logs, kept verbatim in tests/golden/log_heads.json: parse -> format == text"""
    from fbus_ekf_b200 import logio
    heads = json.load(open(os.path.join(ROOT, "tests", "golden", "log_heads.json")))
    assert len(heads) == 8
    for key, lines in heads.items():
        kind = key.split("_")[1]
        for line in lines:
            row = [float(x) for x in line.split()]
            assert len(row) in logio.COLUMNS[kind]
            assert logio.format_row(row, logio._ID_COLUMN[kind]) == line, key


@pytest.mark.parametrize("name", ["land", "water"])
def test_round_trip_of_the_parsed_logs(golden, name, tmp_path):
    """write -> read gives back the parsed logs exactly (they hold 6-significant-digit values), with LF and CRLF line ends"""
    from fbus_ekf_b200 import logio
    for kind in KINDS:
        rows = golden[f"{name}_{kind}"][:3000]
        for nl in ("\n", "\r\n"):
            p = tmp_path / f"{kind}.txt"
            logio.write_log(str(p), rows, kind, newline=nl)
            back = logio.read_log(str(p), kind)
            assert back.shape == rows.shape and np.array_equal(back, rows), (name, kind)
    ds = logio.read_dataset(str(tmp_path))
    assert sorted(ds) == sorted(KINDS)
    # appending mirrors the reference's std::ios::app recording
    logio.write_log(str(tmp_path / "imu.txt"), golden[f"{name}_imu"][3000:3010], "imu", newline="\r\n", append=True)
    assert logio.read_imu_log(str(tmp_path / "imu.txt")).shape == (3010, 7)


def test_byte_exact_against_the_reference_files(tmp_path):
    """read -> write with CRLF line ends (as the bundled logs are stored) gives back the reference's files byte for byte; on
    the first lines of all eight logs, kept verbatim in tests/golden/log_heads.json"""
    from fbus_ekf_b200 import logio
    heads = json.load(open(os.path.join(ROOT, "tests", "golden", "log_heads.json")))
    for key, lines in heads.items():
        kind = key.split("_")[1]
        src = tmp_path / f"{key}.txt"
        src.write_bytes("".join(line + "\r\n" for line in lines).encode())
        out = tmp_path / "x.txt"
        logio.write_log(str(out), logio.read_log(str(src), kind), kind, newline="\r\n")
        assert src.read_bytes() == out.read_bytes(), key


def test_bad_logs_are_rejected(tmp_path):
    from fbus_ekf_b200 import logio
    p = tmp_path / "imu.txt"
    p.write_text("1 2 3\n4 5 6\n")
    with pytest.raises(ValueError):
        logio.read_imu_log(str(p))
    with pytest.raises(ValueError):
        logio.read_log(str(p), "nonsense")
    with pytest.raises(ValueError):
        logio.write_log(str(p), np.zeros((2, 5)), "fusion")
    p.write_text("")
    assert logio.read_imu_log(str(p)).shape == (0, 7)


def _simulate_buffer(t_imu, t_frames, start, cap, drop):
    """literal restatement of SetImuData's push / erase (filter.cpp:36-54) and of the per-frame erase (filter.cpp:493-520)"""
    keep = np.zeros(len(t_imu), dtype=bool)
    keep[:start] = True
    buf, nxt = [], start
    for tf in list(t_frames) + [np.inf]:
        while nxt < len(t_imu) and t_imu[nxt] <= tf:
            buf.append(nxt)
            nxt += 1
            if len(buf) > cap:
                del buf[:drop]
        keep[buf] = True  # what the frame finds in the buffer and consumes
        buf = []
    return keep


def test_buffer_cap_matches_the_push_erase_loop():
    from fbus_ekf_b200 import replay
    rng = np.random.default_rng(5)
    for trial in range(30):
        n = int(rng.integers(50, 9000))
        t_imu = np.cumsum(rng.uniform(0.5e-3, 1.5e-3, size=n))
        nf = int(rng.integers(1, 12))
        t_frames = np.sort(rng.uniform(0, t_imu[-1] * 1.05, size=nf))
        start = int(rng.integers(0, min(n, 600)))
        cap, drop = (2000, 500) if trial % 2 == 0 else (int(rng.integers(20, 400)), int(rng.integers(1, 20)))
        got = replay.buffer_cap_keep(t_imu, t_frames, start, cap, drop)
        want = _simulate_buffer(t_imu, t_frames, start, cap, drop)
        assert np.array_equal(got, want), (trial, n, nf, start, cap, drop)
    # 25 Hz frames on a 1 kHz stream: nothing is ever dropped
    t_imu = np.arange(20000) * 1e-3
    assert replay.buffer_cap_keep(t_imu, np.arange(1, 500) * 0.04, 500).all()
