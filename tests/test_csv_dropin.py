"""Row f2 (CSV reader/writer + main driver, Source.cpp:1437-1598).

CPU: the reference's OWN main() (compiled, unmodified, in oracle/_ref) is run on a generated Test_film_dose.csv with
its hard-coded user settings; reading the same file with this repo's CSV reader, evaluating with the oracle and writing
with this repo's CSV writer must give a byte-identical `_mod.csv`.  GPU: the `aai_main` driver itself."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))


def _build(tmp_path, src, name, link_lib):
    exe = str(tmp_path / name)
    cmd = [os.environ.get("CXX", "g++"), "-std=c++17", src, "-o", exe]
    if link_lib:
        libdir = os.path.join(ROOT, "area_average_interpolation_b200")
        cmd += ["-L" + libdir, "-laai_b200", "-Wl,-rpath," + libdir]
    subprocess.run(cmd, check=True)
    return exe


def _write_input(path, w=300, h=260, seed=3):
    rng = np.random.default_rng(seed)
    img = rng.uniform(0, 4096, size=(h, w))
    with open(path, "w") as f:
        for row in img:
            f.write(",".join(repr(float(v)) for v in row) + "\n")
    return img


def _run_reference_main(cwd):
    from oracle import REF_SO

    code = ("import ctypes,sys; lib=ctypes.CDLL(%r); f=getattr(lib,'_Z18aai_reference_mainv'); f.restype=ctypes.c_int; "
            "sys.exit(f() & 0xff)" % REF_SO)
    return subprocess.run([sys.executable, "-c", code], cwd=cwd, capture_output=True, text=True)


def test_csv_reader_writer_reproduce_the_reference_main_byte_for_byte(tmp_path, built):
    from oracle import port, ref

    if not ref.available:
        pytest.skip("oracle/_ref/libaai_ref.so not present")
    img = _write_input(tmp_path / "Test_film_dose.csv")
    out = _run_reference_main(str(tmp_path))
    assert out.returncode == 0 and "Run terminated correctly." in out.stdout, out.stdout[-500:]
    want = (tmp_path / "Test_film_dose_mod.csv").read_bytes()
    harness = _build(tmp_path, os.path.join(HERE, "csv_host.cpp"), "csv_host", False)
    # reader: same doubles as the text holds
    r = subprocess.run([harness, "read", str(tmp_path / "Test_film_dose.csv"), str(tmp_path / "in.f64")],
                       capture_output=True, text=True, check=True)
    w, h = map(int, r.stdout.split())
    data = np.fromfile(tmp_path / "in.f64", dtype=np.float64).reshape(h, w)
    assert np.array_equal(data, img)
    # the reference's shipped settings (Source.cpp:1528-1534): 150 -> 25.4 dpi, iso (455,455), 1.5 deg, mode 2
    st, dst, _ = port.run(data, 150.0, 25.4, (455.0, 455.0), 1.5, mode=2)
    assert st == 0
    dst.tofile(tmp_path / "out.f64")
    subprocess.run([harness, "write", str(tmp_path / "out.f64"), str(dst.shape[1]), str(dst.shape[0]),
                    str(tmp_path / "mine_mod.csv")], check=True)
    assert (tmp_path / "mine_mod.csv").read_bytes() == want
    # path convention <dir><base>_mod<ext>
    r = subprocess.run([harness, "split", "a/b/Test_film_dose.csv"], capture_output=True, text=True, check=True)
    assert r.stdout.strip() == "a/b/|Test_film_dose|.csv"


def test_csv_reader_tolerant_fields_and_rejected_inputs(tmp_path, built):
    harness = _build(tmp_path, os.path.join(HERE, "csv_host.cpp"), "csv_host", False)
    (tmp_path / "a.csv").write_text("1, 2.5e1,abc,3x\\n 4,5,,6\\n".replace("\\n", "\n"))
    r = subprocess.run([harness, "read", str(tmp_path / "a.csv"), str(tmp_path / "a.f64")], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.split() == ["3", "2"]  # 'abc' and '' are skipped, '3x' reads as 3
    assert np.array_equal(np.fromfile(tmp_path / "a.f64"), [1, 25, 3, 4, 5, 6])
    (tmp_path / "b.csv").write_text("1,2,3\n4,5\n")
    r = subprocess.run([harness, "read", str(tmp_path / "b.csv"), str(tmp_path / "b.f64")], capture_output=True, text=True)
    assert r.returncode == 2 and "different length" in r.stdout
    r = subprocess.run([harness, "read", str(tmp_path / "missing.csv"), str(tmp_path / "c.f64")], capture_output=True, text=True)
    assert r.returncode == 2 and "Failed to read csv file." in r.stdout


def _read_output(path):
    return np.array([[float(v) for v in ln.split(",")] for ln in path.read_text().strip().split("\n")])


@pytest.mark.gpu
def test_aai_main_driver_matches_the_reference_main(tmp_path, built):
    """The driver against the reference's own outputs stored in tests/golden: the reference main's settings (150 ->
    25.4 dpi, 1.5 deg) on a reduced image in fast mode and in area-average mode, and an isocentre outside the image;
    and the shipped settings it runs without arguments against the oracle."""
    from common import golden_source, load_golden
    from oracle import port

    z, meta = load_golden()
    exe = _build(tmp_path, os.path.join(ROOT, "examples", "aai_main.cpp"), "aai_main", True)
    for name in ("fast_dpi_default", "dpi_default_15deg", "neg_angle_far_iso"):
        case = next(c for c in meta["cases"] if c["name"] == name)
        src = golden_source(case).astype(np.float64)
        with open(tmp_path / f"{name}.csv", "w") as f:
            for row in src:
                f.write(",".join(repr(float(v)) for v in row) + "\n")
        args = [case["src_res"], case["dst_res"], case["iso"][0], case["iso"][1], case["angle"], case["mode"]]
        mine = subprocess.run([exe, f"{name}.csv"] + [str(a) for a in args], cwd=str(tmp_path), capture_output=True,
                              text=True)
        assert mine.returncode == 0 and "Run terminated correctly." in mine.stdout, mine.stdout[-500:]
        got, want = _read_output(tmp_path / f"{name}_mod.csv"), z[name]
        assert got.shape == want.shape, name
        # fast mode sums the same values in a different order: identical up to the 6-digit text format
        assert np.abs(got - want).max() <= 2e-5 * np.abs(want).max(), name
        same = sum(np.array_equal(g, [float("%.6g" % v) for v in w]) for g, w in zip(got, want))
        assert same >= 0.9 * len(want), name
    # no arguments: Test_film_dose.csv with the shipped settings, fast mode
    img = _write_input(tmp_path / "Test_film_dose.csv")
    mine = subprocess.run([exe], cwd=str(tmp_path), capture_output=True, text=True)
    assert mine.returncode == 0 and "Run terminated correctly." in mine.stdout, mine.stdout[-500:]
    got = _read_output(tmp_path / "Test_film_dose_mod.csv")
    st, want, _ = port.run(img, 150.0, 25.4, (455.0, 455.0), 1.5, mode=2)
    assert st == 0 and got.shape == want.shape
    assert np.abs(got - want).max() <= 2e-5 * np.abs(want).max()
