"""GPU test of the host drivers: the reference's test/diff.sh contract.

test/diff.sh (reference, lines 1-20) runs the four debug programs next to a.png / b.png and
diffs every file of ser/ against par/ and of sergh/ against pargh/ (96 PPMs per program).
Here par/ and pargh/ come from debug/stereopar and debug/stereopar-ghost (host/driver.c over
the C ABI); ser/ and sergh/ come from the reference's own serial programs when oracle/_ref
holds them (built by `make -C oracle refserial`), and in any case from the CPU oracle's
arrays written with a Python restatement of the reference's PPM writer, whose CRC32s are
stored in tests/golden/ref_cases.json for fixtures 1-3.
"""
import os
import shutil
import subprocess

import numpy as np
import pytest

import oracle
import ref_cases
from util import IMGS, ROOT, THRESHOLD

pytestmark = pytest.mark.gpu

NAMES = (["edges-1.ppm", "edges-2.ppm", "score_best-0.ppm", "web-1.ppm", "web-2.ppm", "output-0.ppm"] +
         ["%s-%d.ppm" % (n, i) for n in ("matches", "score_all", "scores") for i in range(30)])


@pytest.fixture(scope="module")
def workdir(tmp_path_factory):
    d = tmp_path_factory.mktemp("diffsh")
    for f in ("a.png", "b.png"):
        shutil.copy(os.path.join(IMGS, "1-240x135", f), d / f)
    for sub in ("ser", "par", "sergh", "pargh"):
        (d / sub).mkdir()
    for exe in ("stereopar", "stereopar-ghost"):
        path = os.path.join(ROOT, "debug", exe)
        assert os.path.exists(path), "run `make build=debug` (or __graft_entry__.build())"
        r = subprocess.run([path, "a.png", "b.png"], cwd=d, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        f = r.stdout.split()
        assert f[:6] == ["width", "=", "240,", "height", "=", "135,"] and float(f[14]) > 0  # time.sh reads $15
    return d


def test_96_files_each(workdir):
    assert len(NAMES) == 96
    for sub in ("par", "pargh"):
        assert sorted(os.listdir(workdir / sub)) == sorted(NAMES)


@pytest.mark.parametrize("variant,sub", [(0, "par"), (1, "pargh")])
def test_ppms_equal_oracle_arrays(orc, workdir, variant, sub):
    expect = ref_cases.driver_ppms(orc, "1-240x135", variant)
    for name in NAMES:
        assert open(workdir / sub / name).read() == expect[name], name


def _stored_reference_files(fixture):
    return {sub: ref_cases.stored()["driver/%s/%s" % (fixture, v)] for sub, v in (("par", "wrap"), ("pargh", "ghost"))}


def test_diff_sh_against_the_reference_serial_programs(workdir):
    for sub, want in _stored_reference_files("1-240x135").items():
        assert ref_cases.file_crcs(workdir / sub) == want, sub
    ser = os.path.join(ROOT, "oracle", "_ref", "debug", "stereomatch")
    sergh = os.path.join(ROOT, "oracle", "_ref", "debug", "stereomatch-ghost")
    if not (os.path.exists(ser) and os.path.exists(sergh)):
        return  # the live comparison needs the reference's serial programs built into oracle/_ref/debug
    for exe in (ser, sergh):
        r = subprocess.run([exe, "a.png", "b.png"], cwd=workdir, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    problems = []
    for name in sorted(os.listdir(workdir / "ser")):  # the loop of test/diff.sh:14-20
        for x, y in (("ser", "par"), ("sergh", "pargh")):
            if open(workdir / x / name, "rb").read() != open(workdir / y / name, "rb").read():
                problems.append("problem with image %s (%s - %s)" % (name, x, y))
    assert len(os.listdir(workdir / "ser")) == 96
    assert not problems, problems


@pytest.mark.parametrize("fixture", ["2-480x270", "3-960x540"])
def test_diff_sh_larger_fixtures_against_stored_reference_files(tmp_path, fixture):
    """The test/diff.sh loop on fixtures 2 and 3 (fixture 1: the tests above): every file of par/ and pargh/,
    written by debug/stereopar and debug/stereopar-ghost, against the stored CRC32s of ser/ and sergh/."""
    for f in ("a.png", "b.png"):
        shutil.copy(os.path.join(IMGS, fixture, f), tmp_path / f)
    for sub, want in _stored_reference_files(fixture).items():
        (tmp_path / sub).mkdir()
        exe = os.path.join(ROOT, "debug", "stereopar" if sub == "par" else "stereopar-ghost")
        r = subprocess.run([exe, "a.png", "b.png"], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0, (sub, r.stderr)
        assert ref_cases.file_crcs(tmp_path / sub) == want, (fixture, sub)
    shutil.rmtree(tmp_path, ignore_errors=True)


@pytest.mark.parametrize("fixture", ["1-240x135", "2-480x270", "3-960x540"])
def test_diff_sh_with_the_reference_host_side(tmp_path, fixture):
    """INTEGRATION.md section 2 as a real build: host/driver.c compiled with the REFERENCE'S OWN image.c /
    stb_image.h / util.h (oracle/Makefile refhost), images uploaded in the reference's double layout
    (sm_upload_f64).  The test/diff.sh loop: all 96 files of par/ and pargh/ byte-equal to ser/ and sergh/ written
    by the reference's serial programs (src/stereo.cu:350-409, src/image.c:18-88)."""
    dbg = os.path.join(ROOT, "oracle", "_ref", "debug")
    opt = os.path.join(ROOT, "oracle", "_ref", "debugopt")
    exes = {"par": os.path.join(dbg, "stereopar-refhost"), "pargh": os.path.join(dbg, "stereopar-ghost-refhost"),
            "ser": os.path.join(opt, "stereomatch"), "sergh": os.path.join(opt, "stereomatch-ghost")}
    if not all(os.path.exists(e) for e in exes.values()):
        pytest.skip("oracle/_ref refhost / refserialopt not built (needs /root/reference at build time)")
    for f in ("a.png", "b.png"):
        shutil.copy(os.path.join(IMGS, fixture, f), tmp_path / f)
    for sub, exe in exes.items():
        (tmp_path / sub).mkdir()
        r = subprocess.run([exe, "a.png", "b.png"], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0, (sub, r.stderr)
    names = sorted(os.listdir(tmp_path / "ser"))
    assert names == sorted(NAMES)
    problems = [(n, x, y) for n in names for x, y in (("ser", "par"), ("sergh", "pargh"))
                if open(tmp_path / x / n, "rb").read() != open(tmp_path / y / n, "rb").read()]
    assert not problems, problems[:5]
    shutil.rmtree(tmp_path, ignore_errors=True)


def test_timing_build_writes_nothing(tmp_path):
    for f in ("a.png", "b.png"):
        shutil.copy(os.path.join(IMGS, "2-480x270", f), tmp_path / f)
    for exe in ("stereopar", "stereopar-ghost"):
        path = os.path.join(ROOT, "timing", exe)
        assert os.path.exists(path), "run `make build=timing`"
        r = subprocess.run([path, "a.png", "b.png"], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert r.stdout.startswith("width = 480, height = 270, t1 = ")
    assert sorted(os.listdir(tmp_path)) == ["a.png", "b.png"]


def test_degenerate_contour_is_reported(tmp_path):
    from PIL import Image
    flat = np.full((64, 64), 128, np.uint8)
    Image.fromarray(flat, "L").save(tmp_path / "a.png")
    Image.fromarray(flat, "L").save(tmp_path / "b.png")
    r = subprocess.run([os.path.join(ROOT, "timing", "stereopar"), "a.png", "b.png"], cwd=tmp_path,
                       capture_output=True, text=True)
    # flat images: web is 30 everywhere, (max-min)/lines == 0; the reference divides by zero
    assert r.returncode != 0 and "divides by zero" in r.stderr


def test_stereobatch_c_program_over_all_gpus():
    """timing/stereobatch (host/batch.c): whole pairs sharded over every visible GPU from C through sm_multi_*;
    its CRC of the returned webs must equal the oracle's webs of the same synthetic pairs."""
    import zlib
    exe = os.path.join(ROOT, "timing", "stereobatch")
    assert os.path.exists(exe), "run `make build=timing` (or __graft_entry__.build())"
    orc = oracle.Oracle()
    w, h, D, sw, n = 320, 180, 64, 9, 7
    for vname_, variant in (("wrap", 0), ("ghost", 1)):
        for kind, dt in (("i32", np.int32), ("u8", np.uint8)):
            r = subprocess.run([exe, str(w), str(h), str(D), str(sw), str(n), vname_, kind], capture_output=True, text=True)
            assert r.returncode == 0, r.stderr
            fields = dict(kv.split(" = ") for kv in r.stdout.strip().split(", "))
            assert int(fields["pairs"]) == n and float(fields["elapsed"]) > 0 and int(fields["gpus"]) >= 1
            webs = []
            for k in range(n):
                left, right, _ = orc.synth_pair(1234 + 2 * k, w, h, D)
                e1, e2 = orc.edges(left, THRESHOLD, variant), orc.edges(right, THRESHOLD, variant)
                webs.append(orc.match_wta(e1, e2, D, sw, variant)[1].astype(dt))
            crc = "%08x" % (zlib.crc32(np.stack(webs).tobytes()) & 0xFFFFFFFF)
            assert fields["web_crc32"] == crc, (vname_, kind, r.stdout)
