"""The Fortran side of the drop-in boundary, as far as it can be checked without a Fortran compiler (none in this image):
  * the shipped patches apply cleanly to the unmodified reference drivers (needs the CDFTOOLS sources: $CDFTOOLS_REF);
  * every libcdfgpu / cdfio_pinned procedure the patched drivers call is bound by the shipped modules;
  * regenerating the patches from the reference reproduces the shipped files (they are not hand-edited)."""
import os
import re
import shutil
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
PATCHES = ROOT / "cdftools_b200" / "fortran" / "patches"
REF_ROOT = Path(os.environ["CDFTOOLS_REF"]) if os.environ.get("CDFTOOLS_REF") else None
REF = REF_ROOT / "src" if REF_ROOT else None


def _added_lines(name):
    return [l[1:] for l in (PATCHES / name).read_text().split("\n") if l.startswith("+") and not l.startswith("+++")]


def test_patched_drivers_call_only_bound_procedures():
    mod = (ROOT / "cdftools_b200" / "fortran" / "cdfgpu_mod.f90").read_text()
    pinned = (ROOT / "cdftools_b200" / "fortran" / "cdfio_pinned.f90").read_text()
    bound = set(re.findall(r"(?:FUNCTION|SUBROUTINE)\s+(\w+)", mod)) | set(re.findall(r"PUBLIC :: (\w+)", pinned))
    for name in ("cdfmoc.f90.patch", "cdfmocsig.f90.patch", "cdfsigtrp.f90.patch"):
        txt = "\n".join(_added_lines(name))
        used = set(re.findall(r"\b(cdf(?:gpu|moc|mocsig|sigtrp)_gpu?\w*|cdfgpu_\w+|getvar3d_into|close_pinned_files)\s*\(", txt))
        assert used, name
        missing = {u for u in used if u not in bound}
        assert not missing, (name, missing)
        assert "USE cdfgpu" in txt
        if name != "cdfsigtrp.f90.patch":   # the record pipelines read into pinned buffers and take -nc4
            assert "USE cdfio_pinned" in txt and "-nc4" in txt


@pytest.mark.skipif(REF is None or not REF.exists() or shutil.which("patch") is None,
                    reason="needs the CDFTOOLS sources ($CDFTOOLS_REF) and patch(1)")
def test_patches_apply_to_the_reference_and_are_reproducible(tmp_path):
    src = tmp_path / "src"
    src.mkdir()
    for f in ("cdfmoc.f90", "cdfmocsig.f90", "cdfsigtrp.f90"):
        shutil.copy(REF / f, src / f)
    for p in sorted(PATCHES.glob("*.patch")):
        r = subprocess.run(["patch", "-p1", "-i", str(p)], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0 and "FAILED" not in r.stdout, r.stdout + r.stderr
    moc = (src / "cdfmoc.f90").read_text()
    # the hot loop nests are gone, the output block and the rest of the program are untouched
    assert "e1v(ji,jj)*e3v(ji,jj,jk)* ibmask(jbasin,ji,jj)*zv(ji,jj)*1.d0" not in moc
    assert "cdfmoc_gpu_fetch(jslot, dmoc)" in moc and "ierr = putvar (ncout, id_varout(ijvar), REAL(dmoc(jbasin,:,jk))" in moc
    sig = (src / "cdfmocsig.f90").read_text()
    assert "dens(:,:) = sigmai" not in sig and "cdfmocsig_gpu_fetch(jslot, dmoc)" in sig and "CALL CreateOutputFile" in sig
    trp = (src / "cdfsigtrp.f90").read_text()
    assert "dalfa=(dsigma - dsig(ji,jk-1))" not in trp and "cdfsigtrp_gpu_section(npts, npk, nk, eu, zde3" in trp
    assert "IF (lprint) CALL print_out(jsec)" in trp and "CALL CreateOutput (jsec)" in trp
    # regenerate and compare
    before = {p.name: p.read_text() for p in PATCHES.glob("*.patch")}
    r = subprocess.run([sys.executable, str(ROOT / "tools" / "make_fortran_patches.py"), str(REF_ROOT)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    after = {p.name: p.read_text() for p in PATCHES.glob("*.patch")}
    assert before == after
