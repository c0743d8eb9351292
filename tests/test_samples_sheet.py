"""`vargeno-b200 geno-samples` refuses a malformed sample sheet with its line number before it reads the index or touches a
device: the index prefix given here does not exist, so a run that got past the sheet would say so instead."""
import os
import subprocess

import pytest

from vargeno_b200 import build as vb


def _run(tmp_path, sheet_text, out_dir="out"):
    vb.build()
    (tmp_path / "a.fq").write_text("@r\nACGT\n+\nIIII\n")
    (tmp_path / "b.fq").write_text("@r\nACGT\n+\nIIII\n")
    sheet = tmp_path / "samples.tsv"
    sheet.write_text(sheet_text)
    out = tmp_path / out_dir
    p = subprocess.run([vb.HOST_BIN, "geno-samples", str(tmp_path / "no_index"), str(sheet), str(tmp_path / "snps.vcf"), str(out)],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=str(tmp_path))
    return p, out


@pytest.mark.parametrize("text, line, what", [
    ("a\ta.fq\nb b.fq\n", 2, "expected <name><TAB><reads>"),
    ("a\ta.fq\n\tb.fq\n", 2, "empty sample name"),
    ("# cohort\n\na/b\ta.fq\n", 3, "is not made of"),
    ("x\ta.fq\ny\tb.fq\nx\tb.fq\n", 3, "appears twice"),
    ("a\ta.fq,missing.fq\n", 1, "missing.fq does not exist"),
    ("a\t\n", 1, "no reads file"),
])
def test_bad_sheet_is_refused_with_its_line(tmp_path, text, line, what):
    p, out = _run(tmp_path, text)
    assert p.returncode == 1
    assert "samples.tsv:%d: " % line in p.stderr and what in p.stderr, p.stderr
    assert "no_index" not in p.stderr and "Initializing" not in p.stderr
    assert not out.exists()


@pytest.mark.parametrize("text", ["", "# only a comment\n\n"])
def test_empty_sheet_is_refused(tmp_path, text):
    p, out = _run(tmp_path, text)
    assert p.returncode == 1
    assert "samples.tsv: no samples" in p.stderr, p.stderr
    assert "no_index" not in p.stderr and not out.exists()


def test_good_sheet_gets_to_the_index(tmp_path):
    """comments, blank lines, CRLF, a comma list: the sheet passes, the output directory is made with its missing parents, and the missing index is next"""
    p, out = _run(tmp_path, "# name\treads\n\nS-1.a_b\ta.fq\r\nS2\ta.fq,,b.fq\n", "cohort/run1/vcf")
    assert p.returncode == 1
    assert "no_index" in p.stderr and "samples.tsv" not in p.stderr, p.stderr
    assert os.path.isdir(out)


def test_output_path_taken_by_a_file(tmp_path):
    (tmp_path / "taken").write_text("")
    p, out = _run(tmp_path, "S1\ta.fq\n", "taken")
    assert p.returncode == 1 and "cannot create the directory" in p.stderr, p.stderr
    assert "no_index" not in p.stderr
