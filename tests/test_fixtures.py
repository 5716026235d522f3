"""BASELINE.json configs[0]: the reference's own bundled fixtures (test/test.fastq(.gz), test/test_long.fastq(.gz),
used by test/test.cpp:260-443), copied byte for byte into tests/golden/fixtures/.  CPU half: the files are the
reference's, and the oracle + the host report layer reproduce the compiled reference's stdout on them
(captured with oracle/_ref/trew_ref; SURVEY.md 4.2 / 8(c)).  The CUDA half is tests/test_gpu_cli.py."""
import gzip
import hashlib
import os

import pytest

from oracle.oracle import Oracle
from trew_b200 import api
from test_report import split_sections

HERE = os.path.dirname(os.path.abspath(__file__))
FIX = os.path.join(HERE, "golden", "fixtures")

MD5 = {"test.fastq": "93ef68f7a029aded6dd6ef15455ecdfb", "test.fastq.gz": "89725d479ae273c61e2aea655b09c664",
       "test_long.fastq": "a7afb5aeb80e4b071110b95419d367fb", "test_long.fastq.gz": "eaeb30fd3082f2b92e75fca67ecb7cd6"}

# `trew_ref short 3 64 test/test.fastq` (identical at -t 2 and -t 4, plain and .gz): the only bundled-fixture run with rows
L_ROWS_3_64 = ["3,TTA,157,105,0,-", "3,TGA,24,6,0,+", "3,TGG,11,5,0,+", "3,TTG,10,7,0,+", "3,TAG,10,6,0,+"]
PUTATIVE_3_64 = ["3,TGA,4,+", "3,TAG,3,+", "3,TGG,3,+", "3,TTA,3,-", "3,TTG,1,+"]
EMPTY = ">H:%s\n>L:%s\n>Putative_TRM\nNO_PUTATIVE_TRM,-1\n"


def fixture(name):
    return os.path.join(FIX, name)


def records(name):
    data = (gzip.open(fixture(name)) if name.endswith(".gz") else open(fixture(name), "rb")).read()
    return data.split(b"\n")[:-1][1::4]


@pytest.mark.parametrize("name", sorted(MD5))
def test_fixture_files_are_the_references(name):
    # MD5 holds the digests of the reference's own test/ files
    assert hashlib.md5(open(fixture(name), "rb").read()).hexdigest() == MD5[name]


def test_fixture_shapes():
    short, long_ = records("test.fastq"), records("test_long.fastq")
    assert records("test.fastq.gz") == short and records("test_long.fastq.gz") == long_
    assert len(short) == 100 and {len(r) for r in short} == {246}
    assert len(long_) == 10 and min(map(len, long_)) == 9095 and max(map(len, long_)) == 17870


def report_text(mode, mn, mx, reads, name, slice_len=150):
    tables = Oracle(mn, mx, slice_len=slice_len).scan(mode, reads)
    rep = api.Report(mn)
    rep.add_file(name, tables)
    return rep.finish()


def test_oracle_and_report_on_short_fixture_3_64():
    out = report_text(0, 3, 64, records("test.fastq"), "F")
    sec = dict(split_sections(out))
    assert sec[">H:F"] == []
    assert sec[">L:F"] == sorted(L_ROWS_3_64)
    # TTG and TAG tie at forward = 10 on a top-4 cut of get_score_map (src/kmer.cpp:2710-2758), so the reference's
    # scores depend on its hash-map order (SURVEY.md 4.3); units and directions are pinned, scores are not
    strip = lambda rows: sorted((r.split(",")[0], r.split(",")[1], r.split(",")[3]) for r in rows)
    assert strip(sec[">Putative_TRM"]) == strip(PUTATIVE_3_64)


@pytest.mark.parametrize("mode,mn,mx,name", [(0, 5, 32, "test.fastq"), (0, 5, 64, "test.fastq"), (2, 5, 32, "test_long.fastq"),
                                             (2, 5, 64, "test_long.fastq"), (2, 3, 64, "test_long.fastq")])
def test_oracle_and_report_give_the_empty_skeleton(mode, mn, mx, name):
    # test/test.cpp:260-443 (main_test_32/_64, main_test_long_32/_64) only checks "does not throw"; the compiled
    # reference prints the empty skeleton for all of them
    assert report_text(mode, mn, mx, records(name), "F") == EMPTY % ("F", "F")
