"""Host report (process_output / final_process_output restatement) against the reference's stdout captured in
tests/golden/cli_cases.json.gz.  The six count tables fed to it come from the CPU oracle here (the GPU
variant of the same comparison is tests/test_gpu_cli.py).  CPU only."""
from oracle.oracle import Oracle
from trew_b200 import api


def split_sections(text):
    """-> list of (header, sorted rows); rows inside a section tie-break differently in the reference
    (unstable std::sort on tied keys, SURVEY.md 4.3), so sections are compared as sorted multisets."""
    out = []
    for line in text.splitlines():
        if line.startswith(">"):
            out.append([line, []])
        else:
            out[-1][1].append(line)
    return [(h, sorted(r)) for h, r in out]


def parse_cli_args(args):
    mode = api.MODE_LONG if args[0] == "long" else (api.MODE_PAIR if "--paired_end" in args else api.MODE_SHORT)
    mn, mx = int(args[1]), int(args[2])
    files = [a for a in args[3:] if a.endswith(".fastq")]
    return mode, mn, mx, files


def run_case(case, scan):
    mode, mn, mx, files = parse_cli_args(case["args"])
    rep = api.Report(mn)
    if mode == api.MODE_PAIR:
        groups = [(files[0], files[1])]
    else:
        groups = [(f, None) for f in files]
    for f1, f2 in groups:
        r1 = [s.encode() for s in case["files"][f1]]
        r2 = [s.encode() for s in case["files"][f2]] if f2 else None
        if mode == api.MODE_LONG:
            r1 = [r for r in r1 if len(r) >= 150]
        rep.add_file("<%s>" % f1, scan(mode, mn, mx, r1, r2))
    return rep.finish()


def oracle_scan(mode, mn, mx, r1, r2):
    return Oracle(mn, mx).scan(mode, r1, r2)


def putative(sections):
    return [r for h, r in sections if h == ">Putative_TRM"][0]


def test_report_sections_match_reference(cli_cases):
    for case in cli_cases:
        got = split_sections(run_case(case, oracle_scan))
        want = split_sections(case["stdout"])
        assert [h for h, _ in got] == [h for h, _ in want], case["name"]
        for (h, g), (_, w) in zip(got, want):
            if h != ">Putative_TRM":
                assert g == w, (case["name"], h)


def top_rows(rows):
    best = max(int(r.split(",")[2]) for r in rows)
    return sorted(r for r in rows if int(r.split(",")[2]) == best)


def test_putative_trm_matches_where_defined(cli_cases):
    # >Putative_TRM depends on how ties are cut in get_score_map (src/kmer.cpp:2710-2758); the reference is
    # not deterministic there (SURVEY.md 4.3: scores change with -t).  So: the winners (rows with the top
    # score) must always overlap, and the whole section must be identical on inputs without ties at the cuts.
    names = {}
    for case in cli_cases:
        got = putative(split_sections(run_case(case, oracle_scan)))
        want = putative(split_sections(case["stdout"]))
        names[case["name"]] = got == want
        assert set(top_rows(got)) & set(top_rows(want)), case["name"]
    assert names["short_tie_free"] and names["pair_5_32"]


def test_empty_input_gives_the_reference_skeleton():
    rep = api.Report(5)
    rep.add_file("/x/test.fastq.gz", {})
    assert rep.finish() == ">H:/x/test.fastq.gz\n>L:/x/test.fastq.gz\n>Putative_TRM\nNO_PUTATIVE_TRM,-1\n"


def test_reference_fixture_rows_3_64():
    # `trew short 3 64 test/test.fastq` (SURVEY.md 4.2 / 8(c)): the only bundled-fixture run with rows; the reference's
    # test/test.fastq is kept byte for byte in tests/golden/fixtures (tests/test_fixtures.py pins its md5)
    import os
    p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fixtures", "test.fastq")
    rc, _, reads, _ = api.ingest_records(api.MODE_SHORT, p)
    rep = api.Report(3)
    rep.add_file(p, Oracle(3, 64).scan(0, reads))
    text = rep.finish()
    low = dict(split_sections(text))[">L:" + p]
    assert low == sorted(["3,TTA,157,105,0,-", "3,TGA,24,6,0,+", "3,TGG,11,5,0,+", "3,TAG,10,6,0,+", "3,TTG,10,7,0,+"])
