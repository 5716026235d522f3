"""The `trew` binary's argument surface (src/trew.cpp:143-376): validation messages and exit codes, and the loud failure
without a usable GPU.  No GPU needed: every case ends before or at device-context creation."""
import os
import subprocess
import sys

import pytest

from trew_b200 import api, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(args):
    r = subprocess.run([api.CLI_PATH] + args, capture_output=True)
    return r.returncode, r.stdout.decode(), r.stderr.decode()


def test_argument_validation_messages(tmp_path):
    p = os.path.join(str(tmp_path), "a.fastq")
    open(p, "wb").write(synth.fastq_bytes([b"ACGT" * 30]))
    cases = [(["short", "6", "5", p], "MIN_MER must not be greater than MAX_MER."),
             (["short", "2", "5", p], "MIN_MER must be greater than or equal to 3."),
             (["short", "5", "65", p], "MAX_MER must be less than or equal to 64."),
             (["short", "5", "32", p, "-m", "16"], "TABLE_MAX_MER must be less than or equal to 15."),
             (["long", "5", "32", p, "-s", "60"], "SLICE_LENGTH must be greater than or equal to twice of MAX_MER."),
             (["short", "5", "32", p, "-q", "2"], "QUEUE_SIZE must be -1 (unlimited) or greater than or equal to 4."),
             (["short", "5", "32", p, "-t", "1"], "You must use at least two threads."),
             (["short", "5", "32", p, "-L", "0", "-H", "0.8"], "Baseline must be in range 0 to 1."),
             (["short", "5", "32", p, "-L", "0.9", "-H", "0.8"], "Low baseline must be smaller than high baseline."),
             (["short", "5", "32", "--paired_end", "--fq1", p], "--fq1 and --fq2 are required in paired-end mode."),
             (["short", "5", "32", "/nonexistent.fastq"], "/nonexistent.fastq : file not found"),
             # argparse's `--name=value` and glued short-option values reach the same checks
             (["short", "5", "32", p, "--thread=1"], "You must use at least two threads."),
             (["short", "5", "32", p, "-t1"], "You must use at least two threads."),
             (["long", "5", "32", p, "-s60"], "SLICE_LENGTH must be greater than or equal to twice of MAX_MER."),
             (["long", "5", "32", p, "--slice_length=60"], "SLICE_LENGTH must be greater than or equal to twice of MAX_MER."),
             (["short", "5", "32", p, "-L0.9", "-H0.8"], "Low baseline must be smaller than high baseline.")]
    for args, msg in cases:
        rc, out, err = run(args)
        assert rc == 1 and msg in err and out == "", args


def test_slice_length_limit_is_reported(tmp_path):
    """The reference accepts any -s >= 2*MAX_MER (src/trew.cpp:204-207); the GPU path stops at 512 and says so, both
    through the C ABI (trew_dev_last_error(NULL)) and on the command line."""
    p = os.path.join(str(tmp_path), "a.fastq")
    open(p, "wb").write(synth.fastq_bytes([b"ACGT" * 300]))
    rc, out, err = run(["long", "5", "32", p, "-s", "1000"])
    assert rc == 1 and out == "" and "SLICE_LENGTH above 512 is not supported" in err
    with pytest.raises(api.TrewError) as e:
        api.DeviceContext(api.MODE_LONG, 5, 32, slice_length=1000)
    assert e.value.status == 1 and "SLICE_LENGTH above 512" in str(e.value)


def test_version_and_usage():
    rc, out, _ = run(["--version"])
    assert rc == 0 and out.strip() == "0.5.0"     # src/trew.cpp:23
    rc, _, err = run([])
    assert rc == 1 and "Usage: trew" in err
    rc, _, err = run(["medium", "5", "32", "x"])
    assert rc == 1 and "{long,short}" in err


def test_no_cpu_fallback(tmp_path):
    """Without a usable CUDA device the program must fail loudly, never compute on the host.  CUDA_VISIBLE_DEVICES=""
    hides every device, so the check runs the same on a machine with a GPU and on one without."""
    p = os.path.join(str(tmp_path), "a.fastq")
    open(p, "wb").write(synth.fastq_bytes([b"TTAGGG" * 25]))
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([api.CLI_PATH, "short", "5", "32", p], capture_output=True, env=env)
    assert r.returncode == 1 and b"cannot create device context" in r.stderr and r.stdout == b""
    code = ("from trew_b200 import api\n"
            "try:\n"
            "    api.DeviceContext(api.MODE_SHORT, 5, 32)\n"
            "except api.TrewError as e:\n"
            "    print(e.status)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, env=env, cwd=ROOT)
    assert r.stdout.decode().strip() == "2", r.stderr.decode()[-2000:]     # TREW_ERR_CUDA
