"""The device context's grow-on-demand buffers: export, sort, report filter, unit records, finish_merged and the peer
copies of a group are sized by the call that needs them and kept for the next one.  One context (and one group) is
used for a small input and then for a large one, so that every such buffer is first allocated and then grown, and
every result must equal that of a fresh context.  Also the one-read fallback of submit_chunk: a chunk whose coarse
range does not fit a staging slot is cut into single reads."""
import numpy as np
import pytest

from trew_b200 import api, synth

pytestmark = pytest.mark.gpu

SMALL, LARGE = 20_000, 700_000   # reads; each gives two rows, so LARGE passes the first export size of 2^20 rows
REC_CAP = 4 * LARGE
FILTER = 2


def repeat_reads(seed, n, length=150):
    """Tandem repeats of random 13- to 20-base units (two table rows per read, nearly all distinct) plus 1 % of the
    bench shape's reads, with telomeric ones."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(13, 21, size=n)
    units = rng.integers(0, 4, size=(n, 20), dtype=np.uint8)
    idx = np.take_along_axis(units, np.arange(length)[None, :] % lens[:, None], axis=1)
    mat = np.frombuffer(b"ACGT", dtype=np.uint8)[idx]
    return np.concatenate([mat, synth.config_short(seed, n // 100, length, telomeric=0.05)])


def submit(ctx, mat, times=1):
    buf, locs = api.matrix_chunk(mat)
    for _ in range(times):
        ctx.submit_chunk(buf, locs)


def fresh(mat):
    """Tables, report-filtered tables, unit records and the doubled tables, each from a context of its own."""
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as c:
        submit(c, mat)
        tables = c.finish_view().copy()
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as c:
        c.set_report_filter(FILTER)
        submit(c, mat)
        filtered = c.finish_view().copy()
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as c:
        c.enable_unit_records(REC_CAP)
        submit(c, mat)
        recs = c.unit_records()
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as c:
        submit(c, mat, times=2)
        doubled = c.finish_view().copy()
    return tables, filtered, recs, doubled


def same(got, want):
    return got.shape == want.shape and got.tobytes() == want.tobytes()


def test_one_context_grows_every_buffer():
    import torch
    sets = [repeat_reads(31, SMALL), repeat_reads(32, LARGE)]
    wants = [fresh(m) for m in sets]
    assert wants[1][0].shape[0] > (1 << 20) and wants[1][1].shape[0] > 1000
    with api.DeviceContext(api.MODE_SHORT, 5, 32) as ctx, api.DeviceContext(api.MODE_SHORT, 5, 32) as other:
        ctx.enable_unit_records(REC_CAP)
        for mat, (tables, filtered, recs, doubled) in zip(sets, wants):
            ctx.reset()
            other.reset()
            submit(ctx, mat)
            assert same(ctx.finish_view(), tables)
            ctx.set_report_filter(FILTER)
            assert same(ctx.finish_view(), filtered)
            ctx.set_report_filter(0)
            assert same(ctx.unit_records(), recs)
            submit(other, mat)
            n = other.export_rows()
            rows = torch.zeros((n, 4), dtype=torch.int64, device="cuda:0")
            assert other.export_rows(rows.data_ptr(), n) == n
            assert same(ctx.finish_merged_view([(rows.data_ptr(), n)]), doubled)
            del rows
    with api.MultiContext(api.MODE_SHORT, 5, 32, devices=[0, 0]) as m:
        m.enable_unit_records(REC_CAP)
        for mat, (tables, _, recs, _) in zip(sets, wants):
            m.reset()
            buf, locs = api.matrix_chunk(mat)
            half = (mat.shape[0] // 2) * (mat.shape[1] + 1)
            m.submit_chunk(buf[:half], locs[:mat.shape[0] // 2])              # first device
            m.submit_chunk(buf[half:], locs[mat.shape[0] // 2:] - half)       # second device: its rows cross to the first
            assert same(m.finish_view(), tables)
            assert same(m.unit_records(), recs)


def test_one_read_fallback_in_long_mode():
    """With a 64 KiB staging slot, a 173,000-base read fills a slot nearly alone (65,392 of 65,536 bytes), and the
    coarse range it shares with a few 300-base reads does not fit: submit_chunk splits that range into single reads."""
    small = synth.adversarial_long(41, 400, min_len=300, max_len=300)
    big = synth.adversarial_long(42, 1, min_len=173_000, max_len=173_000)
    reads = small[:200] + big + small[200:]
    with api.DeviceContext(api.MODE_LONG, 5, 32, staging_bytes=1 << 16, n_staging=2, host_threads=2) as ctx:
        ctx.submit_reads(reads)
        got = ctx.finish()
    with api.DeviceContext(api.MODE_LONG, 5, 32) as ctx:
        for r in reads:
            ctx.submit_reads([r])
        want = ctx.finish()
    assert got == want and len(got) > 20
