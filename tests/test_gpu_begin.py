"""A tally may begin while the launches of the one before are still queued on the context's stream (a *_begin does not
wait for them): the new tally's tables and counters are reset behind those launches, a table of unchanged size is
reused, one of another size is replaced only after the stream drains, and host-fed text goes to a staging buffer no
queued launch still reads."""
import importlib

import numpy as np
import pytest

from pss_testlib import FkParams, Oracle, PssParams, Synth, reads_cfg_config2

pytestmark = pytest.mark.gpu
pkg = importlib.import_module("pss-bam_b200")


@pytest.fixture(scope="module")
def small():
    g = Synth.genome(81, [90000, 40000], names=["chr1", "chr2"], n_frac=0.01, lower_frac=0.05)
    ora = Oracle(fasta=g.fasta_bytes())
    ctx = pkg.Context(0)
    ctx.upload_genome(ora.contigs())
    sam = Synth.sam(reads_cfg_config2(seed=82, min_len=20, max_len=90), g, 0, 40000)
    yield ora, ctx, sam
    ctx.close()


@pytest.mark.parametrize("r_before, r_after", [(15, 15), (15, 40), (40, 5), (5, 5)])
def test_pss_begin_behind_queued_launches(small, r_before, r_after):
    import torch
    ora, ctx, sam = small
    f, r, st = ora.pss(sam, PssParams(region_len=r_after))
    dev = torch.frombuffer(bytearray(sam), dtype=torch.uint8).cuda()
    ctx.pss_begin(pkg.PssOptions(region_len=r_before))          # abandoned: its launches are still queued
    ctx.feed_device(dev.data_ptr(), len(sam))
    ctx.feed(sam[: len(sam) // 2])                               # host-fed text, a partial line carried
    ctx.pss_begin(pkg.PssOptions(region_len=r_after))
    ctx.feed(sam, last=True)
    gf, gr = ctx.pss_finish()
    assert ctx.stats() == st
    assert np.array_equal(gf, f) and np.array_equal(gr, r)
    ctx.pss_begin(pkg.PssOptions(region_len=r_after))           # device-resident text right behind the host-fed tally
    ctx.feed_device(dev.data_ptr(), len(sam))
    gf, gr = ctx.pss_finish()
    assert ctx.stats() == st
    assert np.array_equal(gf, f) and np.array_equal(gr, r)


def test_fragkon_begin_behind_queued_launches(small):
    ora, ctx, sam = small
    for k_before, k_after in ((8, 8), (8, 5)):
        fp, tp, fst = ora.fragkon(sam, FkParams(klen=k_after))
        ctx.both_begin(pkg.PssOptions(), pkg.FragkonOptions(klen=k_before))
        ctx.feed(sam)
        ctx.fragkon_begin(pkg.FragkonOptions(klen=k_after))
        ctx.feed(sam, last=True)
        gfp, gtp = ctx.fragkon_finish()
        assert ctx.stats() == fst
        assert np.array_equal(gfp, fp) and np.array_equal(gtp, tp)
