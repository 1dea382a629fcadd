"""GPU tier: which in-kernel normalisation scheme the batch extractor launches, and what a failed re-plan leaves behind.

The clustered, ticket and role schemes give bitwise-equal features (test_gpu_parity), so a silent switch from one to
another passes every numerical test. The number of K1 launches of one run_device call tells them apart: one clustered
launch per run of consecutive utterances with equal cluster size, one launch for the ticket or the role scheme."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as ol
from common import afe, synth_utterances, to_afe_params

pytestmark = pytest.mark.gpu

BIG = 1 << 22
MAX_CLUSTER_TILES, MAX_CLUSTER_RUNS, MAX_TICKET_TILES = 4, 8, 8


def _params():
    return to_afe_params(ol.default_params(num_banks=40, norm="cmn", dyn="acc"), BIG)


def _tiles_alone(u):
    """Tiles of an utterance planned on its own; equal to its tiles in any batch whose utterances have at most 8 tiles
    (only batches with a longer utterance re-size the tiles)."""
    b = afe.BatchMfcc(_params(), 0)
    try:
        _, offs, lens = afe.pack_utterances([u])
        b.plan(offs, lens)
        return b.num_tiles
    finally:
        b.close()


def _expected_launches(tiles, flags):
    """The batch's rule, restated: runs of equal cluster size (tiles <= 4, else 0 = ticket scheme) make one clustered launch
    each; with AFE_BATCH_NO_CLUSTER, more than 8 runs or an utterance of more than 8 tiles the batch makes one launch."""
    if flags & afe.BATCH_NO_CLUSTER or max(tiles) > MAX_TICKET_TILES:
        return 1
    sizes = [t if t <= MAX_CLUSTER_TILES else 0 for t in tiles]
    runs = 1 + sum(a != b for a, b in zip(sizes, sizes[1:]))
    return 1 if runs > MAX_CLUSTER_RUNS else runs


def _run_device_launches(utts, flags):
    b = afe.BatchMfcc(_params(), 0, flags=flags)
    pcm, offs, lens = afe.pack_utterances(utts)
    total = b.plan(offs, lens)
    d_pcm = afe.DeviceBuffer(pcm.nbytes + 64); d_pcm.upload(pcm)
    d_out = afe.DeviceBuffer(total * b.width * 4)
    try:
        b.run_device(d_pcm.ptr.value, d_out.ptr.value)
        b.synchronize()
        return b.kernel_launches
    finally:
        b.close(); d_pcm.free(); d_out.free()


def _batches():
    short = synth_utterances(40, 60000, seed=32)        # 1 tile each
    long_ = synth_utterances(40, 160000, seed=31)       # 2 tiles each
    mix = short + synth_utterances(2, 250000, seed=33) + synth_utterances(2, 320000, seed=35) + long_ + \
        synth_utterances(1, 450000, seed=34)            # the batch of test_batch_cluster_normalisation_equals_ticket_scheme
    alternating = [u for pair in zip(short[:10], long_[:10]) for u in pair]
    return {  # name: (utterances, flags, whether clustered launches are expected)
        "sorted_1_2": (short + long_, 0, True),
        "mix_1_to_6": (mix, 0, True),
        "alternating_20_runs": (alternating, 0, False),
        "alternating_no_cluster": (alternating, afe.BATCH_NO_CLUSTER, False),
        "one_long_utterance": (short[:4] + synth_utterances(1, 900000, seed=41), 0, False),
    }


@pytest.mark.parametrize("name", ["sorted_1_2", "mix_1_to_6", "alternating_20_runs", "alternating_no_cluster",
                                  "one_long_utterance"])
def test_batch_scheme_selection_by_launch_count(name):
    utts, flags, clustered = _batches()[name]
    tiles = [_tiles_alone(u) for u in utts]
    want = _expected_launches(tiles, flags)
    assert (want > 1) == clustered, tiles
    assert _run_device_launches(utts, flags) == want


def test_unfused_normalisation_launches_k1_k2_finalize_k3():
    utts = synth_utterances(4, 60000, seed=32) + synth_utterances(4, 160000, seed=31)
    assert _run_device_launches(utts, afe.BATCH_UNFUSED_NORM) == 4


def test_failed_replan_leaves_the_batch_unplanned():
    b = afe.BatchMfcc(_params(), 0)
    try:
        _, offs, lens = afe.pack_utterances(synth_utterances(3, 60000, seed=32) + synth_utterances(3, 160000, seed=31))
        b.plan(offs, lens)
        assert b.num_tiles > 0
        with pytest.raises(afe.AfeError, match="offsets must be even"):
            b.plan(offs + 1, lens)
        assert b.num_tiles == 0
        fo = np.full(len(offs) + 1, -1, np.int64)
        afe.lib().afe_batch_frame_offsets(b._h, fo.ctypes.data_as(C.POINTER(C.c_longlong)))
        assert (fo == -1).all()                     # an unplanned batch has no frame offsets to copy
        with pytest.raises(afe.AfeError, match="afe_batch_plan must be called before running"):
            b.run_device(0, 0)
    finally:
        b.close()
