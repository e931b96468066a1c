"""Chunk counts the fused evaluation takes, decided from the arguments alone (no GPU): 32 chunks per track is accepted,
64 (two epilogue warps per track) and non-powers of two are refused -- the same on every rank, before any collective."""
import pytest
import torch

from wealy_b200 import dist as wd
from wealy_b200 import evaluation as we


def test_32_chunks_per_track_accepted():
    assert wd._chunks_per_track(torch.zeros(10, 32, 8), None, "min", None) == 32
    assert wd._chunks_per_track(torch.zeros(10, 32, 8), 32, "mean", torch.full((10,), 17)) == 32
    assert wd._chunks_per_track(torch.zeros(320, 8), 32, "minmean", None) == 32       # flat [N * s, D] + chunks=
    for redux in ("min", "max", "mean", "meanmin", "minmean"):
        we._check_tracks(32, redux, None)


@pytest.mark.parametrize("s", [64, 24, 3])
def test_other_chunk_counts_refused_before_any_collective(s):
    with pytest.raises(NotImplementedError):
        wd._chunks_per_track(torch.zeros(4, s, 8), None, "min", None)
    with pytest.raises(NotImplementedError):
        wd._chunks_per_track(torch.zeros(4 * s, 8), s, "mean", None)
    with pytest.raises(NotImplementedError):
        we._check_tracks(s, "min", None)


def test_32_chunks_still_refuse_unfused_reductions():
    with pytest.raises(NotImplementedError):
        wd._chunks_per_track(torch.zeros(10, 32, 8), None, "bpwr", None)
