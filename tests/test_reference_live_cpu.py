"""Differential tests against the reference's OWN functions on generated inputs: frame-index math (decoder_utils.find_closest_indices
/ sample_closest), fixed-stride spans, chunk sizes, the stage-replay comparator, shot logic and the InternVideo2 tube formulation
must agree with the reference on inputs nobody hand-picked.  The inputs are the seeded cases of oracle/reference_cases.py; the
reference's answers on them are stored in tests/golden/reference_cases.json (`python -m oracle.make_golden` regenerates them from
a reference checkout)."""

from __future__ import annotations

import json

import pytest
from conftest import GOLDEN

from cosmos_curate_b200 import compare as C
from cosmos_curate_b200 import sampling as S
from cosmos_curate_b200 import spans as SP
from oracle import reference_cases as R


@pytest.fixture(scope="module")
def ref():
    return json.loads((GOLDEN / "reference_cases.json").read_text())


def _cases(ref, name: str, cases: list) -> list:
    assert R.digest(cases) == ref["digest"][name], f"oracle/reference_cases.py no longer generates the {name} cases the golden answers were made for"
    return cases


def test_sample_closest_agrees_with_the_reference(ref):
    for i, (c, want) in enumerate(zip(_cases(ref, "timestamps", R.timestamp_cases()), ref["sample_closest"], strict=True)):
        ts = c["ts"]
        got = S.sample_closest(ts, c["rate"], start=ts[0], stop=ts[-1], endpoint=c["endpoint"], dedup=c["dedup"])
        assert [R.values_sha256(g) for g in got] == want["outputs"], i
        assert R.values_sha256(S.find_closest_indices(ts, R.closest_targets(ts))) == want["find_closest"], i


def test_fixed_stride_spans_and_uuids_agree_with_the_reference(ref):
    for c, want in zip(_cases(ref, "fixed_stride", R.fixed_stride_cases()), ref["fixed_stride"], strict=True):
        got = SP.make_spans_fixed_stride(0.0, c["end"], c["clip_len"], c["stride"], c["min_len"])
        assert len(got) == want["n_spans"] and R.spans_sha256(got) == want["spans_sha256"]
        assert R.uuids_sha256(SP.make_clip_uuids(c["session"], got[:50])) == want["uuids_sha256"]


def test_chunk_sizes_agree_with_the_reference(ref):
    for c, want in zip(_cases(ref, "chunks", R.chunk_cases()), ref["chunks"], strict=True):
        assert [len(ch) for ch in SP.split_by_chunk_size(c["spans"], c["per_chunk"] * 8, R.chunk_size)] == want


def test_compare_values_agrees_with_the_reference(ref):
    for c, want in zip(_cases(ref, "compare", R.compare_cases()), ref["compare"], strict=True):
        for other, w in zip((c["candidate"], c["golden"]), want, strict=True):
            got = [R.diff_key(d) for d in C.compare_values("t", c["golden"], other, atol=c["atol"])]
            assert repr(got) == w  # repr: NaN-carrying details compare equal as text


def test_shot_logic_agrees_with_the_reference(ref):
    """0/1 transition tracks -> scenes -> filtered scenes: transnetv2_extraction_stages._get_scenes / _get_filtered_scenes."""
    from cosmos_curate_b200 import shots

    for i, (c, want) in enumerate(zip(_cases(ref, "shots", R.shot_cases()), ref["shots"], strict=True)):
        got = shots.scenes_from_predictions(c["track"].reshape(-1, 1), entire_scene_as_clip=c["entire"])
        assert len(got) == want["n_scenes"] and R.values_sha256(got) == want["scenes"] and got.dtype.str == want["dtype"], i
        if len(got):
            got_f = shots.filter_scenes(got.copy(), min_length=c["min_len"], max_length=c["max_len"], max_length_mode=c["mode"], crop_length=c["crop"])
            assert R.values_sha256(got_f) == want["filtered"], i


def test_video_tube_oracle_agrees_with_the_reference_formulation(ref):
    """oracle/video_tube.py vs InternVideo2MultiModality._construct_frames (cv2.resize + numpy) on arbitrary sizes, every float32 bit:
    up- and down-scaling, 1-pixel sources and targets, the exact-2x INTER_AREA reroute, the copy for equal sizes."""
    from oracle import video_tube as T

    for c, want in zip(_cases(ref, "tubes", R.tube_cases()), ref["tubes"], strict=True):
        got = T.construct_frames(R.tube_frames(c), fnum=8, target_size=(c["tw"], c["th"]))
        assert list(got.shape) == want["shape"] and got.dtype.str == want["dtype"] and R.tube_sha256(got) == want["sha256"], c
