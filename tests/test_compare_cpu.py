"""cosmos_curate_b200/compare.py: the reference's stage-output comparison semantics (stage_compare.py `_compare_values`), checked
(a) against the reference functions' answers on a case table (oracle/reference_cases.comparator_table, answers stored in
tests/golden/reference_cases.json) and (b) against the known answers of the reference's own tests
(tests/cosmos_curate/core/utils/misc/test_stage_compare.py:112-162), then used the way the reference uses it: on task lists."""

from __future__ import annotations

import json
import uuid

import numpy as np
import pytest
from conftest import GOLDEN

from cosmos_curate_b200 import compare as C
from cosmos_curate_b200.data_model import Clip, SplitPipeTask, Video
from oracle import reference_cases as R


def test_compare_values_equals_the_reference_comparator():
    meta = json.loads((GOLDEN / "reference_cases.json").read_text())
    table = R.comparator_table()
    assert R.digest(table) == meta["digest"]["comparator_table"], "oracle/reference_cases.comparator_table changed since the golden answers were made"
    for name, g, c, atol in table:
        got = [R.diff_key(d) for d in C.compare_values("root", g, c, atol=atol)]
        assert repr(got) == meta["comparator_table"][name], name


def test_reference_known_answers():
    a = np.array([1.0, 2.0], dtype=np.float32)
    assert C.compare_values("", {"x": a}, {"x": a.copy()}, atol=0.0) == []
    assert C.compare_values("", a, a + np.float32(5e-4), atol=1e-3) == []
    d = C.compare_values("arr", np.array([0], np.uint8), np.array([1], np.uint8), atol=0.0)
    assert len(d) == 1 and d[0].max_diff_observed == 1.0  # not 255: the difference is taken in float64
    n = np.array([np.nan, 1.0], np.float32)
    assert C.compare_values("arr", n, n.copy(), atol=0.0) == []
    d = C.compare_values("arr", n, np.array([np.nan, 3.0], np.float32), atol=0.5)
    assert d[0].detail == "max diff 2.0" and d[0].max_diff_observed == 2.0  # the matching NaNs do not poison the maximum
    d = C.compare_values("arr", np.zeros((2, 3)), np.zeros((3, 2)), atol=1.0)
    assert d[0].shape_mismatch and "shape mismatch" in d[0].detail
    assert C.compare_values("v", 1, 1.0, atol=1.0)[0].detail == "type mismatch golden=int new=float"


def test_task_lists_the_way_stage_replay_compares_them():
    """SplitPipeTask semantic fields (session_id, videos, errors): stage_perf and timing never count; an embedding off by more than
    atol, a moved clip or a new error key do."""

    def task(score=4.25, emb_shift=0.0, filtered=False, perf=1.0):
        rng = np.random.default_rng(0)
        e = rng.standard_normal(8).astype(np.float32)
        clip = Clip(uuid=uuid.UUID(int=7), source_video="v.mp4", span=(0.0, 5.0), encoded_data=b"abc")
        clip.aesthetic_score, clip.openai_embedding = score, e + np.float32(emb_shift)
        v = Video(input_video="v.mp4", clips=[] if filtered else [clip], filtered_clips=[clip] if filtered else [])
        t = SplitPipeTask(session_id="s", video=v)
        t.stage_perf["X"] = perf
        return t

    assert C.compare_tasks([task()], [task(perf=9.0)], atol=0.0) == []
    assert C.compare_tasks([task()], [task(emb_shift=5e-4)], atol=1e-3) == []
    bad = C.compare_tasks([task()], [task(emb_shift=5e-3)], atol=1e-3)
    assert [d.field for _, d in bad] == ["videos[0].clips[0].openai_embedding"] and bad[0][1].max_diff_observed == pytest.approx(5e-3, rel=1e-3)
    assert C.compare_tasks([task()], [task(score=4.26)], atol=1e-3)[0][1].field == "videos[0].clips[0].aesthetic_score"  # scalars: exact
    moved = C.compare_tasks([task()], [task(filtered=True)], atol=1e-3)
    assert {d.field for _, d in moved} == {"videos[0].clips", "videos[0].filtered_clips"}
    assert C.compare_tasks([task()], [], atol=0.0)[0][1].field == "tasks"
    assert C.compare_tasks([task()], [task(perf=9.0)], atol=0.0, field_names=None)[0][1].field == "stage_perf.X"  # generic comparator: everything
