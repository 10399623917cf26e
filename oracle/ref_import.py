"""Import the reference's OWN hot-path modules from /root/reference (build container only).

Used by oracle/make_golden.py to produce tests/golden/*; the tests read those vectors and never
call into this module, so they run without a reference checkout.

Two stubs are injected, as established in SURVEY.md 8c / V2:
  * ``av``  (PyAV is not installed; only needed at import time by decoder_utils), and
  * ``cosmos_curate.core.utils.model.model_utils`` (weight-directory lookup; one function).

Test infrastructure only (see oracle/__init__.py).
"""

from __future__ import annotations

import os
import sys
import types
from pathlib import Path

REFERENCE_ROOT = Path(os.environ.get("CURATE_REFERENCE_ROOT", "/root/reference"))
_weights_dirs: dict[str, Path] = {}


def available() -> bool:
    return (REFERENCE_ROOT / "cosmos_curate" / "models" / "clip.py").exists()


def register_weights_dir(model_id: str, path: Path) -> None:
    _weights_dirs[model_id] = Path(path)


def _install_stubs() -> None:
    os.environ.setdefault("CONDA_DEFAULT_ENV", "unified")
    if str(REFERENCE_ROOT) not in sys.path:
        sys.path.insert(0, str(REFERENCE_ROOT))
    if "av" not in sys.modules:
        try:
            import av  # noqa: F401
        except ImportError:
            av_stub = types.ModuleType("av")
            av_stub.VideoFrame = object  # names referenced in annotations only
            container = types.ModuleType("av.container")
            container.InputContainer = object
            av_stub.container = container
            sys.modules["av"] = av_stub
            sys.modules["av.container"] = container
    name = "cosmos_curate.core.utils.model.model_utils"
    if name not in sys.modules:
        stub = types.ModuleType(name)

        def get_local_dir_for_weights_name(weights_name: str) -> Path:
            return _weights_dirs[weights_name]

        stub.get_local_dir_for_weights_name = get_local_dir_for_weights_name
        sys.modules[name] = stub


def decoder_utils():
    _install_stubs()
    import importlib

    return importlib.import_module("cosmos_curate.pipelines.video.utils.decoder_utils")


def clip_module():
    _install_stubs()
    import importlib

    return importlib.import_module("cosmos_curate.models.clip")


def aesthetics_module():
    _install_stubs()
    import importlib

    return importlib.import_module("cosmos_curate.models.aesthetics")


def transnetv2_module():
    _install_stubs()
    import importlib

    return importlib.import_module("cosmos_curate.models.transnetv2")


def transnetv2_stage_functions() -> dict:
    """The module-level shot-logic functions of transnetv2_extraction_stages.py, executed from the reference's source.

    The module itself cannot be imported here (its stage base class needs ray + the cosmos-xenna Rust extension), so the
    function definitions are parsed out of the file under /root/reference and compiled as they stand."""
    import ast
    import math
    from collections.abc import Callable, Generator
    from typing import Literal

    import numpy as np
    import numpy.typing as npt
    import torch

    path = REFERENCE_ROOT / "cosmos_curate" / "pipelines" / "video" / "clipping" / "transnetv2_extraction_stages.py"
    tree = ast.parse(path.read_text())
    wanted = {"_get_batches", "_get_predictions", "_get_scenes", "_get_filtered_scenes", "_crop_scenes", "_create_spans"}
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in wanted]
    assert {n.name for n in body} == wanted
    ns = {"np": np, "npt": npt, "torch": torch, "math": math, "Callable": Callable, "Generator": Generator, "Literal": Literal}
    exec(compile(ast.Module(body=body, type_ignores=[]), str(path), "exec"), ns)  # noqa: S102 - reference code, build container only
    return {k: ns[k] for k in wanted}


def dedup_core():
    """The array section of SemanticDedupActor.dedup (dedup_actor.py, from `norms = cp.linalg.norm(E ...` to `argi[0] = 0`)
    executed from the reference's own source with numpy standing in for cupy (CuPy mirrors the numpy API for every call the
    section makes: linalg.norm, maximum, full, clip, argmax, arange, where, asarray, tril_indices, max).  cudf / cuml / the GPU are
    not needed for this part.  Returns fn(E float32 [m, d] sorted, tile) -> (maxv float32 [m], argi int32 [m])."""
    import ast
    import textwrap

    import numpy as np

    path = REFERENCE_ROOT / "cosmos_curate" / "pipelines" / "video" / "dedup" / "dedup_actor.py"
    lines = path.read_text().splitlines()
    start = next(i for i, ln in enumerate(lines) if ln.strip().startswith("norms = cp.linalg.norm(E, axis=1, keepdims=True)"))
    end = next(i for i, ln in enumerate(lines) if i > start and ln.strip() == "argi[0] = 0")
    block = textwrap.dedent("\n".join(lines[start : end + 1]))
    ast.parse(block)  # must be a self-contained statement list
    src = "def _core(E, TILE, cp):\n    m = E.shape[0]\n" + textwrap.indent(block, "    ") + "\n    return maxv, argi\n"
    ns: dict = {}
    exec(compile(src, str(path), "exec"), ns)  # noqa: S102 - reference code, build container only
    return lambda E, tile=4096: ns["_core"](np.ascontiguousarray(E, dtype=np.float32).copy(), tile, np)


def internvideo2_formulator():
    """An `InternVideo2MultiModality` carrying only what `_construct_frames` / `_construct_image` / `_normalize` read
    (cosmos_curate/models/internvideo2_mm.py:378-415): the reference's own frame formulation, no weights, no tower."""
    _install_stubs()
    import importlib

    import numpy as np

    if "easydict" not in sys.modules:
        try:
            import easydict  # noqa: F401
        except ImportError:
            stub = types.ModuleType("easydict")
            stub.EasyDict = dict  # only used to wrap the tower's config
            sys.modules["easydict"] = stub
    mod = importlib.import_module("cosmos_curate.models.internvideo2_mm")
    obj = object.__new__(mod.InternVideo2MultiModality)
    obj._v_mean = np.array([0.485, 0.456, 0.406], dtype=np.float32).reshape(1, 1, 3)  # setup(), :378-379
    obj._v_std = np.array([0.229, 0.224, 0.225], dtype=np.float32).reshape(1, 1, 3)
    return obj


def fixed_stride_functions():
    """The reference's own span helpers (clip_extraction_stages.py:444-565), executed from its source: the module itself needs ray
    and the Rust extension at import time, these five functions need numpy and uuid only."""
    import ast
    import uuid
    from uuid import UUID

    import numpy as np
    import numpy.typing as npt

    path = REFERENCE_ROOT / "cosmos_curate" / "pipelines" / "video" / "clipping" / "clip_extraction_stages.py"
    tree = ast.parse(path.read_text())
    wanted = {"_validate_video_timestamps", "_get_videos_timestamps", "_get_videos_durations", "_make_spans_fixed_stride", "_make_clip_uuids",
              "_populate_clips_fixed_stride"}  # fmt: skip
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in wanted]
    assert {n.name for n in body} == wanted
    import logging
    import types

    def clip(uuid, source_video, span):  # noqa: A002 - the reference passes these three keywords (:650-654)
        return types.SimpleNamespace(uuid=uuid, source_video=source_video, span=span)

    ns = {"np": np, "npt": npt, "uuid": uuid, "UUID": UUID, "Video": object, "Clip": clip, "logger": logging.getLogger("reference")}
    src = "from __future__ import annotations\n" + "\n\n".join(ast.unparse(n) for n in body)
    exec(compile(src, str(path), "exec"), ns)  # noqa: S102 - reference code, build container only
    return {k: ns[k] for k in wanted}


def grouping_module():
    """cosmos_curate/core/utils/misc/grouping.py (pure Python): split_by_chunk_size is what chunk_tasks sizes its subtasks with."""
    _install_stubs()
    import importlib

    return importlib.import_module("cosmos_curate.core.utils.misc.grouping")


def stage_compare_functions():
    """`_compare_values` and its helpers from the reference's stage-output comparator (core/utils/misc/stage_compare.py:58-66, 173-313),
    executed from source (the module imports ray / xenna at the top; these functions need numpy and attrs only)."""
    import ast
    from collections.abc import Mapping, Sequence
    from typing import Any, cast

    import attrs
    import numpy as np
    import numpy.typing as npt

    path = REFERENCE_ROOT / "cosmos_curate" / "core" / "utils" / "misc" / "stage_compare.py"
    tree = ast.parse(path.read_text())
    wanted = {"FieldDiff", "_compare_arrays", "_compare_attrs", "_compare_mapping", "_compare_sequence", "_compare_values"}
    body = [n for n in tree.body if isinstance(n, (ast.FunctionDef, ast.ClassDef)) and n.name in wanted]
    assert {n.name for n in body} == wanted
    ns = {"np": np, "npt": npt, "attrs": attrs, "Mapping": Mapping, "Sequence": Sequence, "Any": Any, "cast": cast}
    exec(compile(ast.Module(body=body, type_ignores=[]), str(path), "exec"), ns)  # noqa: S102 - reference code, build container only
    return {k: ns[k] for k in wanted}
