"""CPU: the residual-coded synthetic H.264 clips (tools/synth_h264.make_coded_clip) are conforming streams.

libavcodec (cv2) must decode every picture without a single error message, the I_PCM sentinel macroblock that ends every
picture must come back sample-exact (a CAVLC parse error anywhere in a slice would desynchronise everything after it), and
with deblocking off the IDR luma must equal the closed-loop mosaic exactly (every DC level decoded to the intended value).
"""

from __future__ import annotations

import subprocess
import sys
import textwrap

import numpy as np

from conftest import ROOT

_DECODE = textwrap.dedent(
    """
    import sys, os, json
    sys.path.insert(0, sys.argv[1])
    os.environ["OPENCV_FFMPEG_LOGLEVEL"] = "16"   # libavcodec errors to stderr
    import numpy as np, cv2
    from tools import synth_h264 as S
    w, h, fps, secs, deblock = int(sys.argv[2]), int(sys.argv[3]), 30, float(sys.argv[4]), sys.argv[5] == "1"
    mp4, info = S.make_coded_clip(w, h, fps, secs, seed=int(sys.argv[6]), bitrate=float(sys.argv[7]), deblock=deblock,
                                  ac_density=0.25 if deblock else 0.0, return_info=True)
    open(sys.argv[8], "wb").write(mp4)
    cap = cv2.VideoCapture(sys.argv[8])
    cap.set(cv2.CAP_PROP_CONVERT_RGB, 0)
    pcm = info["pcm"][:256].reshape(16, 16)
    rows = h - (h // 16) * 16 or 16   # visible rows of the last macroblock row
    n = ok_sentinel = 0
    idr_exact = []
    while True:
        ok, y = cap.read()
        if not ok:
            break
        ok_sentinel += bool(np.array_equal(y[h - rows:h, w - 16:w][4:], pcm[:rows][4:]))  # rows/cols 0..3 may be deblocked
        if n % fps == 0:
            T = info["mosaics"][n // fps]
            want = np.repeat(np.repeat(T, 16, 0), 16, 1)[:h, :w]
            d = y.astype(int) != want
            d[h - rows:, w - 16:] = False
            idr_exact.append(int(d.sum()))
        n += 1
    print(json.dumps({"frames": n, "sentinel_ok": ok_sentinel, "idr_mismatch": idr_exact, "bitrate": info["bitrate"], "bytes": len(mp4),
                      "coded_share": info["coded_share"]}))
    """
)


def _run(w, h, secs, deblock, seed, bitrate, tmp_path):
    r = subprocess.run([sys.executable, "-c", _DECODE, str(ROOT), str(w), str(h), str(secs), "1" if deblock else "0", str(seed), str(bitrate), str(tmp_path / "coded.mp4")],
                       capture_output=True, text=True, timeout=600)  # fmt: skip
    assert r.returncode == 0, r.stderr[-2000:]
    errs = [line for line in r.stderr.splitlines() if "OPENCV:FFMPEG" in line]
    import json

    return json.loads(r.stdout.strip().splitlines()[-1]), errs


def test_coded_clip_is_conforming_and_closed_loop_exact(tmp_path):
    out, errs = _run(640, 368, 3.0, False, 4, 1.0e6, tmp_path)
    assert errs == []
    assert out["frames"] == 90 and out["sentinel_ok"] == 90
    assert out["idr_mismatch"] == [0, 0, 0]  # deblocking off, DC only: the IDR luma IS the mosaic


def test_coded_clip_1080p_bitrate_and_deblocking(tmp_path):
    out, errs = _run(1920, 1080, 2.0, True, 9, 4.0e6, tmp_path)
    assert errs == []
    assert out["frames"] == 60 and out["sentinel_ok"] == 60  # 1080 = 67.5 macroblock rows: the sentinel is half visible
    assert abs(out["bitrate"] - 4.0e6) / 4.0e6 < 0.12, out  # the reference's transcode default (decoder_utils.py:43)


def test_escape_fast_matches_scalar_rule():
    from tools import synth_h264 as S

    rng = np.random.default_rng(0)
    for _ in range(20):
        a = rng.choice(np.array([0, 0, 0, 1, 2, 3, 4, 255], dtype=np.uint8), size=400)
        assert S._escape_fast(a) == S.escape(a.tobytes())
