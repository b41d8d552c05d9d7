"""CPU-side checks of the window ABI (lh_window_*): struct layout against the header, the interval limit, and the
order in which ShardedEngine folds a snapshot into the window."""
import ctypes
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_window_stats_layout_matches_header(tmp_path):
    from loghisto_b200 import _lib
    cls = _lib.lh_window_stats
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "loghisto_b200.h"', 'int main(void) {',
           'printf("size %zu\\n", sizeof(lh_window_stats));',
           'printf("max %d\\n", LH_MAX_WINDOW_INTERVALS);']
    for f, _ in cls._fields_:
        src.append('printf("%s %%zu\\n", offsetof(lh_window_stats, %s));' % (f, f))
    src.append('return 0; }')
    c = tmp_path / "layout.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(c)],
                   check=True)
    want = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert ctypes.sizeof(cls) == int(want["size"])
    for f, _ in cls._fields_:
        assert getattr(cls, f).offset == int(want[f]), f
    assert int(want["max"]) == _lib.LH_MAX_WINDOW_INTERVALS


def test_window_entry_points_are_declared_and_bound():
    from loghisto_b200 import _lib
    src = open(os.path.join(ROOT, "include", "loghisto_b200.h")).read()
    declared = set(re.findall(r"^LH_API [^;(]*?\b(lh_window_[a-z_]+)\(", src, flags=re.M))
    assert declared == {"lh_window_configure", "lh_window_release", "lh_window_fold", "lh_window_reduce",
                        "lh_window_export", "lh_window_info"}
    assert declared <= set(_lib.SIGNATURES)


class _RecordingEngine:
    """Stands in for Engine: records the calls ShardedEngine makes."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def call(*a, **k):
            self.calls.append(name)
            return ("ticket", 0) if name == "snapshot_reduce_async" else None
        return call


def test_sharded_snapshot_folds_once_between_collective_and_end():
    from loghisto_b200.distributed import ShardedEngine
    eng = _RecordingEngine()
    se = ShardedEngine(eng, 0)
    se.snapshot([0.5], export=True, window=True)
    assert eng.calls == ["snapshot_begin", "window_fold", "snapshot_reduce", "snapshot_export", "snapshot_end"]
    eng.calls.clear()
    se.snapshot_async([0.5], window=True)
    assert eng.calls == ["snapshot_begin", "window_fold", "snapshot_reduce_async", "snapshot_end"]
    eng.calls.clear()
    se.snapshot([0.5])
    se.snapshot_async([0.5])
    assert "window_fold" not in eng.calls
