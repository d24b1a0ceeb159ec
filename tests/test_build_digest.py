"""The rebuild stamp of liblsk.so must follow every file the library is compiled from: a stale
library after an edit to any kernel header would run old code under new source."""
import os
import shutil

import pytest

from layerskip_b200 import build


@pytest.fixture()
def source_copy(tmp_path, monkeypatch):
    csrc = tmp_path / "csrc"
    inc = tmp_path / "include"
    shutil.copytree(build.CSRC, csrc)
    inc.mkdir()
    shutil.copy(os.path.join(build.INCLUDE_DIR, "lsk.h"), inc / "lsk.h")
    monkeypatch.setattr(build, "CSRC", str(csrc))
    monkeypatch.setattr(build, "INCLUDE_DIR", str(inc))
    return csrc, inc


def test_digest_covers_every_source_file(source_copy):
    csrc, inc = source_copy
    inputs = {os.path.basename(p) for p in build._digest_inputs()}
    assert {"engine.cu", "prefill_tc.cuh", "lsk.h"} <= inputs
    assert set(os.listdir(csrc)) <= inputs


def test_digest_changes_when_any_source_file_changes(source_copy):
    csrc, inc = source_copy
    files = [csrc / n for n in sorted(os.listdir(csrc))] + [inc / "lsk.h"]
    base = build._digest()
    for path in files:
        original = path.read_bytes()
        path.write_bytes(original + b"\n// edit\n")
        assert build._digest() != base, f"editing {path.name} leaves the build stamp unchanged"
        path.write_bytes(original)
        assert build._digest() == base


def test_digest_changes_when_a_header_is_added(source_copy):
    csrc, _ = source_copy
    base = build._digest()
    (csrc / "new_kernel.cuh").write_text("#pragma once\n")
    assert build._digest() != base
