"""build.py decides from file times whether a translation unit or the library is out of date: every file
that a unit includes must be in its dependency list, or an edit to that file alone keeps the old library."""
import os
import re

import pytest

from ip_mcmc_b200 import build


def _include_closure(src):
    """Every file reached from csrc/<src> through #include "..." (paths normalised)."""
    seen, todo = set(), [os.path.normpath(os.path.join(build.CSRC, src))]
    while todo:
        path = todo.pop()
        if path in seen:
            continue
        seen.add(path)
        with open(path) as f:
            for inc in re.findall(r'^\s*#\s*include\s+"([^"]+)"', f.read(), re.M):
                todo.append(os.path.normpath(os.path.join(os.path.dirname(path), inc)))
    return seen


@pytest.mark.parametrize("src", ["engine.cu", "burgers_inst.cu"])
def test_unit_deps_cover_includes(src):
    assert src in {s for _, s, _ in build.UNITS}
    listed = {os.path.normpath(os.path.join(build.CSRC, f)) for f in [src] + build.DEPS[src]}
    missing = _include_closure(src) - listed
    assert not missing, "build.DEPS[%r] lacks %s" % (src, sorted(os.path.relpath(m, build.CSRC) for m in missing))


@pytest.mark.parametrize("src", ["engine.cu", "burgers_inst.cu"])
def test_library_stale_after_any_included_file_changes(src, tmp_path, monkeypatch):
    lib = tmp_path / "libipmcmc.so"
    lib.write_bytes(b"")
    os.utime(lib, (1, 1))
    monkeypatch.setattr(build, "LIB", str(lib))
    for path in sorted(_include_closure(src)):
        # every source file older than the library except `path`
        monkeypatch.setattr(build, "_mtime",
                            lambda f, p=path: 2 if os.path.normpath(os.path.join(build.CSRC, f)) == p else 0)
        assert build._stale(), "an edit to %s alone does not rebuild the library" % os.path.relpath(path, build.CSRC)
