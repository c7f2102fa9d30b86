"""The object list the test harnesses link: one object per library source, never an object whose source is gone."""
import os

import pytest

from tests.util import library_objects


def test_library_objects_follow_the_sources(tmp_path):
    csrc = tmp_path / "csrc"
    (csrc / "_build").mkdir(parents=True)
    for stem in ("b", "a"):
        (csrc / f"{stem}.cu").write_text("")
        (csrc / "_build" / f"{stem}.o").write_text("")
    (csrc / "_build" / "removed.o").write_text("")  # left behind by a source deleted since the last build
    assert library_objects(str(csrc)) == [os.path.join(str(csrc), "_build", f"{s}.o") for s in ("a", "b")]
    os.remove(csrc / "_build" / "b.o")
    with pytest.raises(AssertionError, match="b.o"):
        library_objects(str(csrc))
