"""ALNTOOLS_B200_MAX_READ (emitter.max_read): the longest read a conversion accepts.  No GPU needed: bad values are
refused before any file is opened."""
import os

import pytest

from alntools_b200 import bam_utils, bam_utils_multisample, emitter

ENV = "ALNTOOLS_B200_MAX_READ"


@pytest.mark.parametrize("value", ["-1", "abc", "1e6", "1.5", "16 k", "０", "0x4000"])
def test_bad_value_is_refused_before_any_file_is_opened(value, tmp_path, monkeypatch):
    monkeypatch.setenv(ENV, value)
    missing = str(tmp_path / "missing.bam")
    out = str(tmp_path / "x.bin")
    for call in (lambda: bam_utils.convert(missing, out, None),
                 lambda: bam_utils.convert(missing, out, None, collate=True),
                 lambda: bam_utils.convert(missing, out, None, decode="device"),
                 lambda: bam_utils_multisample.convert_files([missing], out, None, 1),
                 lambda: bam_utils_multisample.convert(str(tmp_path / "missing_dir"), out, None, 0, 1, 1, None, None,
                                                       None)):
        with pytest.raises(ValueError, match=ENV):
            call()
    assert not os.path.exists(out)


def test_values(monkeypatch):
    for value, want in ((None, 16384), ("", 16384), ("0", 0), (" 20000 ", 20000), ("16384", 16384),
                        (str((1 << 31) - 8192), (1 << 31) - 8192)):
        if value is None:
            monkeypatch.delenv(ENV, raising=False)
        else:
            monkeypatch.setenv(ENV, value)
        assert emitter.max_read() == want


def test_builder_option_name():
    from alntools_b200 import _native
    assert _native.EcBuilder._OPTIONS["max_read"] == _native.ECB_OPT_MAX_READ == 13
    names = [n for n, _ in _native.EcbStats._fields_]
    assert names[-2:] == ["long_reads", "long_ms"]
