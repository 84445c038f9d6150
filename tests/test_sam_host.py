"""The SAM rule's Python statement (sam_utils.read_header / iter_records), its errors and refusals, and the sam2ec
command line; no GPU.  Every single-sample golden BAM, rendered as SAM, reads back as the BAM file's records."""
import io
import os

import pytest
from click.testing import CliRunner

from conftest import GOLDEN, golden_cases
from alntools_b200 import bam_io, sam_utils
from sam_render import sam_text

REFS = ("T1_A", "T1_B", "T2_A", "T2_B")
LENS = (100, 100, 200, 200)


def _stream(text):
    return io.BufferedReader(io.BytesIO(text))


def _read(text, name="x.sam"):
    s = _stream(text)
    refs, lengths, n = sam_utils.read_header(s, name)
    return refs, lengths, n, list(sam_utils.iter_records(s, refs, n + 1, name))


def _line(*fields):
    return b"\t".join(f if isinstance(f, bytes) else str(f).encode() for f in fields)


HEAD = (b"@HD\tVN:1.6\n@SQ\tSN:T1_A\tLN:100\tAS:x\n@CO\tfree text\n@SQ\tLN:100\tSN:T1_B\n"
        b"@SQ\tSN:T2_A\tLN:200\n@PG\tID:bwa\n@SQ\tSN:T2_B\tLN:200\n")


def test_header_and_lines():
    body = [_line("r1", 99, "T1_A", 5, 255, "10M", "=", 40, 45, "ACGTACGTAC", "*", "NM:i:0"),
            _line("r1 extra", 147, "T1_A", 40, 255, "10M", "T1_A", 5, -45, "*", "*"),
            _line(" lead", 0, "T2_B", 1, 0, "*", "*", 0, 0, "*", "*"),
            _line("r2", 4, "*", 0, 0, "*", "*", 0, 0, "*", "*"),
            _line("r3", 1, "T1_B", 7, 0, "*", "T2_A", 0, 0, "*", "*\r")]
    refs, lengths, n, recs = _read(HEAD + b"\n".join(body))      # the last line has no '\n'
    assert refs == REFS and lengths == LENS and n == 7
    assert recs == [("r1", 99, 0, 4, 0, 39), ("r1 extra", 147, 0, 39, 0, 4), (" lead", 0, 3, 0, -1, -1),
                    ("r2", 4, -1, -1, -1, -1), ("r3", 1, 1, 6, 2, -1)]


def test_empty_body_and_no_header():
    assert _read(HEAD) == (REFS, LENS, 7, [])
    assert _read(b"") == ((), (), 0, [])
    assert _read(_line("q", 4, "*", 0, 0, "*", "*", 0, 0, "*", "*") + b"\n")[3] == [("q", 4, -1, -1, -1, -1)]


GOOD = _line("g", 0, "T1_A", 1, 0, "*", "*", 0, 0, "*", "*")
BAD = [
    (b"@SQ\tSN:late\tLN:5", "a header line (starting with '@') after the first alignment line"),
    (b"", "fewer than 11 tab-separated fields"),
    (_line("a", 0, "T1_A", 1, 0, "*", "*", 0, 0, "*"), "fewer than 11 tab-separated fields"),
    (_line("", 0, "T1_A", 1, 0, "*", "*", 0, 0, "*", "*"), "QNAME empty or longer than 254 bytes"),
    (_line("q" * 255, 0, "T1_A", 1, 0, "*", "*", 0, 0, "*", "*"), "QNAME empty or longer than 254 bytes"),
    (_line("a", 65536, "T1_A", 1, 0, "*", "*", 0, 0, "*", "*"), "FLAG not a decimal integer in [0, 65535]"),
    (_line("a", "0x4", "T1_A", 1, 0, "*", "*", 0, 0, "*", "*"), "FLAG not a decimal integer in [0, 65535]"),
    (_line("a", 0, "T9", 1, 0, "*", "*", 0, 0, "*", "*"), "RNAME not '*' and not an @SQ name"),
    (_line("a", 0, "=", 1, 0, "*", "*", 0, 0, "*", "*"), "RNAME not '*' and not an @SQ name"),
    (_line("a", 0, "T1_A", -1, 0, "*", "*", 0, 0, "*", "*"), "POS not a decimal integer in [0, 2147483647]"),
    (_line("a", 0, "T1_A", 2 ** 31, 0, "*", "*", 0, 0, "*", "*"), "POS not a decimal integer in [0, 2147483647]"),
    (_line("a", 0, "T1_A", 1, 0, "*", "T7", 0, 0, "*", "*"), "RNEXT not '*', '=' or an @SQ name"),
    (_line("a", 0, "T1_A", 1, 0, "*", "*", "", 0, "*", "*"), "PNEXT not a decimal integer in [0, 2147483647]"),
    (_line("a", 0, "*", 0, 0, "*", "*", 0, 0, "*", "*"),
     "alignment with reference id -1 outside the header's 4 references"),
]


@pytest.mark.parametrize("line,what", BAD, ids=[str(i) for i in range(len(BAD))])
def test_every_bad_line_names_input_and_line(line, what):
    text = HEAD + GOOD + b"\n" + GOOD + b"\n" + line + b"\n" + GOOD + b"\n"
    with pytest.raises(ValueError) as err:
        _read(text, "in.sam")
    assert str(err.value) == "in.sam: line 10: %s" % what


def test_unmapped_or_filtered_star_is_not_an_error():
    lines = [_line("a", 4, "*", 0, 0, "*", "*", 0, 0, "*", "*"),          # unmapped
             _line("b", 1 | 0x80 | 2, "*", 0, 0, "*", "*", 0, 0, "*", "*"),  # read 2 of a pair
             _line("c", 1 | 2, "*", 0, 0, "*", "T1_A", 0, 0, "*", "*")]     # mate elsewhere
    assert len(_read(HEAD + b"\n".join(lines))[3]) == 3


@pytest.mark.parametrize("line", [b"@SQ\tLN:5", b"@SQ\tSN:x", b"@SQ\tSN:x\tLN:5k", b"@SQ\tSN:x\tLN:-5", b"@SQ"])
def test_bad_sq_line(line):
    with pytest.raises(ValueError) as err:
        _read(b"@HD\tVN:1.6\n" + line + b"\n")
    assert "x.sam: line 2: @SQ line without SN: or without a decimal LN:" in str(err.value)


def test_gzip_input_is_refused(tmp_path):
    path = str(tmp_path / "x.bam")
    bam_io.write_bam(path, [("T1_A", 100)], [("r", 0, 0)])
    with open(path, "rb") as fh, pytest.raises(ValueError) as err:
        sam_utils.read_header(fh, path)
    assert "bam2ec" in str(err.value)


def _no_builder(monkeypatch):
    def refuse(*a, **k):
        raise AssertionError("a builder was made")
    monkeypatch.setattr(sam_utils, "EcBuilder", refuse)


@pytest.mark.parametrize("line,what", BAD[:3] + BAD[-1:], ids=["at", "empty", "fields", "tid"])
def test_bad_line_writes_nothing(line, what, tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_EMITTER", "python")
    _no_builder(monkeypatch)
    sam, out = str(tmp_path / "in.sam"), str(tmp_path / "out.bin")
    with open(sam, "wb") as fh:
        fh.write(HEAD + GOOD + b"\n" + line + b"\n")
    with pytest.raises(ValueError) as err:
        sam_utils.convert_sam(sam, out)
    assert str(err.value) == "%s: line 9: %s" % (sam, what)
    assert not os.path.exists(out)


@pytest.mark.parametrize("env,out,rangefile", [
    ({}, "x.h5", None),
    ({"ALNTOOLS_GPUS": "2"}, "x.bin", None),
    ({"ALNTOOLS_B200_COLLATE": "1"}, "x.bin", None),
    ({"ALNTOOLS_B200_EMITTER": "python"}, "x.bin", "r.txt"),
], ids=["h5", "gpus", "collate", "python_rangefile"])
def test_refusals_come_before_the_input_is_read(env, out, rangefile, tmp_path, monkeypatch):
    for key, value in env.items():
        monkeypatch.setenv(key, value)
    _no_builder(monkeypatch)
    with pytest.raises(NotImplementedError):
        sam_utils.convert_sam(str(tmp_path / "missing.sam"), str(tmp_path / out),
                              range_filename=None if rangefile is None else str(tmp_path / rangefile))


def test_decode_setting_is_not_read(tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_DECODE", "bogus")
    monkeypatch.setenv("ALNTOOLS_B200_EMITTER", "python")
    _no_builder(monkeypatch)
    sam = str(tmp_path / "in.sam")
    with open(sam, "wb") as fh:
        fh.write(HEAD + _line("a", 0, "T1_A", 1, 0, "*", "*", 0, 0, "*", "*") + b"\n")
    with pytest.raises(AssertionError, match="a builder was made"):
        sam_utils.convert_sam(sam, str(tmp_path / "o.bin"))


def test_command_line_options(tmp_path, monkeypatch):
    from alntools_b200 import sam2ec
    seen = []
    monkeypatch.setattr(sam_utils, "convert_sam", lambda *a, **k: seen.append((a, k)))
    targets = str(tmp_path / "t.txt")
    with open(targets, "w") as fh:
        fh.write("T1\n")
    res = CliRunner().invoke(sam2ec.sam2ec, ["-", str(tmp_path / "o.bin"), "-s", "S1", "-t", targets,
                                            "--rangefile", str(tmp_path / "r.txt"), "-v"])
    assert res.exit_code == 0, res.output
    (args, kw), = seen
    assert args == ("-", str(tmp_path / "o.bin"))
    assert kw == {"range_filename": str(tmp_path / "r.txt"), "sample": "S1", "target_filename": targets}
    res = CliRunner().invoke(sam2ec.sam2ec, ["in.sam", str(tmp_path / "o.bin")])
    assert res.exit_code == 0 and seen[-1][1] == {"range_filename": None, "sample": None, "target_filename": None}


def _single_golden_bams():
    return sorted({c["bam"] for c in golden_cases("single")})


@pytest.mark.parametrize("bam", _single_golden_bams())
@pytest.mark.parametrize("read_len", [0, 100])
def test_golden_bams_rendered_as_sam_read_back_as_their_records(bam, read_len):
    raw = bam_io.inflate_file(os.path.join(GOLDEN, bam))
    header = bam_io.parse_header(raw)
    want = list(bam_io.iter_records(raw, header.records_offset))
    refs, lengths, n, got = _read(sam_text(header.references, header.lengths, want, read_len))
    assert refs == header.references and lengths == header.lengths and n == len(refs) + 2
    assert got == want
