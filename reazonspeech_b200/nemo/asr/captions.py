"""Read SubRip (.srt) and WebVTT (.vtt) caption files into ``Caption`` objects, for re-timing them against their audio
(``align_captions``, the CLI's ``--align-captions``).

A file is WebVTT when its first non-empty line, after an optional byte-order mark, is ``WEBVTT`` (anything may follow on
that line); otherwise it is SubRip.  A cue is a block of lines separated from the next by a blank line: an optional cue
number or identifier, the timing line ``START --> END`` (``HH:MM:SS,mmm`` in SubRip, ``HH:MM:SS.mmm`` or ``MM:SS.mmm`` in
WebVTT; WebVTT cue settings after END are ignored), then the text lines, joined with one space.  WebVTT ``NOTE``, ``STYLE``
and ``REGION`` blocks and the header block are skipped.  CRLF and CR line endings are accepted."""
from __future__ import annotations

import re
from typing import List

from .interface import Caption

_TIME = re.compile(r"^(?:(\d+):)?(\d{1,2}):(\d{1,2})[.,](\d{1,3})$")
_SKIP_VTT = ("NOTE", "STYLE", "REGION")


def parse_timestamp(text: str) -> float:
    """``[H+:]MM:SS(.|,)mmm`` -> seconds."""
    m = _TIME.match(text.strip())
    if m is None:
        raise ValueError(f"not a caption timestamp: {text!r}")
    h, mnt, sec, frac = m.groups()
    return int(h or 0) * 3600 + int(mnt) * 60 + int(sec) + int(frac.ljust(3, "0")) / 1000.0


def parse_captions(text: str) -> List[Caption]:
    """The cues of an SRT or WebVTT document (see the module docstring), in file order."""
    text = text.lstrip("\ufeff").replace("\r\n", "\n").replace("\r", "\n")
    lines = text.split("\n")
    first = next((l.strip() for l in lines if l.strip()), "")
    vtt = first == "WEBVTT" or first.startswith(("WEBVTT ", "WEBVTT\t"))
    blocks, cur = [], []
    for line in lines:
        if line.strip():
            cur.append(line.strip())
        elif cur:
            blocks.append(cur)
            cur = []
    if cur:
        blocks.append(cur)
    out: List[Caption] = []
    for i, block in enumerate(blocks):
        if vtt and (i == 0 and block[0].startswith("WEBVTT") or block[0].split(" ")[0] in _SKIP_VTT):
            continue
        k = next((j for j, l in enumerate(block[:2]) if "-->" in l), None)
        if k is None:
            continue                                     # not a cue (stray text): nothing to time
        start, _, rest = block[k].partition("-->")
        end = rest.split()[0] if rest.split() else ""
        out.append(Caption(parse_timestamp(start), parse_timestamp(end), " ".join(block[k + 1:])))
    return out


def read_captions(path: str) -> List[Caption]:
    """The cues of the SRT or WebVTT file at ``path`` (UTF-8)."""
    with open(path, encoding="utf-8") as f:
        return parse_captions(f.read())
