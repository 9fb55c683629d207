"""Command line of the drop-in package: ``python -m reazonspeech_b200.nemo.asr.cli [options] AUDIO [AUDIO ...]``.

Same contract as the reference's ``reazonspeech-nemo-asr`` entry point (pkg/nemo-asr/src/cli.py:36-74):

  -h / --help          usage on stderr, nothing else happens
  -o FILE / --output=  where the transcript goes (default: stdout)
  --to=FMT             vtt | srt | ass | json | tsv; anything else, or no option, gives the bracketed plain-text
                       lines.  Like the reference, the format is NOT inferred from FILE's extension
                       (see writer.get_writer)
  no AUDIO argument    "no audio file specified" + usage on stderr, exit status 1
  unknown option       getopt.GetoptError propagates, as in the reference
  --align=FILE         forced alignment instead of recognition: FILE holds one transcript line per AUDIO argument, in
                       order; the segments are timed by where the audio says that text.  A line count that differs from
                       the number of AUDIO arguments prints a message on stderr, exit status 1
  --align-captions=FILE
                       re-time the captions of an SRT or WebVTT FILE against exactly one AUDIO argument: each caption is
                       searched for from 25 s before its start time to its end time (live captions lag the speech) and
                       written as one segment with the times where the audio says it.  Captions that cannot be placed are
                       skipped and counted on stderr.  More or fewer than one AUDIO argument, or --align as well, prints
                       a message on stderr, exit status 1

One extension: several AUDIO arguments are transcribed as one batch on the GPU (the reference reads exactly one);
their segments are written one file after the other through the same writer, every file's times shifted by the total
duration of the files before it, i.e. the transcript of the files played back to back (subtitle formats need monotonic times).
Audio decoding: soundfile when installed, scipy for WAV, librosa for compressed containers, see audio.audio_from_path.
"""
import dataclasses
import getopt
import sys
import warnings
from dataclasses import dataclass, field
from typing import List, Optional

SHORT_OPTS = "ho:"
LONG_OPTS = ("help", "output=", "to=", "align=", "align-captions=")


@dataclass
class Options:
    help: bool = False
    output: Optional[str] = None
    fmt: Optional[str] = None
    audio: List[str] = field(default_factory=list)
    align: Optional[str] = None
    align_captions: Optional[str] = None


def parse(argv) -> Options:
    parsed, rest = getopt.getopt(list(argv), SHORT_OPTS, LONG_OPTS)
    opt = Options(audio=rest)
    for flag, value in parsed:
        if flag in ("-h", "--help"):
            opt.help = True
            break                                            # the reference returns at the first -h it meets
        if flag in ("-o", "--output"):
            opt.output = value
        if flag == "--to":
            opt.fmt = value
        if flag == "--align":
            opt.align = value
        if flag == "--align-captions":
            opt.align_captions = value
    return opt


def usage() -> None:
    print(__doc__, file=sys.stderr)


def read_transcripts(path: str) -> List[str]:
    with open(path, encoding="utf-8") as f:
        return [line.rstrip("\r\n") for line in f]


def run(opt: Options, transcripts: Optional[List[str]] = None) -> None:
    from .audio import audio_from_path
    from .transcribe import align_batch, load_model, transcribe, transcribe_batch
    from .writer import get_writer

    sink = sys.stdout if opt.output is None else open(opt.output, "w")
    warnings.simplefilter("ignore")
    clips = [audio_from_path(path) for path in opt.audio]
    if transcripts is not None:
        results = align_batch(load_model(aligner=True), clips, transcripts)
    else:
        model = load_model()
        results = transcribe_batch(model, clips) if len(clips) > 1 else [transcribe(model, clips[0])]
    with sink:
        out = get_writer(sink, opt.fmt)
        out.write_header()
        offset = 0.0
        for clip, result in zip(clips, results):
            for segment in result.segments:
                out.write(segment if offset == 0.0 else
                          dataclasses.replace(segment, start_seconds=segment.start_seconds + offset, end_seconds=segment.end_seconds + offset))
            offset += clip.seconds


def run_captions(opt: Options) -> None:
    from .audio import audio_from_path
    from .captions import read_captions
    from .interface import Segment
    from .transcribe import align_captions, load_model
    from .writer import get_writer

    captions = read_captions(opt.align_captions)
    sink = sys.stdout if opt.output is None else open(opt.output, "w")
    warnings.simplefilter("ignore")
    placed = align_captions(load_model(aligner=True), audio_from_path(opt.audio[0]), captions)
    with sink:
        out = get_writer(sink, opt.fmt)
        out.write_header()
        for r in placed:
            if r is not None:
                out.write(Segment(r.start_seconds, r.end_seconds, r.text))
    missing = sum(r is None for r in placed)
    if missing:
        print(f"{opt.align_captions}: {missing} of {len(placed)} captions could not be placed and were skipped", file=sys.stderr)


def main(argv=None):
    opt = parse(sys.argv[1:] if argv is None else argv)
    if opt.help:
        usage()
        return None
    if not opt.audio:
        print("no audio file specified", file=sys.stderr)
        usage()
        return 1
    if opt.align_captions is not None:
        if opt.align is not None:
            print("--align-captions and --align cannot be combined", file=sys.stderr)
            return 1
        if len(opt.audio) != 1:
            print(f"--align-captions re-times one audio file, got {len(opt.audio)}", file=sys.stderr)
            return 1
        run_captions(opt)
        return None
    transcripts = None
    if opt.align is not None:
        transcripts = read_transcripts(opt.align)
        if len(transcripts) != len(opt.audio):
            print(f"{opt.align}: {len(transcripts)} transcript lines for {len(opt.audio)} audio files (--align wants one line per file)",
                  file=sys.stderr)
            return 1
    run(opt, transcripts)
    return None


if __name__ == "__main__":
    sys.exit(main())
