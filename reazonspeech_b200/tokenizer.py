"""Tokenizers exposing NeMo's ``tokenizer.ids_to_text`` (the only tokenizer call the reference
makes: pkg/nemo-asr/src/decode.py:41,47) and ``text_to_ids`` (what forced alignment tokenises a transcript with).

``SentencePieceTokenizer`` wraps a real ``tokenizer.model`` from the .nemo archive.
``PieceTableTokenizer`` is the stand-in used with synthetic weights: a deterministic table of
3000 pieces decoded with SentencePiece's rules (concatenate pieces, U+2581 -> space, drop the
leading space) so a bare U+2581 decodes to the empty string exactly like the real model does
(which is why decode.py:51-53 filters empty tokens)."""
from __future__ import annotations

from typing import Iterable, List, Sequence

WORD_BOUNDARY = "▁"


class PieceTableTokenizer:
    def __init__(self, pieces: Sequence[str]):
        self.pieces = list(pieces)

    @property
    def vocab_size(self) -> int:
        return len(self.pieces)

    def ids_to_text(self, ids: Iterable[int]) -> str:
        text = "".join(self.pieces[int(i)] for i in ids).replace(WORD_BOUNDARY, " ")
        return text[1:] if text.startswith(" ") else text

    def ids_to_pieces(self, ids: Iterable[int]) -> List[str]:
        return [self.pieces[int(i)] for i in ids]

    def text_to_ids(self, text: str) -> List[int]:
        """One piece per character: a space becomes the word-boundary piece, a character outside the table the unknown
        piece (id 0).  ``ids_to_text(text_to_ids(s)) == s`` for text of table characters and inner spaces."""
        index = self.__dict__.get("_index")
        if index is None:
            index = self._index = {p: i for i, p in reversed(list(enumerate(self.pieces)))}
        return [index.get(WORD_BOUNDARY if ch == " " else ch, 0) for ch in text]


def synthetic_pieces(vocab_size: int) -> List[str]:
    """Deterministic Japanese-looking piece table: <unk>, the word-boundary mark, punctuation,
    kana, then CJK ideographs from U+4E00."""
    pieces = ["⁇", WORD_BOUNDARY, "。", "、", "?", "!", ","]
    pieces += [chr(c) for c in range(0x3041, 0x3094)]       # hiragana
    pieces += [chr(c) for c in range(0x30A1, 0x30F7)]       # katakana
    c = 0x4E00
    while len(pieces) < vocab_size:
        pieces.append(chr(c))
        c += 1
    return pieces[:vocab_size]


class SentencePieceTokenizer:
    def __init__(self, model_bytes: bytes):
        import sentencepiece as spm
        self.sp = spm.SentencePieceProcessor(model_proto=model_bytes)

    @property
    def vocab_size(self) -> int:
        return self.sp.get_piece_size()

    def ids_to_text(self, ids: Iterable[int]) -> str:
        return self.sp.decode_ids([int(i) for i in ids])

    def text_to_ids(self, text: str) -> List[int]:
        return list(self.sp.encode_as_ids(text))
