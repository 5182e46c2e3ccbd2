"""Result carriers of the B200 path (SURVEY.md section 8 rows a11, b-B0, f4).

``make_result(d)`` returns the reference's own ``stable_whisper.WhisperResult`` when that package is importable (a user
switching over has it installed: regrouping, SRT/VTT/ASS output and every other method keep working), and otherwise the
small ``WhisperResult`` below, which keeps the reference's dict schema (stable_whisper/result.py:618-636 segment dict,
:1398-1406 result dict, :928-949 constructor forms) so that ``to_dict()`` / JSON written here load in the reference and
vice versa.  The same dict is the wire format of the multi-GPU gather (sharding.py: word records -> ``records_to_result``).

Nothing here touches the GPU: these are host objects, as in the reference.
"""
import json
from dataclasses import dataclass
from typing import Any, List, Optional, Union

SEGMENT_KEYS = ("start", "end", "text", "seek", "tokens", "temperature", "avg_logprob", "compression_ratio", "no_speech_prob")


def reference_result_class():
    """stable_whisper.WhisperResult if the reference package can be imported, else None."""
    try:
        from stable_whisper.result import WhisperResult as Ref
        return Ref
    except Exception:
        return None


@dataclass
class WordTiming:                     # stable_whisper/result.py WordTiming (the fields to_dict emits)
    word: str
    start: float
    end: float
    probability: Optional[float] = None
    tokens: Optional[List[int]] = None
    segment_id: Optional[int] = None
    id: Optional[int] = None

    @property
    def duration(self) -> float:
        return round(self.end - self.start, 3)

    def to_dict(self) -> dict:
        return dict(word=self.word, start=self.start, end=self.end, probability=self.probability,
                    tokens=None if self.tokens is None else list(self.tokens))


@dataclass
class Segment:                        # stable_whisper/result.py Segment
    start: Optional[float] = None
    end: Optional[float] = None
    text: Optional[str] = None
    seek: Optional[float] = None
    tokens: Optional[List[int]] = None
    temperature: Optional[float] = None
    avg_logprob: Optional[float] = None
    compression_ratio: Optional[float] = None
    no_speech_prob: Optional[float] = None
    words: Optional[List[WordTiming]] = None
    id: Optional[int] = None

    def __post_init__(self):
        if self.words is not None:
            self.words = [w if isinstance(w, WordTiming) else
                          WordTiming(**{k: w.get(k) for k in ("word", "start", "end", "probability", "tokens")}) for w in self.words]
            self._sync()

    def _sync(self):
        if self.words:                # a segment with words takes its text, span and tokens from them (result.py Segment.text/
            self.text = "".join(w.word for w in self.words)     # start/end/tokens: the timestamp tokens are not listed)
            self.start, self.end = self.words[0].start, self.words[-1].end
            if self.words[0].tokens:
                self.tokens = [t for w in self.words for t in w.tokens]

    @property
    def has_words(self) -> bool:
        return bool(self.words)

    @property
    def duration(self) -> float:
        return round((self.end or 0.0) - (self.start or 0.0), 3)

    def to_dict(self) -> dict:
        d = {k: getattr(self, k) for k in SEGMENT_KEYS}
        d["tokens"] = None if self.tokens is None else list(self.tokens)
        if self.words is not None:
            d["words"] = [w.to_dict() for w in self.words]
        return d


class WhisperResult:
    """Schema-compatible stand-in for stable_whisper.WhisperResult (result.py:928): ``segments``, ``text``, ``language``,
    ``all_words()``, ``to_dict()``, ``save_as_json()``; accepts the constructor forms of result.py:957-990
    (dict | list of segment dicts | list of word-dict lists | path of a JSON file)."""

    def __init__(self, result: Union[str, dict, list]):
        self.path = None
        if isinstance(result, str):
            self.path = result
            with open(result, "r", encoding="utf-8") as f:
                result = json.load(f)
        if isinstance(result, list):
            if result and isinstance(result[0], list):
                result = dict(segments=[dict(start=ws[0]["start"], end=ws[-1]["end"], text="".join(w["word"] for w in ws), words=ws)
                                        for ws in result if ws])
            else:
                result = dict(segments=result)
        if not isinstance(result, dict):
            raise TypeError(f"Expect result to be dict, list or str but got {type(result)}")
        self.ori_dict = result.get("ori_dict") or result
        self.language = self.ori_dict.get("language")
        self._regroup_history = result.get("regroup_history", "")
        self._nonspeech_sections = result.get("nonspeech_sections") or []
        self.unfinished_start = result.get("unfinished", -1.0)
        segs = result.get("segments", self.ori_dict.get("segments")) or []
        self.segments = [Segment(**{k: s.get(k) for k in (*SEGMENT_KEYS, "words")}) for s in segs]
        if any(s.has_words for s in self.segments):           # remove_no_word_segments (result.py:946)
            self.segments = [s for s in self.segments if s.has_words]
        self.reassign_ids()

    def reassign_ids(self):
        for i, s in enumerate(self.segments):
            s.id = i
            for j, w in enumerate(s.words or []):
                w.segment_id, w.id = i, j

    def __getitem__(self, i: int) -> Segment:
        return self.segments[i]

    def __len__(self) -> int:
        return len(self.segments)

    @property
    def text(self) -> str:
        return "".join(s.text or "" for s in self.segments)

    @property
    def has_words(self) -> bool:
        return bool(self.segments) and all(s.has_words for s in self.segments)

    @property
    def duration(self) -> float:
        return round(self.segments[-1].end - self.segments[0].start, 3) if self.segments else 0.0

    def all_words(self) -> List[WordTiming]:
        return [w for s in self.segments for w in (s.words or [])]

    def all_tokens(self) -> List[int]:
        return [t for w in self.all_words() for t in (w.tokens or [])]

    def segments_to_dicts(self) -> List[dict]:
        return [s.to_dict() for s in self.segments]

    def to_dict(self, keep_orig: bool = True) -> dict:          # result.py:1398-1406
        return dict(text=self.text, segments=self.segments_to_dicts(), language=self.language,
                    ori_dict=self.ori_dict if keep_orig else {}, regroup_history=self._regroup_history,
                    nonspeech_sections=self._nonspeech_sections, unfinished=self.unfinished_start)

    def save_as_json(self, path: str, ensure_ascii: bool = False, **kw):
        d = self.to_dict(keep_orig=False)
        with open(path if path.endswith(".json") else path + ".json", "w", encoding="utf-8") as f:
            json.dump(d, f, ensure_ascii=ensure_ascii, **kw)


def make_result(d: Union[dict, list], prefer_reference: bool = True):
    """dict(text, segments, language) -> the reference's WhisperResult when importable, else the stand-in above."""
    Ref = reference_result_class() if prefer_reference else None
    return Ref(d) if Ref is not None else WhisperResult(d)


def result_to_dict(result: Any) -> dict:
    """WhisperResult (either class) | dict | list of segment dicts -> plain dict(text, segments, language)."""
    if hasattr(result, "to_dict"):
        try:
            return result.to_dict(keep_orig=False)
        except TypeError:
            return result.to_dict()
    if isinstance(result, dict):
        return result
    return dict(segments=list(result))


def result_segments(result: Any) -> List[dict]:
    return list(result_to_dict(result).get("segments") or [])
