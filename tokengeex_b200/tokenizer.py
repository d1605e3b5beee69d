"""``tokengeex.Tokenizer`` — the reference's Python surface, served by the B200 hot path.

Mirrors /root/reference/bindings/python/src/lib.rs:39-224 (stub: bindings/python/tokengeex.pyi)
over /root/reference/src/tokenizer.rs: same class and method names, argument meaning, return
types and error text (``TokenGeeXError(str(tokengeex::Error))``).  Everything string-shaped
(JSON v"2.0", special-token splitting, decode, id <-> token lookups) is host logic here;
``Model::encode`` — the hot loop — runs on the GPU through the C ABI (``_native.Model``).
There is no CPU encode path: without a CUDA device encode* raises TokenGeeXError.
"""
from __future__ import annotations

import base64
import json
import os
import secrets
import threading
import unicodedata
from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np

from . import _native as N


class TokenGeeXError(Exception):
    """Base class for exceptions raised by TokenGeeX (bindings/python/src/lib.rs:9)."""


SERIALIZATION_VERSION = "2.0"  # src/tokenizer.rs:349


# ---- f64 formatting as serde_json does it (ryu, shortest round-trip) ---------------------------------
def fmt_f64(x: float) -> str:
    if x != x or x in (float("inf"), float("-inf")):
        return "null"  # serde_json writes non-finite floats as null
    r = repr(float(x))
    sign = ""
    if r.startswith("-"):
        sign, r = "-", r[1:]
    mant, _, exp = r.partition("e")
    e10 = int(exp) if exp else 0
    ip, _, fp = mant.partition(".")
    digits = (ip + fp).lstrip("0")
    if not digits:
        return sign + "0.0"
    stripped = digits.rstrip("0")
    k = e10 - len(fp) + (len(digits) - len(stripped))  # value = int(stripped) * 10^k
    digits = stripped
    n = len(digits)
    kk = n + k
    if 0 <= k and kk <= 16:    # 1234e7 -> 12340000000.0
        return sign + digits + "0" * k + ".0"
    if 0 < kk <= 16:           # 1234e-2 -> 12.34
        return sign + digits[:kk] + "." + digits[kk:]
    if -5 < kk <= 0:           # 1234e-6 -> 0.001234
        return sign + "0." + "0" * (-kk) + digits
    m = digits[0] + ("." + digits[1:] if n > 1 else "")
    return f"{sign}{m}e{kk - 1}"


def _jstr(s: str) -> str:
    return json.dumps(s, ensure_ascii=False)


class _Processor:
    def __init__(self, kind: str, form: Optional[str] = None):
        self.kind, self.form = kind, form

    def preprocess(self, s: str) -> str:
        if self.kind == "crlf":
            return s.replace("\r\n", "\n")  # src/processor.rs:47-49
        return unicodedata.normalize(self.form.upper(), s)  # src/processor.rs:127-132

    def to_json(self) -> dict:
        return {"type": "crlf"} if self.kind == "crlf" else {"type": "unicode", "form": self.form}

    @staticmethod
    def from_json(obj) -> "_Processor":
        # #[serde(untagged)] with Crlf tried first; Crlf's visitor ignores unknown keys, so any object
        # whose "type" is absent or "crlf" is a CrlfProcessor (src/processor.rs:13-18,87-101; quirk Q18)
        if not isinstance(obj, dict):
            raise TokenGeeXError("data did not match any variant of untagged enum ProcessorWrapper")
        t = obj.get("type", "crlf")
        if t == "crlf":
            return _Processor("crlf")
        if t == "unicode" and set(obj) <= {"type", "form"} and obj.get("form") in ("nfc", "nfd", "nfkc", "nfkd"):
            return _Processor("unicode", obj["form"])
        raise TokenGeeXError("data did not match any variant of untagged enum ProcessorWrapper")


def split_special_tokens(text: str, special_tokens: Sequence[str]) -> List[Tuple[str, bool]]:
    """SpecialTokenSplitter (src/tokenizer.rs:299-347): at every char boundary the specials are tried
    in LIST order (first in the list wins, not the longest)."""
    out: List[Tuple[str, bool]] = []
    cursor, n = 0, len(text)
    specials = [s for s in special_tokens]
    while cursor < n:
        hit = None
        if specials:
            i = cursor
            while i < n and hit is None:
                for sp in specials:
                    # NB: str.startswith("") is true in Rust as well: an empty special token matches at once
                    if text.startswith(sp, i):
                        hit = (i, sp)
                        break
                if hit is None:
                    i += 1
        if hit is None:
            out.append((text[cursor:], False))
            break
        i, sp = hit
        if i > cursor:
            out.append((text[cursor:i], False))
            cursor = i
        else:
            out.append((sp, True))
            cursor += len(sp)
            if len(sp) == 0:  # an empty special token would never advance in the reference either
                raise TokenGeeXError("empty special token")
    return out


def id_rows(ids: np.ndarray, id_off: np.ndarray) -> List[List[int]]:
    """The ids of a batch as the `Vec<Vec<u32>>` of src/tokenizer.rs:93-123 turned into Python lists: row i =
    ids[id_off[i]:id_off[i + 1]].  Building 10^7 Python ints is what `encode_batch` costs above the GPU call, so each
    list is built once: per row for rows of some length (measured: 0.65 s against 1.15 s for 18 M ids in 10 803 rows),
    one conversion of the whole batch and list slices when the rows are a few ids each (numpy's per-slice cost)."""
    cut = id_off.tolist()
    n = len(cut) - 1
    if len(ids) >= 8 * n:
        return [ids[cut[i]:cut[i + 1]].tolist() for i in range(n)]
    flat = ids.tolist()
    return [flat[cut[i]:cut[i + 1]] for i in range(n)]


def corpus_layout(ids: np.ndarray, id_off: np.ndarray, sep_id: int, dt: np.dtype) -> Tuple[np.ndarray, np.ndarray]:
    """u32 ids + offsets → the output of encode_corpus: ids as `dt`, `sep_id` (if >= 0) after every sample."""
    id_off = np.asarray(id_off, np.uint64)
    if sep_id < 0:
        return np.asarray(ids).astype(dt), id_off.copy()
    S = len(id_off) - 1
    lens = np.diff(id_off).astype(np.int64)
    out = np.empty(len(ids) + S, dt)
    rows = np.repeat(np.arange(S, dtype=np.int64), lens)
    out[np.arange(len(ids), dtype=np.int64) + rows] = ids
    out[id_off[1:].astype(np.int64) + np.arange(S, dtype=np.int64)] = sep_id
    return out, id_off + np.arange(S + 1, dtype=np.uint64)


class Tokenizer:
    """tokengeex.Tokenizer (bindings/python/tokengeex.pyi:10-255)."""

    def __init__(self, tokens: Sequence[bytes], scores, keep=None, processors: Sequence[_Processor] = (),
                 special_tokens: Sequence[str] = (), device: Optional[int] = None):
        self._tokens: List[bytes] = list(tokens)
        self._scores = np.ascontiguousarray(scores, np.float64).copy()
        self._keep = np.zeros(len(self._tokens), np.uint8) if keep is None else np.asarray(keep, np.uint8).copy()
        self._processors = list(processors)
        self._special: List[str] = []
        self._special_map = {}
        self._token_to_id = {}
        for i, t in enumerate(self._tokens):
            self._token_to_id[t] = i  # HashMap::insert: the last duplicate wins (src/model.rs:20-23)
        self.add_special_tokens(special_tokens)
        self._device = device if device is not None else int(os.environ.get("TGX_DEVICE", "0"))
        self._model: Optional[N.Model] = None          # device model, created on first encode
        self._model_bytes_only: Optional[N.Model] = None  # dropout >= 1.0: multi-byte tokens never match
        # 0 < dropout < 1: None = a fresh 64-bit seed per call (the reference's unseeded behaviour); an int makes the
        # calls reproducible (draw keyed by seed, piece index within the call, start byte, token length)
        self.dropout_seed: Optional[int] = None
        self._dropout_lock = threading.Lock()  # set_dropout .. encode .. reset must not interleave between threads
        self._host_model: Optional[N.Model] = None

    # ---- construction / serialisation (src/tokenizer.rs:261-297, 349-435; src/lib.rs:109-204) --------
    @staticmethod
    def from_str(s: str, device: Optional[int] = None) -> "Tokenizer":
        try:
            obj = json.loads(s)
        except json.JSONDecodeError as e:
            raise TokenGeeXError(str(e))
        if not isinstance(obj, dict):
            raise TokenGeeXError("invalid type: expected struct Tokenizer")
        fields = ["version", "special_tokens", "processors", "vocab"]
        for k in obj:
            if k not in fields:
                raise TokenGeeXError(f"unknown field `{k}`, expected one of `version`, `special_tokens`, "
                                     "`processors`, `vocab`")
        if "version" not in obj:
            raise TokenGeeXError("missing field `version`")
        if obj["version"] != SERIALIZATION_VERSION:
            raise TokenGeeXError(f"unsupported version: {obj['version']}")
        tokens, scores, keep = [], [], []
        for ent in obj.get("vocab", []):
            for k in ent:
                if k not in ("value", "score", "encoded", "keep"):
                    raise TokenGeeXError(f"unknown field `{k}`, expected one of `value`, `score`, `encoded`, `keep`")
            if "value" not in ent or ent["value"] is None:
                raise TokenGeeXError("missing field `token`")  # sic: src/lib.rs:190
            if "score" not in ent or ent["score"] is None:
                raise TokenGeeXError("missing field `score`")
            v = ent["value"]
            if ent.get("encoded", False):
                try:
                    pad = "=" * (-len(v) % 4)  # STANDARD_NO_PAD (src/lib.rs:8)
                    if "=" in v:
                        raise ValueError("padding")
                    raw = base64.b64decode(v + pad, validate=True)
                except Exception as e:
                    raise TokenGeeXError(f"Invalid base64: {e}")
            else:
                raw = v.encode("utf-8")
            tokens.append(raw)
            scores.append(float(ent["score"]))
            keep.append(bool(ent.get("keep", False)))
        procs = [_Processor.from_json(p) for p in obj.get("processors", [])]
        return Tokenizer(tokens, scores, keep, procs, obj.get("special_tokens", []), device=device)

    @staticmethod
    def from_file(filepath: str, device: Optional[int] = None) -> "Tokenizer":
        try:
            with open(filepath, "r", encoding="utf-8") as f:
                s = f.read()
        except OSError as e:
            raise TokenGeeXError(str(e))
        return Tokenizer.from_str(s, device=device)

    def _vocab_json(self, i: int) -> List[str]:
        raw = self._tokens[i]
        try:
            value, encoded = raw.decode("utf-8"), False
        except UnicodeDecodeError:
            value, encoded = base64.b64encode(raw).decode().rstrip("="), True
        parts = [f'"value":{_jstr(value)}', f'"score":{fmt_f64(float(self._scores[i]))}']
        if encoded:
            parts.append('"encoded":true')
        if self._keep[i]:
            parts.append('"keep":true')
        return parts

    def to_string(self) -> str:
        """serde_json::to_string (compact)."""
        vocab = ",".join("{" + ",".join(self._vocab_json(i)) + "}" for i in range(len(self._tokens)))
        procs = ",".join(json.dumps(p.to_json(), separators=(",", ":")) for p in self._processors)
        specials = ",".join(_jstr(s) for s in self._special)
        return (f'{{"version":{_jstr(SERIALIZATION_VERSION)},"special_tokens":[{specials}],'
                f'"processors":[{procs}],"vocab":[{vocab}]}}')

    def save(self, filepath: str) -> None:
        """serde_json::to_string_pretty (2-space indent), src/tokenizer.rs:261-265."""
        def arr(items: List[str], ind: str) -> str:
            if not items:
                return "[]"
            inner = (",\n").join(ind + "  " + it for it in items)
            return "[\n" + inner + "\n" + ind + "]"

        def obj(parts: List[str], ind: str) -> str:
            return "{\n" + ",\n".join(ind + "  " + p.replace('":', '": ', 1) for p in parts) + "\n" + ind + "}"

        vocab = [obj(self._vocab_json(i), "    ") for i in range(len(self._tokens))]
        procs = [obj([f'"{k}":{_jstr(v)}' for k, v in p.to_json().items()], "    ") for p in self._processors]
        specials = [_jstr(s) for s in self._special]
        text = ("{\n" + f'  "version": {_jstr(SERIALIZATION_VERSION)},\n' + f'  "special_tokens": {arr(specials, "  ")},\n'
                + f'  "processors": {arr(procs, "  ")},\n' + f'  "vocab": {arr(vocab, "  ")}\n' + "}")
        with open(filepath, "w", encoding="utf-8") as f:
            f.write(text)

    def __getstate__(self):
        return self.to_string().encode("utf-8")

    def __setstate__(self, state):
        t = Tokenizer.from_str(state.decode("utf-8"))
        self.__dict__.update(t.__dict__)

    # ---- special tokens (src/tokenizer.rs:39-53, 203-259) ----------------------------------------------
    def add_special_tokens(self, tokens: Sequence[str]) -> None:
        for t in tokens:
            if t in self._special_map:
                continue
            self._special_map[t] = len(self._special)
            self._special.append(t)

    def special_tokens(self) -> List[str]:
        return list(self._special)

    def add_base_tokens(self, tokens: Sequence[Tuple[bytes, float]], keep: bool = False) -> None:
        """Tokenizer::add_base_tokens -> Model::add_tokens (src/tokenizer.rs:56-61, src/model.rs:184-194; Rust API
        only, used by `merge`): the tokens get the next ids, the token -> id map takes the new id of a duplicate (the
        trie's last-duplicate-wins rule) and the device model is rebuilt with the extended vocabulary on the next
        encode.  Special-token ids move up by len(tokens), as in the reference (ids >= base_vocab_size())."""
        for value, score in tokens:
            value = bytes(value)
            self._token_to_id[value] = len(self._tokens)
            self._tokens.append(value)
        if tokens:
            self._scores = np.concatenate([self._scores, np.asarray([float(s) for _, s in tokens], np.float64)])
            self._keep = np.concatenate([self._keep, np.full(len(tokens), 1 if keep else 0, np.uint8)])
            for m in (self._model, self._model_bytes_only, self._host_model):
                if m is not None:
                    m.close()
            self._model = self._model_bytes_only = self._host_model = None

    def vocab_size(self) -> int:
        return len(self._tokens) + len(self._special)

    def base_vocab_size(self) -> int:
        return len(self._tokens)

    def special_vocab_size(self) -> int:
        return len(self._special)

    def is_special(self, id: int) -> bool:
        return id >= len(self._tokens) and id - len(self._tokens) < len(self._special)

    def is_base(self, id: int) -> bool:
        return id < len(self._tokens)

    def token_to_id(self, token: bytes) -> Optional[int]:
        r = self.base_token_to_id(token)
        if r is not None:
            return r
        try:
            return self.special_token_to_id(bytes(token).decode("utf-8"))
        except UnicodeDecodeError:
            return None

    def base_token_to_id(self, token: bytes) -> Optional[int]:
        return self._token_to_id.get(bytes(token))

    def special_token_to_id(self, token: str) -> Optional[int]:
        i = self._special_map.get(token)
        return None if i is None else i + len(self._tokens)

    def id_to_token(self, id: int) -> Optional[bytes]:
        s = self.id_to_special_token(id)
        if s is not None:
            return s.encode("utf-8")
        b = self.id_to_base_token(id)
        return None if b is None else b[0]

    def id_to_base_token(self, id: int) -> Optional[Tuple[bytes, float]]:
        if 0 <= id < len(self._tokens):
            return self._tokens[id], float(self._scores[id])
        return None

    def id_to_special_token(self, id: int) -> Optional[str]:
        i = id - len(self._tokens)
        if id < len(self._tokens) or i >= len(self._special):
            return None
        return self._special[i]

    # ---- models ---------------------------------------------------------------------------------------
    def _host(self) -> N.Model:
        if self._host_model is None:
            self._host_model = N.Model(self._tokens, self._scores, device=None)
        return self._host_model

    def _dev(self, dropout: float) -> N.Model:
        try:
            if dropout <= 0.0:
                if self._model is None:
                    self._model = N.Model(self._tokens, self._scores, device=self._device)
                return self._model
            if dropout >= 1.0 or dropout != dropout:  # (NaN: `dropout < rand` is false for every draw, like >= 1.0)
                # every token longer than one byte is skipped (src/model.rs:100 with rand() in [0,1)):
                # same ids, but the multi-byte entries can never match
                if self._model_bytes_only is None:
                    toks = [t if len(t) <= 1 else b"" for t in self._tokens]
                    self._model_bytes_only = N.Model(toks, self._scores, device=self._device)
                return self._model_bytes_only
            # 0 < dropout < 1: the reference draws from an unseeded thread_rng (src/model.rs:100), so each call
            # takes a fresh seed unless `dropout_seed` is set; the draw itself is keyed (tgx_model_set_dropout)
            if self._model is None:
                self._model = N.Model(self._tokens, self._scores, device=self._device)
            return self._model
        except N.TgxError as e:
            raise TokenGeeXError(e.msg)

    def common_prefix_search(self, text: str) -> Iterable[int]:
        return self._host().common_prefix_search(text.encode("utf-8"))[0]

    # ---- encode (src/tokenizer.rs:65-123) ----------------------------------------------------------------
    def _preprocess(self, s: str) -> Tuple[bytes, bool]:
        """Applies the processors; the trailing crlf processor (if it is the last one) is left to the
        GPU kernel.  → (utf-8 bytes, run crlf on the device)."""
        procs = self._processors
        gpu_crlf = bool(procs) and procs[-1].kind == "crlf"
        for p in (procs[:-1] if gpu_crlf else procs):
            s = p.preprocess(s)
        return s.encode("utf-8"), gpu_crlf

    def _encode_pieces(self, pieces: List[bytes], gpu_crlf: bool, dropout: float) -> Tuple[np.ndarray, np.ndarray]:
        """→ (ids u32[T], id_off u64[len(pieces) + 1])"""
        if not pieces:
            return np.zeros(0, np.uint32), np.zeros(1, np.uint64)
        model = self._dev(dropout)
        blob, off = N.pack(pieces)
        drawn = 0.0 < dropout < 1.0
        try:
            # The dropout setting is state of the native handle: EVERY encode through the handle takes the lock, so a
            # deterministic call (dropout 0.0) can never run between another thread's set_dropout(p) and its reset.
            with self._dropout_lock:
                if drawn:
                    seed = self.dropout_seed
                    model.set_dropout(dropout, secrets.randbits(64) if seed is None else seed)
                try:
                    ids, id_off, status, plen, rc, bad = model.encode_batch(blob, off, crlf=gpu_crlf)
                finally:
                    if drawn:
                        model.set_dropout(0.0, 0)
        except N.TgxError as e:
            raise TokenGeeXError(e.msg)
        if rc == N.TGX_ERR_NO_PATH:
            n = int(plen[bad])
            raise TokenGeeXError(f"no path to position {n}/{n}")  # Display of Error::NoPath, src/lib.rs:243-245
        return ids, id_off

    def _encode_many(self, texts: Sequence[str], dropout: float, ordinary: bool) -> List[List[int]]:
        V = len(self._tokens)
        plan, pieces, gpu_crlf = [], [], False
        for text in texts:
            if ordinary or not self._special:
                parts = [(text, False)]
            else:
                parts = split_special_tokens(text, self._special)
            row = []
            for sub, is_special in parts:
                if is_special:
                    row.append(("s", V + self._special_map[sub]))
                else:
                    raw, gpu_crlf = self._preprocess(sub)
                    row.append(("p", len(pieces)))
                    pieces.append(raw)
            plan.append(row)
        ids, id_off = self._encode_pieces(pieces, gpu_crlf, dropout)
        rows = id_rows(ids, id_off)
        if len(pieces) == len(plan) and all(len(row) == 1 and row[0][0] == "p" for row in plan):
            return rows  # no special token anywhere: the common batch
        out = []
        for row in plan:
            r: List[int] = []
            for kind, v in row:
                if kind == "s":
                    r.append(v)
                else:
                    r.extend(rows[v])
            out.append(r)
        return out

    def encode(self, text: str, dropout: float) -> List[int]:
        return self._encode_many([text], dropout, ordinary=False)[0]

    def encode_ordinary(self, text: str, dropout: float) -> List[int]:
        return self._encode_many([text], dropout, ordinary=True)[0]

    def encode_batch(self, texts: List[str], dropout: float) -> List[List[int]]:
        return self._encode_many(texts, dropout, ordinary=False)

    def encode_ordinary_batch(self, texts: List[str], dropout: float) -> List[List[int]]:
        return self._encode_many(texts, dropout, ordinary=True)

    # ---- corpus images (tokengeex_b200/corpus.py) -------------------------------------------------------------
    def corpus_dtype(self, dtype=None) -> np.dtype:
        """dtype=None: uint16 when every id fits (vocab_size() <= 65536), else uint32."""
        if dtype is None:
            return np.dtype(np.uint16 if self.vocab_size() <= 65536 else np.uint32)
        dt = np.dtype(dtype)
        if dt not in (np.dtype(np.uint16), np.dtype(np.uint32)):
            raise TokenGeeXError(f"unsupported id dtype {dt}: uint16 or uint32")
        return dt

    def separator_id(self, separator: Optional[str]) -> int:
        """-1 for None, else the id of the token (usually a special token such as "<eos>")."""
        if separator is None:
            return -1
        i = self.token_to_id(separator.encode("utf-8"))
        if i is None:
            raise TokenGeeXError(f"unknown separator token {separator!r}")
        return i

    def corpus_on_device(self) -> bool:
        """The device splits the corpus when the processors are [] or exactly [crlf] (crlf twice is not crlf once:
        "\r\r\n"); any other list takes the host path of encode_corpus."""
        return [p.kind for p in self._processors] in ([], ["crlf"])

    def encode_corpus(self, data, dropout: float = 0.0, separator: Optional[str] = None, dtype=None,
                      source: str = "<corpus>"):
        """Ordinary encoding (special tokens in the text are not split out) of every non-empty sample of a
        NUL-separated corpus image (bytes-like or uint8 array), as `load_sources` + `Model::encode` would do.
        → (ids, offsets u64[S+1]): sample i (and its separator) is ids[offsets[i]:offsets[i+1]].  Invalid UTF-8
        raises ValueError with load_sources' text (`source` names the file in it)."""
        arr = data if isinstance(data, np.ndarray) else np.frombuffer(data, np.uint8)
        seed = self.dropout_seed if self.dropout_seed is not None else secrets.randbits(64)
        return self._encode_corpus(np.ascontiguousarray(arr, np.uint8).reshape(-1), dropout, self.separator_id(separator),
                                   self.corpus_dtype(dtype), 0, seed, source)

    def _encode_corpus(self, arr: np.ndarray, dropout: float, sep_id: int, dt: np.dtype, sample_base: int, seed: int,
                       source: str, ids_out=None, off_out=None):
        if dt == np.uint16 and (len(self._tokens) > 65536 or sep_id >= 65536):
            raise TokenGeeXError("uint16 ids need a vocabulary (and separator) below 65536")
        if not self.corpus_on_device():
            return self._encode_corpus_host(arr, dropout, sep_id, dt, seed, source)
        model = self._dev(dropout)
        drawn = 0.0 < dropout < 1.0
        try:
            with self._dropout_lock:
                if drawn:
                    model.set_dropout(dropout, seed)
                try:
                    ids, off, rc, bad, pos = model.encode_corpus(arr, crlf=bool(self._processors),
                                                                 sample_base=sample_base, sep_id=sep_id, dtype=dt,
                                                                 ids_out=ids_out, off_out=off_out)
                finally:
                    if drawn:
                        model.set_dropout(0.0, 0)
        except N.TgxError as e:
            raise TokenGeeXError(e.msg)
        if rc == N.TGX_ERR_NOT_UTF8:
            z = np.flatnonzero(arr[pos:] == 0)
            end = pos + int(z[0]) if z.size else arr.size
            try:
                arr[pos:end].tobytes().decode("utf-8")
            except UnicodeDecodeError as e:
                raise ValueError(f"Sample in {source!r} is not valid UTF-8: {e}") from None
            raise TokenGeeXError(f"sample {bad} reported as invalid UTF-8 decodes on the host")
        if rc == N.TGX_ERR_NO_PATH:
            raise TokenGeeXError(f"no path to position {pos}/{pos}")  # Display of Error::NoPath, src/lib.rs:243-245
        return ids, off

    def _encode_corpus_host(self, arr: np.ndarray, dropout: float, sep_id: int, dt: np.dtype, seed: int, source: str):
        """load_sources' split, check and processors on the host, then Model.encode_batch and the same layout."""
        samples = []
        for piece in arr.tobytes().split(b"\x00"):
            if not piece:
                continue
            try:
                s = piece.decode("utf-8")
            except UnicodeDecodeError as e:
                raise ValueError(f"Sample in {source!r} is not valid UTF-8: {e}") from None
            for p in self._processors:
                s = p.preprocess(s)
            if s:
                samples.append(s.encode("utf-8"))
        saved = self.dropout_seed
        self.dropout_seed = seed
        try:
            ids, id_off = self._encode_pieces(samples, False, dropout)
        finally:
            self.dropout_seed = saved
        return corpus_layout(ids, id_off, sep_id, dt)

    # ---- decode (src/tokenizer.rs:126-187, src/model.rs:146-160) ------------------------------------------
    def _decode_base(self, ids: Sequence[int]) -> str:
        buf = bytearray()
        V = len(self._tokens)
        for i in ids:
            if i >= V or i < 0:
                raise TokenGeeXError(f"token id {i} is out of bounds")
            buf += self._tokens[i]
        return buf.decode("utf-8", errors="replace")  # String::from_utf8_lossy

    def decode(self, ids: List[int], include_special_tokens: bool) -> str:
        V = len(self._tokens)
        out, seg = [], []
        for i in ids:
            if i >= V:
                out.append(self._decode_base(seg))  # processors' postprocess is the identity
                seg = []
                k = i - V
                if k >= len(self._special):
                    raise TokenGeeXError(f"token id {i} is out of bounds")
                if include_special_tokens:
                    out.append(self._special[k])
            else:
                seg.append(i)
        out.append(self._decode_base(seg))
        return "".join(out)

    def decode_batch(self, ids: List[List[int]], include_special_tokens: bool) -> List[str]:
        return [self.decode(x, include_special_tokens) for x in ids]
