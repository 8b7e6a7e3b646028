"""tokzig_b200 -- Python (ctypes) face of the B200-native batch encoder for jrc2139/tokenizer-zig's encode path.

The names mirror the reference's public API (/root/reference/src/lib.zig:32-224): ``Tokenizer.from_json`` /
``from_file`` (fromJson / fromFile), ``encode(text, add_special_tokens)``, ``token_to_id``, ``id_to_token``,
``get_vocab_size``, ``add_special_tokens``, and the public fields ``truncation`` / ``padding``; ``Encoding`` carries
ids / type_ids / tokens / offsets / special_tokens_mask / attention_mask (src/encoding.zig:231-243).  ``encode_batch``
is the batch form the GPU path exists for.  Everything computes on the GPU through the C ABI of
include/tokzig_b200.h; there is no CPU fallback and the import fails loudly when the CUDA library is not built.

The directory name contains a hyphen, so import it through ``tokzig_b200`` (the shim at the repo root).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libtokzig_b200.so")

# status codes (include/tokzig_b200.h)
OK, ERR_OOM, ERR_MISSING_UNK, ERR_INVALID_UTF8, ERR_CUDA, ERR_INVALID_ARG = 0, -1, -2, -3, -4, -5
ERR_INVALID_JSON, ERR_MISSING_MODEL, ERR_UNSUPPORTED_MODEL, ERR_MISSING_VOCAB, ERR_INVALID_VOCAB_ENTRY, ERR_IO = -10, -11, -12, -13, -14, -20
_ERR_NAMES = {ERR_OOM: "OutOfMemory", ERR_MISSING_UNK: "MissingUnkToken", ERR_INVALID_UTF8: "InvalidUtf8", ERR_CUDA: "CudaError",
              ERR_INVALID_ARG: "InvalidArgument", ERR_INVALID_JSON: "InvalidJson", ERR_MISSING_MODEL: "MissingModel",
              ERR_UNSUPPORTED_MODEL: "UnsupportedModelType", ERR_MISSING_VOCAB: "MissingVocab",
              ERR_INVALID_VOCAB_ENTRY: "InvalidVocabEntry", ERR_IO: "IoError"}

OUT_IDS, OUT_OFFSETS, OUT_ATTENTION, OUT_TYPE_IDS, OUT_SPECIAL, OUT_ALL = 1, 2, 4, 8, 16, 31
OUT_SPAN_TOKENS = 128            # 16-byte SpanToken records (src/token.zig:19-33)
OUT_IDS_U16 = 64                 # ids as u16 (ids16) when every id of the vocabulary is < 65536
OUT_OFFSETS_PACKED = 32          # one u16 per token (start | end << 8); falls back to OUT_OFFSETS when a pre-token has >= 256 bytes
OUT_WORD_IDS = 256               # word ids: each token's pre-token index in its document, WORD_NONE for specials and padding
WORD_NONE = 0xFFFFFFFF
NORM_CFG_LOWER, NORM_BERT_STRUCT, NORM_LOWER_STRUCT = 1, 2, 3
PT_WS_CFG, PT_BERT_CFG, PT_WS_STRUCT, PT_BERT_STRUCT, PT_BYTELEVEL_STRUCT = 1, 2, 3, 4, 5
MODEL_BPE, MODEL_WORDPIECE = 0, 1


class TokzigError(Exception):
    def __init__(self, code: int, msg: str = "", doc: int = -1):
        self.code = code
        self.name = _ERR_NAMES.get(code, str(code))
        self.doc = doc
        super().__init__(f"{self.name}: {msg}" if msg else self.name)


class ModelDesc(C.Structure):
    _fields_ = [
        ("model_kind", C.c_int32),
        ("norm_lut", C.POINTER(C.c_uint16)),
        ("class_lut", C.POINTER(C.c_uint8)),
        ("vocab_bytes", C.POINTER(C.c_uint8)),
        ("vocab_off", C.POINTER(C.c_uint64)),
        ("vocab_ids", C.POINTER(C.c_uint32)),
        ("vocab_n", C.c_uint32),
        ("merge_first", C.POINTER(C.c_uint32)),
        ("merge_second", C.POINTER(C.c_uint32)),
        ("merge_rank", C.POINTER(C.c_uint32)),
        ("merge_new", C.POINTER(C.c_uint32)),
        ("merges_n", C.c_uint32),
        ("has_unk", C.c_int32),
        ("unk_id", C.c_uint32),
        ("prefix", C.POINTER(C.c_uint8)),
        ("prefix_len", C.c_uint32),
        ("max_input_chars_per_word", C.c_uint64),
    ]


class EncodeParams(C.Structure):
    _fields_ = [
        ("has_truncation", C.c_int32),
        ("max_length", C.c_uint64),
        ("has_padding", C.c_int32),
        ("pad_length", C.c_uint64),
        ("pad_id", C.c_uint32),
        ("pad_type_id", C.c_uint32),
        ("pad_left", C.c_int32),
        ("outputs", C.c_uint32),
        ("fast", C.c_int32),
        ("fast_max_sequence_length", C.c_uint32),
        ("fast_max_tokens", C.c_uint32),
        ("hf_flags", C.c_uint32),
        ("tpl_n_prefix", C.c_uint32),
        ("tpl_n_suffix", C.c_uint32),
        ("tpl_prefix_id", C.c_uint32 * 4),
        ("tpl_prefix_type", C.c_uint32 * 4),
        ("tpl_suffix_id", C.c_uint32 * 4),
        ("tpl_suffix_type", C.c_uint32 * 4),
        ("tpl_seq_type", C.c_uint32),
    ]


HF_TEMPLATE, HF_DOC_OFFSETS = 1, 2


class BatchResult(C.Structure):
    _fields_ = [
        ("n_docs", C.c_uint64),
        ("n_tokens", C.c_uint64),
        ("n_real_tokens", C.c_uint64),
        ("doc_tok_off", C.c_void_p),
        ("ids", C.c_void_p),
        ("offsets", C.c_void_p),
        ("attention_mask", C.c_void_p),
        ("type_ids", C.c_void_p),
        ("special_tokens_mask", C.c_void_p),
        ("err_doc", C.c_int64),
        ("offsets_packed", C.c_void_p),
        ("ids16", C.c_void_p),
        ("span_tokens", C.c_void_p),
        ("n_wide", C.c_uint64),
        ("wide_tokens", C.c_void_p),
        ("word_ids", C.c_void_p),
    ]


class CompactResult(C.Structure):
    """tkz_compact_result: kept real tokens only; padding / masks are rebuilt on the host (tkz_compact_expand)."""
    _fields_ = [
        ("n_docs", C.c_uint64),
        ("n_kept", C.c_uint64),
        ("n_real_tokens", C.c_uint64),
        ("doc_kept_off", C.c_void_p),
        ("ids", C.c_void_p),
        ("ids16", C.c_void_p),
        ("offsets_packed", C.c_void_p),
        ("offsets", C.c_void_p),
        ("params", EncodeParams),
        ("err_doc", C.c_int64),
        ("n_wide", C.c_uint64),
        ("wide_tokens", C.c_void_p),
    ]


class DecodeResult(C.Structure):
    _fields_ = [("n_seqs", C.c_uint64), ("n_bytes", C.c_uint64), ("byte_off", C.c_void_p), ("bytes", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("arena_bytes", C.c_uint64), ("n_words", C.c_uint64), ("n_unique_words", C.c_uint64),
                ("n_long_words", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("ms_split", C.c_float), ("ms_model", C.c_float), ("ms_scan", C.c_float), ("ms_emit", C.c_float), ("ms_total", C.c_float),
                ("model_flags", C.c_uint32), ("ms_call_kernels", C.c_float), ("reserved0", C.c_uint32), ("path", C.c_uint32)]


# every symbol include/tokzig_b200.h declares (checked by tests/test_cabi_symbols.py)
EXPORTED_SYMBOLS = [
    "tkz_ctx_create", "tkz_ctx_destroy", "tkz_last_error", "tkz_ctx_get_stats", "tkz_model_upload", "tkz_encode_batch",
    "tkz_ctx_numa_node", "tkzm_create", "tkzm_destroy", "tkzm_size", "tkzm_ctx", "tkzm_last_error", "tkzm_model_upload", "tkzm_shard_bounds",
    "tkzm_document_costs", "tkzm_encode_batch_compact",
    "tkz_encode_batch_device", "tkz_encode_batch_compact", "tkz_compact_slots", "tkz_compact_expand", "tkz_decode_upload", "tkz_decode_batch",
    "tkzh_from_json", "tkzh_from_file", "tkzh_free", "tkzh_last_error", "tkzh_ctx", "tkzh_set_truncation", "tkzh_set_padding",
    "tkzh_set_normalizer", "tkzh_set_pretokenizer", "tkzh_encode_batch", "tkzh_encode_batch_fast", "tkzh_decode", "tkzh_decode_batch", "tkzh_get_vocab_size", "tkzh_token_to_id",
    "tkzh_id_to_token", "tkzh_model_id_to_token", "tkzh_add_special_tokens", "tkzh_model_vocab_count", "tkzh_merge_count", "tkzh_has_normalizer",
    "tkzh_has_pretokenizer", "tkzh_has_post_processor", "tkzh_set_hf_compat", "tkzh_hf_template", "tkzh_added_token_count", "tkzh_added_token", "tkzh_model_desc",
]

_lib = None


def lib():
    """Loads the in-tree CUDA library.  No fallback: a missing library is a hard error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(tokzig_b200 has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
    L.tkz_ctx_create.argtypes = [i32, vp, u64, C.POINTER(vp)]
    L.tkz_ctx_destroy.argtypes = [vp]
    L.tkz_last_error.argtypes = [vp]
    L.tkz_last_error.restype = C.c_char_p
    L.tkz_ctx_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.tkz_model_upload.argtypes = [vp, C.POINTER(ModelDesc)]
    L.tkz_encode_batch.argtypes = [vp, vp, vp, u64, C.POINTER(EncodeParams), C.POINTER(BatchResult)]
    L.tkz_encode_batch_device.argtypes = [vp, vp, vp, u64, u64, C.POINTER(EncodeParams), C.POINTER(BatchResult)]
    L.tkz_encode_batch_compact.argtypes = [vp, vp, vp, u64, C.POINTER(EncodeParams), i32, C.POINTER(CompactResult)]
    L.tkz_compact_slots.argtypes = [C.POINTER(CompactResult), u64, u64]
    L.tkz_compact_slots.restype = u64
    L.tkz_compact_expand.argtypes = [C.POINTER(CompactResult), u64, u64, vp, vp, vp, vp, vp, vp]
    L.tkz_ctx_numa_node.argtypes = [vp]
    L.tkzm_create.argtypes = [vp, C.c_int32, C.POINTER(vp)]
    L.tkzm_destroy.argtypes = [vp]
    L.tkzm_size.argtypes = [vp]
    L.tkzm_size.restype = C.c_int32
    L.tkzm_ctx.argtypes = [vp, C.c_int32]
    L.tkzm_ctx.restype = vp
    L.tkzm_last_error.argtypes = [vp]
    L.tkzm_last_error.restype = C.c_char_p
    L.tkzm_model_upload.argtypes = [vp, C.POINTER(ModelDesc)]
    L.tkzm_shard_bounds.argtypes = [vp, u64, C.c_int32, vp, vp]
    L.tkzm_document_costs.argtypes = [vp, vp, u64, vp, C.c_int32, vp]
    L.tkzm_encode_batch_compact.argtypes = [vp, vp, vp, u64, C.POINTER(EncodeParams), i32, i32, vp, vp, vp]
    L.tkzh_from_json.argtypes = [C.c_char_p, u64, i32, vp, C.POINTER(vp)]
    L.tkzh_from_file.argtypes = [C.c_char_p, i32, vp, C.POINTER(vp)]
    L.tkzh_free.argtypes = [vp]
    L.tkzh_last_error.argtypes = [vp]
    L.tkzh_last_error.restype = C.c_char_p
    L.tkzh_ctx.argtypes = [vp]
    L.tkzh_ctx.restype = vp
    L.tkzh_set_truncation.argtypes = [vp, i32, u64]
    L.tkzh_set_hf_compat.argtypes = [vp, C.c_uint32]
    L.tkzh_set_hf_compat.restype = C.c_int
    L.tkzh_hf_template.argtypes = [vp] + [vp] * 7
    L.tkzh_hf_template.restype = C.c_int
    L.tkzh_set_padding.argtypes = [vp, i32, i32, u64, u32, u32, i32]
    L.tkzh_set_normalizer.argtypes = [vp, vp, vp, C.c_int32]
    L.tkzh_set_pretokenizer.argtypes = [vp, vp, C.c_int32]
    L.tkzh_encode_batch.argtypes = [vp, vp, vp, u64, i32, u32, C.POINTER(BatchResult)]
    L.tkzh_encode_batch_fast.argtypes = [vp, vp, vp, u64, u32, u32, u32, C.POINTER(BatchResult)]
    L.tkzh_decode.argtypes = [vp, vp, u64, i32, C.POINTER(vp), C.POINTER(u64)]
    L.tkzh_decode_batch.argtypes = [vp, vp, vp, u64, i32, C.POINTER(DecodeResult)]
    L.tkz_decode_upload.argtypes = [vp, vp]
    L.tkz_decode_batch.argtypes = [vp, vp, vp, u64, i32, C.POINTER(DecodeResult)]
    L.tkzh_get_vocab_size.argtypes = [vp]
    L.tkzh_get_vocab_size.restype = u64
    L.tkzh_token_to_id.argtypes = [vp, C.c_char_p, u64, C.POINTER(u32)]
    L.tkzh_id_to_token.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(u64)]
    L.tkzh_model_id_to_token.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(u64)]
    L.tkzh_add_special_tokens.argtypes = [vp, C.c_char_p, vp, u64, C.POINTER(u64)]
    L.tkzh_model_vocab_count.argtypes = [vp]
    L.tkzh_model_vocab_count.restype = u64
    L.tkzh_merge_count.argtypes = [vp]
    L.tkzh_merge_count.restype = u64
    for f in ("tkzh_has_normalizer", "tkzh_has_pretokenizer", "tkzh_has_post_processor"):
        getattr(L, f).argtypes = [vp]
    L.tkzh_added_token_count.argtypes = [vp]
    L.tkzh_added_token_count.restype = u64
    L.tkzh_added_token.argtypes = [vp, u64, C.POINTER(vp), C.POINTER(u64), C.POINTER(C.c_int64), C.POINTER(i32)]
    L.tkzh_model_desc.argtypes = [vp, C.POINTER(ModelDesc)]
    _lib = L
    return L


def _copy(ptr, n, dtype):
    if not ptr or n == 0:
        return np.zeros(0, dtype)
    buf = (C.c_uint8 * (n * np.dtype(dtype).itemsize)).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype, count=n).copy()


# --------------------------------------------------------------------------- results
@dataclass
class Encoding:
    """src/encoding.zig:231-243 (words is always null and overflowing always empty in the reference)."""
    ids: np.ndarray
    type_ids: np.ndarray
    tokens: List[bytes]
    offsets: np.ndarray              # (n, 2) u32, byte offsets into the normalised pre-token
    special_tokens_mask: np.ndarray
    attention_mask: np.ndarray

    def __len__(self):
        return len(self.ids)

    def get_ids(self):
        return self.ids

    def get_tokens(self):
        return self.tokens

    def get_attention_mask(self):
        return self.attention_mask


@dataclass
class BatchEncoding:
    """CSR over documents (tkz_batch_result)."""
    doc_tok_off: np.ndarray
    ids: np.ndarray
    offsets: Optional[np.ndarray]
    attention_mask: Optional[np.ndarray]
    type_ids: Optional[np.ndarray]
    special_tokens_mask: Optional[np.ndarray]
    n_real_tokens: int = 0
    offsets_packed: Optional[np.ndarray] = None     # u16 per token: start | end << 8 (OUT_OFFSETS_PACKED); 0xFFFF = see wide_tokens
    wide_tokens: Optional[np.ndarray] = None        # (n_wide, 4) u32: slot low, slot high, start, end -- tokens of pre-tokens of 256+ bytes
    span_tokens: Optional[np.ndarray] = None        # (n, 4) u32: id, start, end, type_id | flags << 8 (OUT_SPAN_TOKENS)
    word_ids: Optional[np.ndarray] = None           # u32 per slot: pre-token index in the document, WORD_NONE for specials / padding (OUT_WORD_IDS)

    def __len__(self):
        return len(self.doc_tok_off) - 1

    def unpacked_offsets(self) -> Optional[np.ndarray]:
        """(n, 2) u32 offsets whichever form the call delivered."""
        if self.offsets is not None or self.offsets_packed is None:
            return self.offsets
        o = np.stack([self.offsets_packed & 0xFF, self.offsets_packed >> 8], axis=1).astype(np.uint32)
        if self.wide_tokens is not None and len(self.wide_tokens):
            slots = self.wide_tokens[:, 0].astype(np.uint64) | (self.wide_tokens[:, 1].astype(np.uint64) << np.uint64(32))
            assert np.all(self.offsets_packed[slots] == 0xFFFF)
            o[slots] = self.wide_tokens[:, 2:4]
        assert not np.any((self.offsets_packed == 0xFFFF) & (o[:, 0] == 255) & (o[:, 1] == 255))
        return o

    def doc_slice(self, i):
        return slice(int(self.doc_tok_off[i]), int(self.doc_tok_off[i + 1]))


def _result_to_batch(r: BatchResult) -> BatchEncoding:
    T, n = int(r.n_tokens), int(r.n_docs)
    offs = _copy(r.offsets, 2 * T, np.uint32).reshape(-1, 2) if r.offsets else None
    return BatchEncoding(
        doc_tok_off=_copy(r.doc_tok_off, n + 1, np.uint64),
        ids=_copy(r.ids16, T, np.uint16).astype(np.uint32) if r.ids16 else _copy(r.ids, T, np.uint32),
        offsets=offs,
        attention_mask=_copy(r.attention_mask, T, np.uint32) if r.attention_mask else None,
        type_ids=_copy(r.type_ids, T, np.uint32) if r.type_ids else None,
        special_tokens_mask=_copy(r.special_tokens_mask, T, np.uint32) if r.special_tokens_mask else None,
        n_real_tokens=int(r.n_real_tokens),
        offsets_packed=_copy(r.offsets_packed, T, np.uint16) if r.offsets_packed else None,
        wide_tokens=_copy(r.wide_tokens, 4 * int(r.n_wide), np.uint32).reshape(-1, 4) if (r.wide_tokens and r.n_wide) else None,
        span_tokens=_copy(r.span_tokens, 4 * T, np.uint32).reshape(-1, 4) if r.span_tokens else None,
        word_ids=_copy(r.word_ids, T, np.uint32) if r.word_ids else None,
    )


def expand_compact(r: CompactResult, d0: int = 0, d1: Optional[int] = None) -> BatchEncoding:
    """tkz_compact_expand for documents [d0, d1): the six arrays of the reference's Encoding (src/encoding.zig:231-243), CSR."""
    L = lib()
    d1 = int(r.n_docs) if d1 is None else d1
    n = int(L.tkz_compact_slots(C.byref(r), d0, d1))
    off = np.zeros(d1 - d0 + 1, np.uint64)
    ids, attn, typ, sp = (np.zeros(n, np.uint32) for _ in range(4))
    has_off = bool(r.offsets_packed or r.offsets)
    offs = np.zeros((n, 2), np.uint32) if has_off else None
    rc = L.tkz_compact_expand(C.byref(r), d0, d1, off.ctypes.data, ids.ctypes.data, offs.ctypes.data if has_off else None, attn.ctypes.data,
                              typ.ctypes.data, sp.ctypes.data)
    if rc != OK:
        raise TokzigError(rc, "tkz_compact_expand")
    return BatchEncoding(off, ids, offs, attn, typ, sp, int(r.n_real_tokens))


def pack_docs(docs: Sequence[bytes]):
    lens = np.fromiter((len(d) for d in docs), dtype=np.uint64, count=len(docs))
    off = np.zeros(len(docs) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    text = np.frombuffer(b"".join(docs), dtype=np.uint8) if len(docs) else np.zeros(0, np.uint8)
    return np.ascontiguousarray(text), off


# --------------------------------------------------------------------------- device layer
class Context:
    """tkz_ctx: one per GPU.  ``stream`` is a raw cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) or 0."""

    def __init__(self, device: int = 0, stream: int = 0):
        self._L = lib()
        h = C.c_void_p()
        rc = self._L.tkz_ctx_create(device, C.c_void_p(stream) if stream else None, 0, C.byref(h))
        if rc != OK:
            raise TokzigError(rc, (self._L.tkz_last_error(None) or b"").decode())
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._L.tkz_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _err(self):
        return (self._L.tkz_last_error(self._h) or b"").decode()

    def upload(self, desc: ModelDesc):
        rc = self._L.tkz_model_upload(self._h, C.byref(desc))
        if rc != OK:
            raise TokzigError(rc, self._err())

    def stats(self) -> Stats:
        s = Stats()
        self._L.tkz_ctx_get_stats(self._h, C.byref(s))
        return s

    def encode_batch(self, text: np.ndarray, doc_off: np.ndarray, params: Optional[EncodeParams] = None) -> BatchEncoding:
        """Host buffers in, host arrays out (tkz_encode_batch)."""
        text = np.ascontiguousarray(text, dtype=np.uint8)
        doc_off = np.ascontiguousarray(doc_off, dtype=np.uint64)
        r = BatchResult()
        p = params if params is not None else EncodeParams()
        rc = self._L.tkz_encode_batch(self._h, text.ctypes.data if text.size else None, doc_off.ctypes.data, len(doc_off) - 1,
                                      C.byref(p), C.byref(r))
        if rc != OK:
            raise TokzigError(rc, self._err(), int(r.err_doc))
        return _result_to_batch(r)

    def encode_batch_compact(self, text: np.ndarray, doc_off: np.ndarray, params: Optional[EncodeParams] = None, want_offsets: bool = True) -> CompactResult:
        """tkz_encode_batch_compact: the raw struct (its arrays belong to the context until the next encode); see expand_compact."""
        text = np.ascontiguousarray(text, dtype=np.uint8)
        doc_off = np.ascontiguousarray(doc_off, dtype=np.uint64)
        r = CompactResult()
        p = params if params is not None else EncodeParams()
        rc = self._L.tkz_encode_batch_compact(self._h, text.ctypes.data if text.size else None, doc_off.ctypes.data, len(doc_off) - 1,
                                              C.byref(p), 1 if want_offsets else 0, C.byref(r))
        if rc != OK:
            raise TokzigError(rc, self._err(), int(r.err_doc))
        return r

    def encode_batch_device(self, d_text_ptr: int, d_doc_off_ptr: int, n_docs: int, text_bytes: int,
                            params: Optional[EncodeParams] = None) -> BatchResult:
        """Device pointers in, device pointers out (tkz_encode_batch_device); returns the raw result struct."""
        r = BatchResult()
        p = params if params is not None else EncodeParams()
        rc = self._L.tkz_encode_batch_device(self._h, C.c_void_p(d_text_ptr), C.c_void_p(d_doc_off_ptr), n_docs, text_bytes,
                                             C.byref(p), C.byref(r))
        if rc != OK:
            raise TokzigError(rc, self._err(), int(r.err_doc))
        return r


# --------------------------------------------------------------------------- host mirror of src/lib.zig
class Tokenizer:
    """Tokenizer (src/lib.zig:32-224) on the GPU.  ``device=None`` loads the configuration only."""

    def __init__(self, handle, L):
        self._h = handle
        self._L = L
        self.truncation: Optional[dict] = None     # {"max_length": 512}          src/types.zig:55-59
        self.padding: Optional[dict] = None        # {"length":..,"pad_id":..,"pad_type_id":..,"direction":"right"}  src/types.zig:39-45

    @classmethod
    def from_json(cls, json_content, device: Optional[int] = 0, stream: int = 0) -> "Tokenizer":
        L = lib()
        if isinstance(json_content, str):
            json_content = json_content.encode("utf-8", "surrogatepass")
        h = C.c_void_p()
        rc = L.tkzh_from_json(json_content, len(json_content), -1 if device is None else device, C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != OK:
            raise TokzigError(rc, (L.tkzh_last_error(None) or b"").decode())
        return cls(h, L)

    @classmethod
    def from_file(cls, path: str, device: Optional[int] = 0, stream: int = 0) -> "Tokenizer":
        L = lib()
        h = C.c_void_p()
        rc = L.tkzh_from_file(path.encode(), -1 if device is None else device, C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != OK:
            raise TokzigError(rc, (L.tkzh_last_error(None) or b"").decode())
        return cls(h, L)

    def close(self):
        if getattr(self, "_h", None):
            self._L.tkzh_free(self._h)
            self._h = None

    deinit = close

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- hand-wiring (normalizer_impl / pretokenizer_impl are public fields in the reference)
    def set_normalizer(self, ops: Optional[Sequence]):
        """ops: None (no normalizer) or a list of (kind, flags) -- a list is a normalizer.Sequence."""
        if ops is None:
            self._L.tkzh_set_normalizer(self._h, None, None, -1)
            return
        k = np.array([o[0] for o in ops], dtype=np.int32)
        f = np.array([o[1] for o in ops], dtype=np.int32)
        self._L.tkzh_set_normalizer(self._h, k.ctypes.data if len(ops) else None, f.ctypes.data if len(ops) else None, len(ops))

    def set_pretokenizer(self, ops: Optional[Sequence[int]]):
        if ops is None:
            self._L.tkzh_set_pretokenizer(self._h, None, -1)
            return
        k = np.array(list(ops), dtype=np.int32)
        self._L.tkzh_set_pretokenizer(self._h, k.ctypes.data if len(ops) else None, len(ops))

    def set_hf_compat(self, flags: int) -> bool:
        """hf_compat (beyond the reference, off by default): HF_TEMPLATE applies the post_processor's single-sequence template
        (its special tokens only when encode is called with add_special_tokens), HF_DOC_OFFSETS reports document-relative
        offsets.  Returns whether the tokenizer.json carried a template this mode can apply."""
        rc = self._L.tkzh_set_hf_compat(self._h, int(flags))
        if rc < 0:
            raise TokzigError(rc, "tkzh_set_hf_compat", -1)
        return rc == 1

    def hf_template(self):
        """(prefix, suffix, seq_type) of the single-sequence template parsed from the tokenizer.json, prefix / suffix =
        [(special id, type id)], or None when there is none this mode can apply."""
        n1, n2, st = C.c_uint32(), C.c_uint32(), C.c_uint32()
        a, b, c, d = ((C.c_uint32 * 4)() for _ in range(4))
        if self._L.tkzh_hf_template(self._h, C.byref(n1), a, b, C.byref(n2), c, d, C.byref(st)) != 1:
            return None
        return [(a[i], b[i]) for i in range(n1.value)], [(c[i], d[i]) for i in range(n2.value)], st.value

    def _push_params(self):
        if self.truncation is None:
            self._L.tkzh_set_truncation(self._h, 0, 0)
        else:
            self._L.tkzh_set_truncation(self._h, 1, int(self.truncation.get("max_length", 512)))
        if self.padding is None:
            self._L.tkzh_set_padding(self._h, 0, 0, 0, 0, 0, 0)
        else:
            p = self.padding
            length = p.get("length")
            self._L.tkzh_set_padding(self._h, 1, 0 if length is None else 1, 0 if length is None else int(length), int(p.get("pad_id", 0)),
                                     int(p.get("pad_type_id", 0)), 1 if p.get("direction", "right") == "left" else 0)

    def encode_packed(self, text: np.ndarray, doc_off: np.ndarray, add_special_tokens: bool = True, outputs: int = OUT_ALL) -> BatchEncoding:
        self._push_params()
        text = np.ascontiguousarray(text, dtype=np.uint8)
        doc_off = np.ascontiguousarray(doc_off, dtype=np.uint64)
        r = BatchResult()
        rc = self._L.tkzh_encode_batch(self._h, text.ctypes.data if text.size else None, doc_off.ctypes.data, len(doc_off) - 1,
                                       1 if add_special_tokens else 0, outputs, C.byref(r))
        if rc != OK:
            raise TokzigError(rc, (self._L.tkzh_last_error(self._h) or b"").decode(), int(r.err_doc))
        return _result_to_batch(r)

    def params(self, outputs: int = OUT_ALL) -> EncodeParams:
        """the public fields truncation / padding as the tkz_encode_params of a device-layer call"""
        p = EncodeParams()
        if self.truncation is not None:
            p.has_truncation, p.max_length = 1, int(self.truncation.get("max_length", 512))
        if self.padding is not None and self.padding.get("length") is not None:
            p.has_padding, p.pad_length = 1, int(self.padding["length"])
            p.pad_id, p.pad_type_id = int(self.padding.get("pad_id", 0)), int(self.padding.get("pad_type_id", 0))
            p.pad_left = 1 if self.padding.get("direction", "right") == "left" else 0
        p.outputs = outputs
        return p

    def encode_compact(self, text: np.ndarray, doc_off: np.ndarray, want_offsets: bool = True) -> CompactResult:
        """tkz_encode_batch_compact with this tokenizer's truncation / padding (what crosses PCIe: kept ids + packed offsets)."""
        text = np.ascontiguousarray(text, dtype=np.uint8)
        doc_off = np.ascontiguousarray(doc_off, dtype=np.uint64)
        r = CompactResult()
        p = self.params()
        rc = self._L.tkz_encode_batch_compact(self.context_handle(), text.ctypes.data if text.size else None, doc_off.ctypes.data, len(doc_off) - 1,
                                              C.byref(p), 1 if want_offsets else 0, C.byref(r))
        if rc != OK:
            raise TokzigError(rc, (self._L.tkz_last_error(self.context_handle()) or b"").decode(), int(r.err_doc))
        return r

    def encode_fast_packed(self, text: np.ndarray, doc_off: np.ndarray, max_sequence_length: int = 8192, max_tokens: int = 512,
                           outputs: int = OUT_IDS | OUT_OFFSETS | OUT_ATTENTION | OUT_TYPE_IDS | OUT_SPAN_TOKENS) -> BatchEncoding:
        """FastTokenizer.encode (src/lib.zig:356-422) for a batch: arena variants of the models and the arena's caps
        (FastTokenizerOptions.arena_config, src/lib.zig:240-246); truncation / padding fields are not applied."""
        text = np.ascontiguousarray(text, dtype=np.uint8)
        doc_off = np.ascontiguousarray(doc_off, dtype=np.uint64)
        r = BatchResult()
        rc = self._L.tkzh_encode_batch_fast(self._h, text.ctypes.data if text.size else None, doc_off.ctypes.data, len(doc_off) - 1,
                                            max_sequence_length, max_tokens, outputs, C.byref(r))
        if rc != OK:
            raise TokzigError(rc, (self._L.tkzh_last_error(self._h) or b"").decode(), int(r.err_doc))
        return _result_to_batch(r)

    def encode_fast_batch(self, docs: Sequence, **kw) -> BatchEncoding:
        text, off = pack_docs([d if isinstance(d, (bytes, bytearray)) else d.encode("utf-8") for d in docs])
        return self.encode_fast_packed(text, off, **kw)

    def encode_batch(self, docs: Sequence, add_special_tokens: bool = True, outputs: int = OUT_ALL) -> BatchEncoding:
        text, off = pack_docs([d if isinstance(d, (bytes, bytearray)) else d.encode("utf-8") for d in docs])
        return self.encode_packed(text, off, add_special_tokens, outputs)

    def encode(self, text, add_special_tokens: bool = True) -> Encoding:
        """Tokenizer.encode (src/lib.zig:109-160)."""
        b = self.encode_batch([text], add_special_tokens)
        pad_token = (self.padding or {}).get("pad_token", "[PAD]")
        toks = []
        for i, a in zip(b.ids.tolist(), b.attention_mask.tolist()):
            if a == 0:
                toks.append(pad_token.encode() if isinstance(pad_token, str) else pad_token)     # encoding.zig:410,421
            else:
                toks.append(self._model_id_to_token(i) or b"")                                    # bpe.zig:258, wordpiece.zig:200-205
        return Encoding(b.ids, b.type_ids, toks, b.offsets, b.special_tokens_mask, b.attention_mask)

    def decode(self, ids, skip_special_tokens: bool = False) -> bytes:
        """Tokenizer.decode (src/lib.zig:163-189); host side."""
        a = np.ascontiguousarray(ids, dtype=np.uint32)
        p, n = C.c_void_p(), C.c_uint64(0)
        rc = self._L.tkzh_decode(self._h, a.ctypes.data if a.size else None, a.size, 1 if skip_special_tokens else 0, C.byref(p), C.byref(n))
        if rc != OK:
            raise TokzigError(rc)
        return C.string_at(p.value, n.value) if n.value else b""

    def decode_batch(self, seqs: Sequence, skip_special_tokens: bool = False) -> list:
        """Tokenizer.decode for a batch of id sequences on the GPU (tkz_decode_batch); returns one bytes object per sequence."""
        lens = np.fromiter((len(x) for x in seqs), dtype=np.uint64, count=len(seqs))
        off = np.zeros(len(seqs) + 1, dtype=np.uint64)
        np.cumsum(lens, out=off[1:])
        ids = np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=np.uint32) for x in seqs]) if len(seqs) and off[-1] else np.zeros(0, np.uint32), dtype=np.uint32)
        r = DecodeResult()
        rc = self._L.tkzh_decode_batch(self._h, ids.ctypes.data if ids.size else None, off.ctypes.data, len(seqs), 1 if skip_special_tokens else 0, C.byref(r))
        if rc != OK:
            raise TokzigError(rc, (self._L.tkzh_last_error(self._h) or b"").decode())
        boff = _copy(r.byte_off, len(seqs) + 1, np.uint64)
        data = C.string_at(r.bytes, int(r.n_bytes)) if r.n_bytes else b""
        return [data[int(boff[i]):int(boff[i + 1])] for i in range(len(seqs))]

    # -- lookups (src/lib.zig:203-223)
    def get_vocab_size(self) -> int:
        return int(self._L.tkzh_get_vocab_size(self._h))

    def token_to_id(self, token) -> Optional[int]:
        t = token.encode() if isinstance(token, str) else token
        out = C.c_uint32(0)
        return int(out.value) if self._L.tkzh_token_to_id(self._h, t, len(t), C.byref(out)) else None

    def id_to_token(self, i: int) -> Optional[bytes]:
        p, n = C.c_void_p(), C.c_uint64(0)
        if not self._L.tkzh_id_to_token(self._h, i, C.byref(p), C.byref(n)):
            return None
        return C.string_at(p.value, n.value) if n.value else b""

    def _model_id_to_token(self, i: int) -> Optional[bytes]:
        """the model's own id -> token map (bpe.zig:258): an added token with the same id does not change Encoding.tokens"""
        p, n = C.c_void_p(), C.c_uint64(0)
        if not self._L.tkzh_model_id_to_token(self._h, i, C.byref(p), C.byref(n)):
            return None
        return C.string_at(p.value, n.value) if n.value else b""

    def add_special_tokens(self, tokens: Sequence) -> int:
        bs = [t.encode() if isinstance(t, str) else t for t in tokens]
        off = np.zeros(len(bs) + 1, dtype=np.uint64)
        np.cumsum(np.array([len(b) for b in bs], dtype=np.uint64), out=off[1:])
        added = C.c_uint64(0)
        self._L.tkzh_add_special_tokens(self._h, b"".join(bs), off.ctypes.data, len(bs), C.byref(added))
        return int(added.value)

    # -- loader facts
    def model_vocab_count(self) -> int:
        return int(self._L.tkzh_model_vocab_count(self._h))

    def merge_count(self) -> int:
        return int(self._L.tkzh_merge_count(self._h))

    def has_normalizer(self) -> bool:
        return bool(self._L.tkzh_has_normalizer(self._h))

    def has_pretokenizer(self) -> bool:
        return bool(self._L.tkzh_has_pretokenizer(self._h))

    def has_post_processor(self) -> bool:
        return bool(self._L.tkzh_has_post_processor(self._h))

    def added_tokens(self):
        out = []
        for i in range(int(self._L.tkzh_added_token_count(self._h))):
            p, n, idv, sp = C.c_void_p(), C.c_uint64(0), C.c_int64(0), C.c_int(0)
            self._L.tkzh_added_token(self._h, i, C.byref(p), C.byref(n), C.byref(idv), C.byref(sp))
            out.append((C.string_at(p.value, n.value) if n.value else b"", None if idv.value < 0 else int(idv.value), bool(sp.value)))
        return out

    def model_desc(self) -> dict:
        """The flattened model exactly as it is uploaded to the GPU, as numpy arrays (for loader parity tests)."""
        d = ModelDesc()
        self._L.tkzh_model_desc(self._h, C.byref(d))
        n, mn = d.vocab_n, d.merges_n
        off = np.ctypeslib.as_array(d.vocab_off, shape=(n + 1,)).copy() if n else np.zeros(1, np.uint64)
        blob = bytes(np.ctypeslib.as_array(d.vocab_bytes, shape=(int(off[-1]),))) if n and off[-1] else b""
        keys = [blob[int(off[i]):int(off[i + 1])] for i in range(n)]
        ids = np.ctypeslib.as_array(d.vocab_ids, shape=(n,)).copy() if n else np.zeros(0, np.uint32)

        def arr(p):
            return np.ctypeslib.as_array(p, shape=(mn,)).copy() if mn else np.zeros(0, np.uint32)

        return dict(
            model_kind=d.model_kind, keys=keys, ids=ids,
            merges=np.stack([arr(d.merge_first), arr(d.merge_second), arr(d.merge_rank), arr(d.merge_new)], axis=1) if mn else np.zeros((0, 4), np.uint32),
            has_unk=bool(d.has_unk), unk_id=int(d.unk_id),
            prefix=bytes(np.ctypeslib.as_array(d.prefix, shape=(d.prefix_len,))) if d.prefix_len else b"",
            max_chars=int(d.max_input_chars_per_word),
            norm_lut=np.ctypeslib.as_array(d.norm_lut, shape=(256,)).copy() if d.norm_lut else None,
            class_lut=np.ctypeslib.as_array(d.class_lut, shape=(256,)).copy() if d.class_lut else None,
        )

    def context_handle(self):
        return self._L.tkzh_ctx(self._h)

    def stats(self) -> Stats:
        s = Stats()
        self._L.tkz_ctx_get_stats(self.context_handle(), C.byref(s))
        return s


# --------------------------------------------------------------------------- several GPUs of one box (tkzm_*)
class MultiPool:
    """tkzm_pool: one context per entry of `devices` (a GPU may be named more than once), one host thread per context; the model
    of `tokenizer` (a Tokenizer loaded with device=None is enough) is replicated on all of them."""

    def __init__(self, tokenizer: "Tokenizer", devices: Sequence[int]):
        self._L = lib()
        dv = np.asarray(list(devices), dtype=np.int32)
        h = C.c_void_p()
        rc = self._L.tkzm_create(dv.ctypes.data, len(dv), C.byref(h))
        if rc != OK:
            raise TokzigError(rc, (self._L.tkz_last_error(None) or b"").decode())
        self._h = h
        self.n = len(dv)
        self.tokenizer = tokenizer
        d = ModelDesc()
        self._L.tkzh_model_desc(tokenizer._h, C.byref(d))
        rc = self._L.tkzm_model_upload(self._h, C.byref(d))
        if rc != OK:
            msg = (self._L.tkzm_last_error(self._h) or b"").decode()
            self.close()
            raise TokzigError(rc, msg)

    def close(self):
        if getattr(self, "_h", None):
            self._L.tkzm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def raw_class(self) -> Optional[np.ndarray]:
        """TKZ_CLS_* of every raw byte under the tokenizer's normalizer + pre-tokenizer (None: no pre-tokenizer), for document_costs_c"""
        d = self.tokenizer.model_desc()
        if d["class_lut"] is None:
            return None
        nl = d["norm_lut"] if d["norm_lut"] is not None else np.arange(256, dtype=np.uint16)
        return np.where(nl == 0xFFFF, 1, d["class_lut"][nl & 0xFF]).astype(np.uint8)

    def encode_compact(self, text: np.ndarray, doc_off: np.ndarray, want_offsets: bool = True, cost_balanced: bool = False, bounds: np.ndarray = None):
        """tkzm_encode_batch_compact with the tokenizer's truncation / padding: (bounds, [CompactResult per shard], shard_ms).
        `bounds` (n + 1 document indices) = the caller's own cut."""
        text = np.ascontiguousarray(text, dtype=np.uint8)
        doc_off = np.ascontiguousarray(doc_off, dtype=np.uint64)
        if bounds is not None:
            bounds = np.ascontiguousarray(bounds, dtype=np.uint64).copy()
            cost_balanced = 2
        else:
            bounds = np.zeros(self.n + 1, np.uint64)
        results = (CompactResult * self.n)()
        ms = np.zeros(self.n, np.float64)
        p = self.tokenizer.params()
        rc = self._L.tkzm_encode_batch_compact(self._h, text.ctypes.data if text.size else None, doc_off.ctypes.data, len(doc_off) - 1, C.byref(p),
                                               1 if want_offsets else 0, int(cost_balanced), bounds.ctypes.data, C.cast(results, C.c_void_p), ms.ctypes.data)
        if rc != OK:
            docs = [int(r.err_doc) for r in results if int(r.err_doc) >= 0]
            raise TokzigError(rc, (self._L.tkzm_last_error(self._h) or b"").decode(), min(docs) if docs else -1)
        return bounds, list(results), ms

    def shard_kernel_ms(self) -> np.ndarray:
        """device time of every shard's last call (all chunks), from the contexts' stage events"""
        out = np.zeros(self.n)
        for k in range(self.n):
            s = Stats()
            self._L.tkz_ctx_get_stats(self._L.tkzm_ctx(self._h, k), C.byref(s))
            out[k] = s.ms_call_kernels
        return out

    def encode_expanded(self, text, doc_off, cost_balanced: bool = False) -> BatchEncoding:
        """the whole batch as one BatchEncoding (verification: results are gathered to the host in document order)"""
        bounds, results, _ = self.encode_compact(text, doc_off, True, cost_balanced)
        parts = [expand_compact(r) for r in results]
        base = np.cumsum([0] + [int(p.doc_tok_off[-1]) for p in parts])
        off = np.concatenate([p.doc_tok_off[:-1] + np.uint64(b) for p, b in zip(parts, base)] + [np.array([base[-1]], np.uint64)])
        cat = lambda f: np.concatenate([getattr(p, f) for p in parts])
        return BatchEncoding(off.astype(np.uint64), cat("ids"), np.concatenate([p.offsets for p in parts]), cat("attention_mask"), cat("type_ids"),
                             cat("special_tokens_mask"), sum(p.n_real_tokens for p in parts))


def shard_bounds_c(doc_off: np.ndarray, n_shards: int, cost: np.ndarray = None) -> np.ndarray:
    """tkzm_shard_bounds (the product's cut; `shard_bounds` below is the numpy statement of the same rule)"""
    doc_off = np.ascontiguousarray(doc_off, dtype=np.uint64)
    b = np.zeros(n_shards + 1, np.uint64)
    c = None if cost is None else np.ascontiguousarray(cost, dtype=np.float64)
    rc = lib().tkzm_shard_bounds(doc_off.ctypes.data, len(doc_off) - 1, n_shards, None if c is None else c.ctypes.data, b.ctypes.data)
    if rc != OK:
        raise TokzigError(rc)
    return b.astype(np.int64)


def document_costs_c(text: np.ndarray, doc_off: np.ndarray, raw_class: Optional[np.ndarray], threads: int = 0) -> np.ndarray:
    """tkzm_document_costs; raw_class = 256 x TKZ_CLS_* (None: no pre-tokenizer)"""
    text = np.ascontiguousarray(text, dtype=np.uint8)
    doc_off = np.ascontiguousarray(doc_off, dtype=np.uint64)
    out = np.zeros(len(doc_off) - 1, np.float64)
    rcl = None if raw_class is None else np.ascontiguousarray(raw_class, dtype=np.uint8)
    rc = lib().tkzm_document_costs(text.ctypes.data if text.size else None, doc_off.ctypes.data, len(doc_off) - 1, None if rcl is None else rcl.ctypes.data, threads, out.ctypes.data)
    if rc != OK:
        raise TokzigError(rc)
    return out


# --------------------------------------------------------------------------- multi-GPU sharding (host logic, no collective)
# Modelled device time per input byte, relative to ordinary text (B200, round 1: c2b 5.2 ms / GiB; pre-tokens of 65 B .. 12 KiB
# in the windowed block kernels 104 ms / GiB (c2a); longer ones on the cooperative grid 43 ms per 245 MB (c5b)).
COST_LONG_WORD = 20.0
COST_HUGE_WORD = 36.0


def document_costs(text: np.ndarray, doc_off: np.ndarray, delimiters: bytes = b" \t\n\r") -> np.ndarray:
    """Modelled encode cost per document, in units of "one byte of ordinary text" (SURVEY 8e: "cost model (bytes x per-bucket
    factor)" for skewed corpora): bytes + (COST_LONG_WORD - 1) x bytes in pre-tokens of 65..12288 bytes + (COST_HUGE_WORD - 1)
    x bytes in longer ones.  `delimiters` = the bytes the pre-tokenizer drops (b"" = no pre-tokenizer: a document is one
    pre-token).  Host-side helper for cutting shards; plain numpy over the text, nothing is encoded."""
    text = np.asarray(text, dtype=np.uint8)
    doc_off = np.asarray(doc_off, dtype=np.int64)
    nd = len(doc_off) - 1
    lens = np.diff(doc_off).astype(np.float64)
    if nd == 0:
        return lens
    if len(delimiters) == 0:
        wlen, wdoc = np.diff(doc_off), np.arange(nd)
    else:
        base, end_ = int(doc_off[0]), int(doc_off[-1])
        is_delim = np.zeros(256, dtype=bool)
        is_delim[np.frombuffer(delimiters, dtype=np.uint8)] = True
        nb = ~is_delim[text[base:end_]]                                       # byte belongs to a word
        n = len(nb)
        first = np.zeros(n, dtype=bool); last = np.zeros(n, dtype=bool)     # first / last byte of a document
        nonempty = doc_off[1:] > doc_off[:-1]
        first[doc_off[:-1][nonempty] - base] = True
        last[doc_off[1:][nonempty] - 1 - base] = True
        prev = np.zeros(n, dtype=bool); prev[1:] = nb[:-1]
        nxt = np.zeros(n, dtype=bool); nxt[:-1] = nb[1:]
        s_idx = np.flatnonzero(nb & (~prev | first))                          # a word starts behind a delimiter or a document start
        e_idx = np.flatnonzero(nb & (~nxt | last))
        wlen = e_idx - s_idx + 1
        sel = wlen > 64                                                       # only long words change the cost
        wlen = wlen[sel]
        wdoc = np.searchsorted(doc_off, s_idx[sel] + base, side="right") - 1
    extra = np.where(wlen > 12288, COST_HUGE_WORD - 1.0, np.where(wlen > 64, COST_LONG_WORD - 1.0, 0.0)) * wlen
    keep = (extra > 0) & (wdoc >= 0) & (wdoc < nd)
    return lens + np.bincount(wdoc[keep], weights=extra[keep], minlength=nd)[:nd]


def shard_bounds(doc_off: np.ndarray, n_shards: int, cost: np.ndarray = None) -> np.ndarray:
    """Balanced contiguous document ranges (north star: "sharded ... by byte-balanced ranges with no collective"):
    shard k takes documents [b[k], b[k+1]), cut at the document boundary nearest to k * total / n_shards.  The measure is
    bytes, or `cost` (one value per document, e.g. `document_costs`) for corpora whose bytes are not equally expensive."""
    doc_off = np.asarray(doc_off, dtype=np.uint64)
    nd = len(doc_off) - 1
    if cost is not None:
        acc = np.zeros(nd + 1, dtype=np.float64)
        np.cumsum(np.asarray(cost, dtype=np.float64), out=acc[1:])
    else:
        acc = doc_off.astype(np.float64) - float(doc_off[0])
    total = float(acc[-1])
    b = np.zeros(n_shards + 1, dtype=np.int64)
    for k in range(1, n_shards):
        target = total * k / n_shards
        i = int(np.searchsorted(acc, target, side="left"))
        if i > 0 and i <= nd and (target - acc[i - 1]) < (acc[min(i, nd)] - target):
            i -= 1
        b[k] = max(b[k - 1], min(i, nd))
    b[n_shards] = nd
    return b


def shard(text: np.ndarray, doc_off: np.ndarray, rank: int, world: int, cost: np.ndarray = None):
    """The (text, doc_off) slice rank `rank` of `world` encodes; offsets rebased to 0."""
    b = shard_bounds(doc_off, world, cost)
    lo, hi = int(b[rank]), int(b[rank + 1])
    base = int(doc_off[lo])
    return text[base:int(doc_off[hi])], (np.asarray(doc_off[lo:hi + 1], dtype=np.uint64) - np.uint64(base)), (lo, hi)
