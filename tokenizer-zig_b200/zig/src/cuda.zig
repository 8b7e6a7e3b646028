//! cuda.zig -- `extern fn` mirror of include/tokzig_b200.h (device layer only).
//! The host side of tokenizer-zig stays in Zig: src/lib.zig keeps its public API and calls these symbols, which
//! build.zig links from the static sm_100a library (libtokzig_b200.a) plus cudart.
//! NOT COMPILED in the build image (no zig toolchain there): kept a 1:1 transcription of the C header so review is
//! mechanical.

pub const Ctx = opaque {};

pub const OK: c_int = 0;
pub const ERR_OOM: c_int = -1; // error.OutOfMemory
pub const ERR_MISSING_UNK: c_int = -2; // error.MissingUnkToken (src/model/wordpiece.zig:150,212)
pub const ERR_INVALID_UTF8: c_int = -3; // reference: unreachable in Utf8Iterator (src/model/bpe.zig:186-187)
pub const ERR_CUDA: c_int = -4;
pub const ERR_INVALID_ARG: c_int = -5;

pub const MODEL_BPE: i32 = 0;
pub const MODEL_WORDPIECE: i32 = 1;
pub const CLS_WORD: u8 = 0;
pub const CLS_DELIM: u8 = 1;
pub const CLS_ISOLATE: u8 = 2;
pub const NORM_DROP: u16 = 0xFFFF;

pub const OUT_IDS: u32 = 1;
pub const OUT_OFFSETS: u32 = 2;
pub const OUT_ATTENTION: u32 = 4;
pub const OUT_TYPE_IDS: u32 = 8;
pub const OUT_SPECIAL: u32 = 16;
pub const OUT_ALL: u32 = 31;
pub const OUT_OFFSETS_PACKED: u32 = 32; // one u16 per token (start | end << 8) when every pre-token is < 256 bytes
pub const OUT_IDS_U16: u32 = 64;
pub const OUT_SPAN_TOKENS: u32 = 128; // 16-byte SpanToken records // ids as u16 when every vocabulary id is < 65536
pub const OUT_WORD_IDS: u32 = 256; // each token's pre-token index in its document, WORD_NONE for specials and padding (not in OUT_ALL)
pub const WORD_NONE: u32 = 0xFFFFFFFF;

pub const ModelDesc = extern struct {
    model_kind: i32,
    norm_lut: ?[*]const u16, // [256] or null
    class_lut: ?[*]const u8, // [256] or null
    vocab_bytes: ?[*]const u8,
    vocab_off: ?[*]const u64,
    vocab_ids: ?[*]const u32,
    vocab_n: u32,
    merge_first: ?[*]const u32,
    merge_second: ?[*]const u32,
    merge_rank: ?[*]const u32,
    merge_new: ?[*]const u32,
    merges_n: u32,
    has_unk: i32,
    unk_id: u32,
    prefix: ?[*]const u8,
    prefix_len: u32,
    max_input_chars_per_word: u64,
};

pub const EncodeParams = extern struct {
    has_truncation: i32 = 0,
    max_length: u64 = 0,
    has_padding: i32 = 0,
    pad_length: u64 = 0,
    pad_id: u32 = 0,
    pad_type_id: u32 = 0,
    pad_left: i32 = 0,
    outputs: u32 = OUT_ALL,
    fast: i32 = 0, // FastTokenizer.encode semantics (src/lib.zig:356-422)
    fast_max_sequence_length: u32 = 0, // 0 = 8192
    fast_max_tokens: u32 = 0, // 0 = 512
    // hf_compat (beyond the reference, opt-in; 0 = reference behaviour): single-sequence template + document-relative offsets
    hf_flags: u32 = 0, // HF_TEMPLATE | HF_DOC_OFFSETS
    tpl_n_prefix: u32 = 0,
    tpl_n_suffix: u32 = 0,
    tpl_prefix_id: [4]u32 = .{ 0, 0, 0, 0 },
    tpl_prefix_type: [4]u32 = .{ 0, 0, 0, 0 },
    tpl_suffix_id: [4]u32 = .{ 0, 0, 0, 0 },
    tpl_suffix_type: [4]u32 = .{ 0, 0, 0, 0 },
    tpl_seq_type: u32 = 0,
};
pub const HF_TEMPLATE: u32 = 1;
pub const HF_DOC_OFFSETS: u32 = 2;

pub const BatchResult = extern struct {
    n_docs: u64,
    n_tokens: u64,
    n_real_tokens: u64,
    doc_tok_off: ?[*]const u64,
    ids: ?[*]const u32,
    offsets: ?[*]const u32,
    attention_mask: ?[*]const u32,
    type_ids: ?[*]const u32,
    special_tokens_mask: ?[*]const u32,
    err_doc: i64,
    offsets_packed: ?[*]const u16,
    ids16: ?[*]const u16,
    span_tokens: ?[*]const u32, // 4 u32 per slot = SpanToken (src/token.zig:19-33)
    n_wide: u64, // offsets_packed: tokens whose u16 is 0xFFFF (pre-tokens of 256+ bytes)
    wide_tokens: ?[*]const u32, // {slot low, slot high, start, end} each, sorted by slot in host-buffer results
    word_ids: ?[*]const u32, // OUT_WORD_IDS: n_tokens entries
};

/// tkz_compact_result: kept real tokens only; masks and padding slots are rebuilt on the host (tkz_compact_expand)
pub const CompactResult = extern struct {
    n_docs: u64,
    n_kept: u64,
    n_real_tokens: u64,
    doc_kept_off: ?[*]const u64, // n_docs + 1
    ids: ?[*]const u32, // null when ids16 is delivered
    ids16: ?[*]const u16,
    offsets_packed: ?[*]const u16, // 0xFFFF = look the token up in wide_tokens; null when the call fell back to `offsets`
    offsets: ?[*]const u32,
    params: EncodeParams,
    err_doc: i64,
    n_wide: u64,
    wide_tokens: ?[*]const u32, // {kept index low, high, start, end}, sorted by kept index
};

pub const Stats = extern struct {
    arena_bytes: u64,
    n_words: u64,
    n_unique_words: u64,
    n_long_words: u64,
    kernel_launches: u64,
    ms_split: f32,
    ms_model: f32,
    ms_scan: f32,
    ms_emit: f32,
    ms_total: f32,
    model_flags: u32,
    ms_call_kernels: f32, // host-buffer calls: device time of all chunks of the last call
    reserved0: u32,
    path: u32, // pipeline of the last encode: 0 per-occurrence, 2 slice pipeline
};

pub const DecodeDesc = extern struct {
    tok_bytes: ?[*]const u8,
    tok_off: [*]const u64, // n_ids + 1
    n_ids: u32,
    special_ids: ?[*]const u32,
    n_special: u32,
    decoder_kind: i32, // 0 none, 1 WordPiece, 2 ByteLevel, 3 BPE (src/config.zig:459-530)
};
pub const DecodeResult = extern struct {
    n_seqs: u64,
    n_bytes: u64,
    byte_off: ?[*]const u64,
    bytes: ?[*]const u8,
};

pub extern fn tkz_ctx_create(device: c_int, stream: ?*anyopaque, arena_hint_bytes: u64, out: *?*Ctx) c_int;
pub extern fn tkz_ctx_destroy(ctx: ?*Ctx) void;
pub extern fn tkz_last_error(ctx: ?*Ctx) [*:0]const u8;
pub extern fn tkz_ctx_get_stats(ctx: *Ctx, out: *Stats) c_int;
pub extern fn tkz_model_upload(ctx: *Ctx, desc: *const ModelDesc) c_int;
pub extern fn tkz_encode_batch(ctx: *Ctx, text: ?[*]const u8, doc_off: [*]const u64, n_docs: u64, params: *const EncodeParams, out: *BatchResult) c_int;
pub extern fn tkz_encode_batch_device(ctx: *Ctx, d_text: ?*const anyopaque, d_doc_off: *const anyopaque, n_docs: u64, text_bytes: u64, params: *const EncodeParams, out: *BatchResult) c_int;
pub extern fn tkz_ctx_numa_node(ctx: *Ctx) c_int;
pub extern fn tkz_encode_batch_compact(ctx: *Ctx, text: ?[*]const u8, doc_off: [*]const u64, n_docs: u64, params: *const EncodeParams, want_offsets: c_int, out: *CompactResult) c_int;
pub extern fn tkz_compact_slots(r: *const CompactResult, d0: u64, d1: u64) u64;
pub extern fn tkz_compact_expand(r: *const CompactResult, d0: u64, d1: u64, doc_tok_off: ?[*]u64, ids: ?[*]u32, offsets: ?[*]u32, attention_mask: ?[*]u32, type_ids: ?[*]u32, special_tokens_mask: ?[*]u32) c_int;

// several GPUs of one box: one context + one host thread per GPU, no collective (include/tokzig_b200.h, tkzm_*)
pub const Pool = opaque {};
pub extern fn tkzm_create(devices: [*]const i32, n: i32, out: *?*Pool) c_int;
pub extern fn tkzm_destroy(pool: ?*Pool) void;
pub extern fn tkzm_size(pool: *Pool) i32;
pub extern fn tkzm_ctx(pool: *Pool, i: i32) ?*Ctx;
pub extern fn tkzm_last_error(pool: ?*Pool) [*:0]const u8;
pub extern fn tkzm_model_upload(pool: *Pool, desc: *const ModelDesc) c_int;
pub extern fn tkzm_shard_bounds(doc_off: [*]const u64, n_docs: u64, n_shards: i32, cost: ?[*]const f64, bounds: [*]u64) c_int;
pub extern fn tkzm_document_costs(text: ?[*]const u8, doc_off: [*]const u64, n_docs: u64, raw_class: ?[*]const u8, threads: i32, cost: [*]f64) c_int;
pub extern fn tkzm_encode_batch_compact(pool: *Pool, text: ?[*]const u8, doc_off: [*]const u64, n_docs: u64, params: *const EncodeParams, want_offsets: c_int, cost_balanced: c_int, bounds: [*]u64, results: [*]CompactResult, shard_ms: ?[*]f64) c_int;
pub extern fn tkz_decode_upload(ctx: *Ctx, desc: *const DecodeDesc) c_int;
pub extern fn tkz_decode_batch(ctx: *Ctx, ids: ?[*]const u32, seq_off: [*]const u64, n_seqs: u64, skip_special_tokens: c_int, out: *DecodeResult) c_int;
