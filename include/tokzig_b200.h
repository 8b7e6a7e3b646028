/*
 * tokzig_b200.h -- C ABI of the B200-native batch encoder that replaces the encode hot path of
 * jrc2139/tokenizer-zig (Tokenizer.encode, src/lib.zig:109-160, applied to a batch of documents).
 *
 * The reference has no FFI of its own (SURVEY.md 8b): its plug points are in-process Zig vtables that take ONE
 * pre-token per call (Model.tokenize src/model/model.zig:7,26-28; Normalizer.normalize src/normalizer/normalizer.zig:9,20;
 * PreTokenizer.preTokenize src/pretokenizer/pretokenizer.zig:16,27; PostProcessor.process src/processor/processor.zig:10,23).
 * This header is therefore the boundary the new src/lib.zig binds with `extern fn` (tokenizer-zig_b200/zig/src/cuda.zig);
 * every entry point names the reference interface it stands in for.
 *
 * Two layers, one shared library (libtokzig_b200.so) / static archive (libtokzig_b200.a):
 *   tkz_*   device layer: flattened model tables in, CSR batch encoding out.  No JSON, no strings.
 *   tkzh_*  host mirror of the reference's public API (Tokenizer.fromJson / encode / tokenToId ...), written in C++
 *           because no Zig toolchain exists in the build image; the Zig host layer binds the same tkz_* symbols.
 *
 * Conventions: plain pointers and sizes; 0 = ok, negative = error (codes below, mapped 1:1 onto the Zig error set);
 * inputs are borrowed for the duration of the call; results are owned by the context and stay valid until the next
 * encode on that context or tkz_ctx_destroy (the contract of SpanEncoding, "valid until next encode", src/lib.zig:353-356).
 * One context per GPU, not re-entrant.  There is NO CPU fallback: every call fails with TKZ_ERR_CUDA without a device.
 */
#ifndef TOKZIG_B200_H
#define TOKZIG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ status codes */
#define TKZ_OK 0
#define TKZ_ERR_OOM (-1)              /* error.OutOfMemory */
#define TKZ_ERR_MISSING_UNK (-2)      /* error.MissingUnkToken      src/model/wordpiece.zig:150,212 */
#define TKZ_ERR_INVALID_UTF8 (-3)     /* reference: `unreachable` in std.unicode.Utf8Iterator (src/model/bpe.zig:186-187) */
#define TKZ_ERR_CUDA (-4)             /* no device / driver error / extension not built for this device */
#define TKZ_ERR_INVALID_ARG (-5)
#define TKZ_ERR_INVALID_JSON (-10)    /* ConfigError.InvalidJson            src/config.zig:18-30 */
#define TKZ_ERR_MISSING_MODEL (-11)   /* ConfigError.MissingModel */
#define TKZ_ERR_UNSUPPORTED_MODEL (-12) /* ConfigError.UnsupportedModelType */
#define TKZ_ERR_MISSING_VOCAB (-13)   /* ConfigError.MissingVocab */
#define TKZ_ERR_INVALID_VOCAB_ENTRY (-14) /* ConfigError.InvalidVocabEntry */
#define TKZ_ERR_IO (-20)              /* file errors of Tokenizer.fromFile  src/lib.zig:48-56 */

/* ------------------------------------------------------------------ device layer */
typedef struct tkz_ctx tkz_ctx;   /* one per GPU: stream, device arenas (replace src/arena.zig), uploaded tables */

#define TKZ_MODEL_BPE 0           /* src/model/bpe.zig */
#define TKZ_MODEL_WORDPIECE 1     /* src/model/wordpiece.zig */

/* byte classes of the composed pre-tokenizer (class_lut) */
#define TKZ_CLS_WORD 0            /* part of a maximal run = one pre-token */
#define TKZ_CLS_DELIM 1           /* dropped separator */
#define TKZ_CLS_ISOLATE 2         /* its own one-byte pre-token (punctuation) */
#define TKZ_NORM_DROP 0xFFFFu     /* norm_lut value: byte removed by the normalizer */

/* Flattened model.  Built on the host from tokenizer.json (src/config.zig:59-117) or by hand, uploaded once.
 * The reference's normalizers and pre-tokenizers are all byte-wise (SURVEY.md section 0): any chain of them composes
 * into one 256-entry byte map and one 256-entry class table, which is what crosses the ABI. */
typedef struct tkz_model_desc {
    int32_t model_kind;                 /* TKZ_MODEL_*                               src/config.zig:130-138 */
    const uint16_t* norm_lut;           /* [256] normalised byte or TKZ_NORM_DROP; NULL = no normalizer
                                           (src/config.zig:364-379, src/normalizer/normalizer.zig:47-152) */
    const uint8_t* class_lut;           /* [256] TKZ_CLS_* of the NORMALISED byte; NULL = no pre-tokenizer: the whole
                                           document is one pre-token (src/lib.zig:121; src/config.zig:405-450,
                                           src/pretokenizer/pretokenizer.zig:49-241) */
    /* model vocabulary: n keys, bytes concatenated, off[n+1] (src/model/bpe.zig:38, src/model/wordpiece.zig:15) */
    const uint8_t* vocab_bytes;
    const uint64_t* vocab_off;
    const uint32_t* vocab_ids;
    uint32_t vocab_n;
    /* BPE merges already filtered and ranked by the loader rule of src/config.zig:228-273, in put order (a later
     * entry for the same pair overwrites): key = first<<32|second (Pair.hash src/model/bpe.zig:24-26) */
    const uint32_t* merge_first;
    const uint32_t* merge_second;
    const uint32_t* merge_rank;
    const uint32_t* merge_new;
    uint32_t merges_n;
    /* unknown token.  BPE: optional, used only if configured AND present in vocab (src/model/bpe.zig:198-207), else
     * the character is dropped.  WordPiece: has_unk = unk_token present in vocab; needing it when absent is
     * TKZ_ERR_MISSING_UNK (src/model/wordpiece.zig:150,212). */
    int32_t has_unk;
    uint32_t unk_id;
    /* WordPiece only (src/model/wordpiece.zig:17-19) */
    const uint8_t* prefix;              /* continuing_subword_prefix */
    uint32_t prefix_len;
    uint64_t max_input_chars_per_word;  /* compared with the pre-token's BYTE length */
} tkz_model_desc;

/* which output arrays a call materialises (ids always) */
#define TKZ_OUT_IDS 1u
#define TKZ_OUT_OFFSETS 2u
#define TKZ_OUT_ATTENTION 4u
#define TKZ_OUT_TYPE_IDS 8u
#define TKZ_OUT_SPECIAL 16u
#define TKZ_OUT_ALL 31u
/* Offsets as ONE u16 per token (start | end << 8) in tkz_batch_result.offsets_packed instead of two u32: possible because
 * the reference's offsets are relative to the pre-token (src/lib.zig:133-137).  The few tokens of pre-tokens of 256 bytes
 * or more get the value 0xFFFF (no real token has start = end = 255) and their offsets travel in a side list
 * (tkz_batch_result.n_wide / wide_tokens).  A batch where those tokens are many (above an eighth of all tokens or 4 M), a
 * tokenizer without pre-tokenizer, and TKZ_HF_DOC_OFFSETS fall back to TKZ_OUT_OFFSETS for the whole call: exactly one of
 * offsets / offsets_packed is then non-NULL. */
#define TKZ_OUT_OFFSETS_PACKED 32u
/* Ids as u16 in tkz_batch_result.ids16 instead of u32 in ids: honoured when every id of the uploaded vocabulary is below
 * 65536 (GPT-2- and BERT-sized vocabularies), ignored otherwise: exactly one of ids / ids16 is non-NULL. */
#define TKZ_OUT_IDS_U16 64u
/* SpanToken records (src/token.zig:11-76): 16 bytes per slot {id u32, start u32, end u32, type_id u8, flags u8, pad u16} in
 * tkz_batch_result.span_tokens; flags bit 2 = is_padding (SpanToken.initPadding), the other flags are never set by the path */
#define TKZ_OUT_SPAN_TOKENS 128u
/* Word ids (Hugging Face Encoding.word_ids for a single sequence) in tkz_batch_result.word_ids: for every real token the
 * ordinal of the pre-token that produced it among the pre-tokens of its document, counting from 0.  A pre-token that yields
 * no token still uses up its index; without a pre-tokenizer every token has word id 0; template special tokens and padding
 * slots get 0xFFFFFFFF; truncation keeps the kept tokens' word ids.  Works with any hf_flags (in reference mode the pieces of
 * the pre-tokenizer are the words).  Not part of TKZ_OUT_ALL.  TKZ_ERR_INVALID_ARG with `fast`, in the compact result
 * (tkz_encode_batch_compact / tkzm_encode_batch_compact), and with a model whose largest id is 2^22 or more. */
#define TKZ_OUT_WORD_IDS 256u

/* Per-call knobs = the public fields Tokenizer.truncation / Tokenizer.padding (src/lib.zig:41-42,149-157;
 * src/types.zig:39-45,55-59).  stride / strategy / pad_token are ignored by the reference's encode. */
typedef struct tkz_encode_params {
    int32_t has_truncation;
    uint64_t max_length;                /* Encoding.truncate  src/encoding.zig:363-380 */
    int32_t has_padding;                /* padding != null AND padding.length != null (src/encoding.zig:386) */
    uint64_t pad_length;                /* Encoding.pad       src/encoding.zig:385-463 */
    uint32_t pad_id;
    uint32_t pad_type_id;
    int32_t pad_left;
    uint32_t outputs;                   /* TKZ_OUT_* mask; 0 means TKZ_OUT_ALL */
    /* FastTokenizer.encode (src/lib.zig:356-422) instead of Tokenizer.encode: BPE.tokenizeFast / WordPiece.tokenizeFast
     * (heap pop order, stale entries, src/model/bpe.zig:285-430, src/model/wordpiece.zig:233-301) with the caps of the arena
     * (src/arena.zig:140-245): at most fast_max_sequence_length symbols per pre-token and / 4 pre-tokens per document, at most
     * fast_max_tokens tokens per document; truncation / padding above are ignored (FastTokenizer.encode applies none). */
    int32_t fast;
    uint32_t fast_max_sequence_length;  /* ArenaConfig.max_sequence_length (default 8192); 4 .. 65535 */
    uint32_t fast_max_tokens;           /* ArenaConfig.max_tokens (default 512) */
    /* hf_compat -- BEYOND the reference, opt-in, 0 = the reference's behaviour (SURVEY.md section 8(f) row 4).  What
     * src/processor/processor.zig:41-152 declares (BertProcessing, TemplateProcessing) and leaves as TODO, with the semantics of
     * Hugging Face tokenizers 0.22 (tests/golden/hf_compat_vectors.json): TKZ_HF_TEMPLATE puts tpl_n_prefix special tokens
     * before and tpl_n_suffix after every document's kept tokens (offsets (0,0), special 1, attention 1, their own type id),
     * gives the document's tokens tpl_seq_type, lets the added tokens count against max_length and towards pad_length;
     * TKZ_HF_DOC_OFFSETS reports offsets relative to the (normalised) document instead of the pre-token.  A caller passes the
     * prefix / suffix only when it encodes with add_special_tokens (tokenizers keeps the type id either way).  Not available in
     * the FastTokenizer mode and the compact result. */
    uint32_t hf_flags;                  /* TKZ_HF_* */
    uint32_t tpl_n_prefix, tpl_n_suffix;             /* <= TKZ_TPL_MAX each */
    uint32_t tpl_prefix_id[4], tpl_prefix_type[4], tpl_suffix_id[4], tpl_suffix_type[4];
    uint32_t tpl_seq_type;
} tkz_encode_params;
#define TKZ_HF_TEMPLATE 1u
#define TKZ_HF_DOC_OFFSETS 2u
#define TKZ_TPL_MAX 4u

/* CSR batch encoding = n_docs Encodings (src/encoding.zig:231-243) back to back.  Document d owns slots
 * [doc_tok_off[d], doc_tok_off[d+1]).  offsets holds (start,end) pairs (Offset, src/types.zig:4-11), byte offsets into
 * the NORMALISED PRE-TOKEN (the reference never adds the pre-token start, src/lib.zig:133-137).  Arrays not requested
 * in `outputs` are NULL.  Token strings are not materialised: tokens[i] == idToToken(ids[i]) always. */
typedef struct tkz_batch_result {
    uint64_t n_docs;
    uint64_t n_tokens;                  /* total slots incl. padding */
    uint64_t n_real_tokens;             /* model tokens before truncation/padding */
    const uint64_t* doc_tok_off;        /* n_docs + 1 */
    const uint32_t* ids;
    const uint32_t* offsets;            /* 2 * n_tokens */
    const uint32_t* attention_mask;
    const uint32_t* type_ids;
    const uint32_t* special_tokens_mask;
    int64_t err_doc;                    /* document index of the first error, -1 if none */
    const uint16_t* offsets_packed;     /* n_tokens x (start | end << 8), see TKZ_OUT_OFFSETS_PACKED; padding slots are 0 */
    const uint16_t* ids16;              /* n_tokens, see TKZ_OUT_IDS_U16 */
    const uint32_t* span_tokens;        /* 4 u32 per slot, see TKZ_OUT_SPAN_TOKENS */
    /* TKZ_OUT_OFFSETS_PACKED, tokens of pre-tokens of 256 bytes or more: their u16 is 0xFFFF and their offsets are here,
     * n_wide records of four u32 {slot low, slot high, start, end}; sorted by slot in host-buffer results, in no particular
     * order in device-resident results.  (A call with too many of them -- above an eighth of its tokens or 4 M -- delivers
     * 32-bit offsets for every token instead, as a call without pre-tokenizer does.) */
    uint64_t n_wide;
    const uint32_t* wide_tokens;
    const uint32_t* word_ids;           /* n_tokens, see TKZ_OUT_WORD_IDS; 0xFFFFFFFF for special tokens and padding */
} tkz_batch_result;

/* counters of the last encode (FastTokenizer.arenaMemoryUsage analogue, src/lib.zig:451-453) */
typedef struct tkz_stats {
    uint64_t arena_bytes;               /* device bytes held by the context */
    uint64_t n_words;                   /* pre-tokens */
    uint64_t n_unique_words;            /* pre-tokens actually run through the model (after per-batch dedup) */
    uint64_t n_long_words;              /* pre-tokens taken by the block-per-word path */
    uint64_t kernel_launches;           /* kernels launched by the last encode */
    /* device time of the last encode by stage, CUDA events on the context's stream (ms) */
    float ms_split;                     /* K0 + K1: normalise / classify / split */
    float ms_model;                     /* K3 | K4: BPE merge loop or WordPiece match */
    float ms_scan;                      /* prefix sums: tokens per word -> per document -> CSR */
    float ms_emit;                      /* K5: fused truncate / pad / output write */
    float ms_total;                     /* first kernel to last kernel */
    uint32_t model_flags;               /* bit 0: merge table proven "proper" -> long words use the windowed block kernels; bit 1: the last encode ran the grid-wide kernel on huge words; bit 2: it re-ran the slice pipeline with worst-case capacities */
    float ms_call_kernels;              /* host-buffer calls: device time of ALL chunks of the last call (sum of their ms_total) */
    uint32_t reserved0;
    uint32_t path;                      /* pipeline of the last encode: 0 per-occurrence, 2 slice pipeline
                                           (then ms_split = pass A, ms_model = word-list kernels, ms_emit = pass B) */
} tkz_stats;

/* `device` = CUDA ordinal.  `stream` = a cudaStream_t the caller owns (e.g. torch's current stream) or NULL for a
 * private stream.  arena_hint_bytes pre-sizes the device arenas (0 = grow on demand). */
int tkz_ctx_create(int device, void* stream, uint64_t arena_hint_bytes, tkz_ctx** out);
void tkz_ctx_destroy(tkz_ctx* ctx);
const char* tkz_last_error(tkz_ctx* ctx);           /* NULL ctx: last error of a failed tkz_ctx_create */
int tkz_ctx_get_stats(tkz_ctx* ctx, tkz_stats* out);
int tkz_ctx_numa_node(tkz_ctx* ctx);                /* NUMA node of the context's GPU (sysfs), -1 if unknown */

/* replaces BPE.init / WordPiece.init table construction (src/model/bpe.zig:84-110, src/model/wordpiece.zig:51-74) */
int tkz_model_upload(tkz_ctx* ctx, const tkz_model_desc* desc);

/* Replaces the caller loop over Tokenizer.encode (src/lib.zig:109-160): text = all documents back to back,
 * doc_off[n_docs+1] byte offsets into text.  HOST pointers (pinned preferred); result arrays are HOST pointers owned
 * by the context.  Total text must be < 4 GiB per call (offsets are u32, src/types.zig:4-6). */
int tkz_encode_batch(tkz_ctx* ctx, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs,
                     const tkz_encode_params* params, tkz_batch_result* out);

/* Compact batch encoding: ONLY what has to cross PCIe.  Everything in an Encoding that is a constant of (kept token count,
 * padding parameters) -- attention_mask, type_ids, special_tokens_mask, every padding slot (src/encoding.zig:246-294,
 * 385-463) -- is rebuilt on the host by tkz_compact_expand when and where the caller wants it; ids travel as u16 when the
 * vocabulary allows, offsets as one u16 per token (TKZ_OUT_OFFSETS_PACKED).  Truncation is applied on the device.
 * Arrays are HOST pointers owned by the context (valid until the next encode on it). */
typedef struct tkz_compact_result {
    uint64_t n_docs;
    uint64_t n_kept;                    /* real tokens after truncation, all documents */
    uint64_t n_real_tokens;             /* before truncation */
    const uint64_t* doc_kept_off;       /* n_docs + 1: document d keeps tokens [doc_kept_off[d], doc_kept_off[d+1]) */
    const uint32_t* ids;                /* n_kept, or NULL when ids16 is delivered */
    const uint16_t* ids16;
    const uint16_t* offsets_packed;     /* n_kept x (start | end << 8), 0xFFFF = see wide_tokens; or NULL (then offsets) */
    const uint32_t* offsets;            /* 2 * n_kept, or NULL */
    tkz_encode_params params;           /* truncation / padding the expanded Encodings have */
    int64_t err_doc;
    uint64_t n_wide;                    /* offsets_packed: kept tokens whose u16 is 0xFFFF, sorted by kept index */
    const uint32_t* wide_tokens;        /* {kept index low, high, start, end} each */
} tkz_compact_result;
int tkz_encode_batch_compact(tkz_ctx* ctx, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs,
                             const tkz_encode_params* params, int want_offsets, tkz_compact_result* out);
/* slots documents [d0, d1) occupy after padding (the sizes tkz_compact_expand needs) */
uint64_t tkz_compact_slots(const tkz_compact_result* r, uint64_t d0, uint64_t d1);
/* Encoding.fromTokens + Encoding.pad for documents [d0, d1) on the host: fills the arrays that are not NULL (offsets: 2 u32
 * per slot; doc_tok_off: d1 - d0 + 1 entries relative to d0).  Plain CPU code: nothing is tokenized here. */
int tkz_compact_expand(const tkz_compact_result* r, uint64_t d0, uint64_t d1, uint64_t* doc_tok_off, uint32_t* ids,
                       uint32_t* offsets, uint32_t* attention_mask, uint32_t* type_ids, uint32_t* special_tokens_mask);

/* Same, text and doc_off already DEVICE resident; result arrays are DEVICE pointers (scalars in *out are host
 * values).  All work is enqueued on the context's stream; the call returns after the stream has drained. */
int tkz_encode_batch_device(tkz_ctx* ctx, const void* d_text, const void* d_doc_off, uint64_t n_docs,
                            uint64_t text_bytes, const tkz_encode_params* params, tkz_batch_result* out);

/* ------------------------------------------------------------------ several GPUs of one box (SURVEY.md 8e)
 * N contexts on N GPUs, one host thread per GPU; documents are cut into N contiguous shards with NO collective on the data
 * path (they are independent); model tables are replicated.  Closest reference analogue: the per-thread arena pool,
 * src/arena.zig:252-335.  Every entry point below leaves the caller's current CUDA device unchanged. */
typedef struct tkzm_pool tkzm_pool;
int tkzm_create(const int32_t* devices, int32_t n, tkzm_pool** out);         /* devices[i] = CUDA ordinal of shard i's GPU */
void tkzm_destroy(tkzm_pool* pool);
int32_t tkzm_size(tkzm_pool* pool);
tkz_ctx* tkzm_ctx(tkzm_pool* pool, int32_t i);
const char* tkzm_last_error(tkzm_pool* pool);
int tkzm_model_upload(tkzm_pool* pool, const tkz_model_desc* desc);          /* the same tables on every GPU */
/* shard k = documents [bounds[k], bounds[k+1]), cut at the document boundary nearest to k / n_shards of the total of the
 * measure: bytes when cost is NULL ("byte-balanced ranges"), else cost[d] per document.  bounds has n_shards + 1 entries. */
int tkzm_shard_bounds(const uint64_t* doc_off, uint64_t n_docs, int32_t n_shards, const double* cost, uint64_t* bounds);
/* modelled encode cost per document in units of "one byte of ordinary text": its bytes, with the bytes inside pre-tokens of
 * 65..12288 bytes counted 20x and inside longer ones 36x (the measured per-byte times of the long-word kernels).
 * raw_class[256] = TKZ_CLS_* of every RAW byte, NULL = no pre-tokenizer.  One pass over the text on `threads` host threads
 * (0 = all).  For corpora with skewed document and word lengths (BASELINE config 5). */
int tkzm_document_costs(const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs, const uint8_t* raw_class, int32_t threads, double* cost);
/* The batch over all GPUs of the pool: cuts it (cost_balanced 0: by bytes, 1: by tkzm_document_costs, 2: bounds as given), runs one
 * tkz_encode_batch_compact per shard concurrently, and returns the cut (bounds[n + 1]) and the n compact results (arrays owned
 * by the shard's context; err_doc is a document index of the whole batch).  shard_ms (n entries, may be NULL) = wall time of
 * every shard's call. */
int tkzm_encode_batch_compact(tkzm_pool* pool, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs, const tkz_encode_params* params,
                              int want_offsets, int cost_balanced, uint64_t* bounds, tkz_compact_result* results, double* shard_ms);

/* ------------------------------------------------------------------ decode (the inverse direction, SURVEY.md 8f) */
/* Tables of Tokenizer.decode (src/lib.zig:163-189): token strings come from the MODEL vocabulary by id
 * (model_impl.idToToken); special_ids = ids flagged special in the ADDED vocabulary (skipped when skip_special_tokens,
 * src/lib.zig:169-177); decoder_kind as the config loader selects it (src/config.zig:459-530): 0 none, 1 "WordPiece"
 * (drops every "##" pair), 2 "ByteLevel" (copy), 3 "BPE" (U+0120 -> space). */
typedef struct tkz_decode_desc {
    const uint8_t* tok_bytes;
    const uint64_t* tok_off;            /* n_ids + 1; ids without a token have an empty range */
    uint32_t n_ids;
    const uint32_t* special_ids;
    uint32_t n_special;
    int32_t decoder_kind;
} tkz_decode_desc;
typedef struct tkz_decode_result {
    uint64_t n_seqs;
    uint64_t n_bytes;
    const uint64_t* byte_off;           /* n_seqs + 1: sequence s decodes to bytes[byte_off[s] .. byte_off[s+1]) */
    const uint8_t* bytes;
} tkz_decode_result;
int tkz_decode_upload(tkz_ctx* ctx, const tkz_decode_desc* desc);
/* Replaces the caller loop over Tokenizer.decode: ids = all sequences back to back, seq_off[n_seqs+1].  HOST pointers;
 * the result arrays are HOST pointers owned by the context (valid until the next decode on it). */
int tkz_decode_batch(tkz_ctx* ctx, const uint32_t* ids, const uint64_t* seq_off, uint64_t n_seqs, int skip_special_tokens,
                     tkz_decode_result* out);

/* ------------------------------------------------------------------ host mirror of src/lib.zig (C++ behind a C ABI) */
typedef struct tkzh_tokenizer tkzh_tokenizer;

/* Tokenizer.fromJson / fromFile  src/lib.zig:48-85 (+ src/config.zig:59-117).  `device` as in tkz_ctx_create;
 * device < 0 loads the configuration only (no context; encode then fails with TKZ_ERR_CUDA). */
int tkzh_from_json(const char* json, uint64_t len, int device, void* stream, tkzh_tokenizer** out);
int tkzh_from_file(const char* path, int device, void* stream, tkzh_tokenizer** out);
void tkzh_free(tkzh_tokenizer* t);                                   /* Tokenizer.deinit src/lib.zig:87-106 */
const char* tkzh_last_error(tkzh_tokenizer* t);                      /* NULL: last error of a failed tkzh_from_* */
tkz_ctx* tkzh_ctx(tkzh_tokenizer* t);

/* public fields truncation / padding  src/lib.zig:41-42 */
int tkzh_set_truncation(tkzh_tokenizer* t, int has, uint64_t max_length);
int tkzh_set_padding(tkzh_tokenizer* t, int has, int has_length, uint64_t length, uint32_t pad_id, uint32_t pad_type_id,
                     int pad_left);
/* hand-wiring normalizer_impl / pretokenizer_impl (src/lib.zig:37-38): op lists, see TKZH_NORM_* / TKZH_PT_*.
 * n = -1 removes the component (null); n = 0 installs an empty Sequence. */
#define TKZH_NORM_CFG_LOWER 1      /* src/config.zig:364-379 */
#define TKZH_NORM_BERT_STRUCT 2    /* src/normalizer/normalizer.zig:32-74  flags: 1 clean_text | 2 lowercase */
#define TKZH_NORM_LOWER_STRUCT 3   /* src/normalizer/normalizer.zig:77-98 */
#define TKZH_PT_WS_CFG 1           /* src/config.zig:440-450 */
#define TKZH_PT_BERT_CFG 2         /* src/config.zig:405-438 */
#define TKZH_PT_WS_STRUCT 3        /* src/pretokenizer/pretokenizer.zig:39-78 */
#define TKZH_PT_BERT_STRUCT 4      /* src/pretokenizer/pretokenizer.zig:81-133 */
#define TKZH_PT_BYTELEVEL_STRUCT 5 /* src/pretokenizer/pretokenizer.zig:136-183 */
int tkzh_set_normalizer(tkzh_tokenizer* t, const int32_t* kinds, const int32_t* flags, int32_t n);
int tkzh_set_pretokenizer(tkzh_tokenizer* t, const int32_t* kinds, int32_t n);

/* Tokenizer.encode src/lib.zig:109-160 for a batch (n_docs = 1 is the reference call).  add_special_tokens is
 * accepted and has no effect: every post-processor of the reference is a no-op (src/config.zig:551-555). */
int tkzh_encode_batch(tkzh_tokenizer* t, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs,
                      int add_special_tokens, uint32_t outputs, tkz_batch_result* out);

/* FastTokenizer.encode src/lib.zig:356-422 for a batch (FastTokenizerOptions.arena_config = {max_sequence_length, max_tokens},
 * src/lib.zig:240-246; 0 = the defaults 8192 / 512).  The result is the SpanEncoding of every document back to back: ids,
 * offsets, attention_mask 1, type_ids 0 and, with TKZ_OUT_SPAN_TOKENS, the 16-byte SpanToken records. */
int tkzh_encode_batch_fast(tkzh_tokenizer* t, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs,
                           uint32_t max_sequence_length, uint32_t max_tokens, uint32_t outputs, tkz_batch_result* out);

/* Tokenizer.decode  src/lib.zig:163-189 with the config-path decoders (src/config.zig:459-530): host side only (the
 * decode direction is outside the GPU hot path).  *out points into the tokenizer and is valid until the next decode. */
int tkzh_decode(tkzh_tokenizer* t, const uint32_t* ids, uint64_t n, int skip_special_tokens, const uint8_t** out, uint64_t* out_len);
/* the same for a batch of sequences on the GPU (tkz_decode_batch with this tokenizer's tables) */
int tkzh_decode_batch(tkzh_tokenizer* t, const uint32_t* ids, const uint64_t* seq_off, uint64_t n_seqs, int skip_special_tokens,
                      tkz_decode_result* out);

/* lookups  src/lib.zig:203-223 (added vocab first, then the model) */
uint64_t tkzh_get_vocab_size(tkzh_tokenizer* t);
int tkzh_token_to_id(tkzh_tokenizer* t, const uint8_t* token, uint64_t len, uint32_t* id);       /* 1 found, 0 not */
int tkzh_id_to_token(tkzh_tokenizer* t, uint32_t id, const uint8_t** token, uint64_t* len);       /* 1 found, 0 not */
/* the model's own map only (src/model/bpe.zig:258): the strings of Encoding.tokens, which ignore the added vocabulary */
int tkzh_model_id_to_token(tkzh_tokenizer* t, uint32_t id, const uint8_t** token, uint64_t* len);
/* hf_compat switch of the host mirror (TKZ_HF_* flags; 0 = the reference's behaviour, the default): with TKZ_HF_TEMPLATE the
 * single-sequence template of the tokenizer.json post_processor (BertProcessing, TemplateProcessing  specials* $A specials*)
 * is applied, its special tokens only when tkzh_encode_batch is called with add_special_tokens != 0.  Returns 1 when such a
 * template was found at load time, 0 when there is none to apply. */
int tkzh_set_hf_compat(tkzh_tokenizer* t, uint32_t flags);
/* the template found at load time (arrays of TKZ_TPL_MAX entries; any pointer may be NULL): 1 and the outputs filled, or 0 */
int tkzh_hf_template(tkzh_tokenizer* t, uint32_t* n_prefix, uint32_t* prefix_id, uint32_t* prefix_type, uint32_t* n_suffix,
                     uint32_t* suffix_id, uint32_t* suffix_type, uint32_t* seq_type);
int tkzh_add_special_tokens(tkzh_tokenizer* t, const uint8_t* contents, const uint64_t* off, uint64_t n, uint64_t* added);
/* loader facts used by the parity tests */
uint64_t tkzh_model_vocab_count(tkzh_tokenizer* t);
uint64_t tkzh_merge_count(tkzh_tokenizer* t);      /* distinct pairs in the merge map */
int tkzh_has_normalizer(tkzh_tokenizer* t);
int tkzh_has_pretokenizer(tkzh_tokenizer* t);
int tkzh_has_post_processor(tkzh_tokenizer* t);
uint64_t tkzh_added_token_count(tkzh_tokenizer* t);
int tkzh_added_token(tkzh_tokenizer* t, uint64_t i, const uint8_t** content, uint64_t* len, int64_t* id, int* special);
/* flattened model as uploaded (so a test can diff it against the oracle's loader) */
int tkzh_model_desc(tkzh_tokenizer* t, tkz_model_desc* out);

#ifdef __cplusplus
}
#endif
#endif /* TOKZIG_B200_H */
