// tokzig_host.cpp -- host mirror of the reference's public API (src/lib.zig:32-224) behind the tkzh_* C ABI.
//
// The reference's host language is Zig; no Zig toolchain exists in the build image, so this C++ layer is the testable
// host side above the tkz_* device ABI (the Zig layer in ../zig binds the same tkz_* symbols).  It restates
//   * the tokenizer.json loader            src/config.zig:59-117, 141-192, 194-295, 297-337, 339-362, 381-403, 532-549
//   * Tokenizer.{fromJson,fromFile,encode,tokenToId,idToToken,getVocabSize,addSpecialTokens}   src/lib.zig:48-223
//   * the added-token side vocabulary      src/vocab.zig:8-102
// and flattens the model for the GPU: any chain of the reference's byte-wise normalizers / pre-tokenizers is composed
// into one 256-entry byte map and one 256-entry class table (include/tokzig_b200.h).
// encode has NO CPU implementation here: it is one tkz_encode_batch call.
#include <cerrno>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/tokzig_b200.h"
#include "json.hpp"

namespace {

thread_local std::string g_load_error;

struct AddedToken {            // src/types.zig:14-31
    std::string content;
    bool has_id = false; uint32_t id = 0;
    bool single_word = false, lstrip = false, rstrip = false, normalized = true, special = false;
};

struct SideVocab {             // src/vocab.zig:8-102
    std::unordered_map<std::string, uint32_t> token_to_id;
    std::unordered_map<uint32_t, std::string> id_to_token;
    std::unordered_map<std::string, bool> special;
    uint32_t next_id = 0;
    bool add(const AddedToken& t, bool force_special) {          // addSpecialToken :39-58 / addToken :60-81
        if (token_to_id.count(t.content)) return false;
        const uint32_t id = t.has_id ? t.id : next_id;
        if (id >= next_id) next_id = id + 1;
        token_to_id[t.content] = id;
        id_to_token[id] = t.content;
        if (force_special || t.special) special[t.content] = true;
        return true;
    }
};

struct Op { int kind; int flags; };

}  // namespace

struct tkzh_tokenizer {
    std::string err;
    // model (src/model/bpe.zig:36-46, src/model/wordpiece.zig:13-20)
    int model_kind = TKZ_MODEL_WORDPIECE;
    std::vector<std::string> keys; std::vector<uint32_t> ids;            // JSON insertion order
    std::unordered_map<std::string, uint32_t> vocab;
    std::unordered_map<uint32_t, std::string> vocab_r;
    std::vector<uint32_t> mf, ms, mr, mn;                                 // accepted merges in put order
    std::unordered_map<uint64_t, uint32_t> merge_pairs;                   // distinct pairs (count only)
    bool has_unk_token = false; std::string unk_token;
    bool has_prefix = false; std::string prefix;
    bool has_suffix = false; std::string suffix;
    uint64_t max_chars = 100;
    // components (src/lib.zig:37-42)
    bool has_norm = false; std::vector<Op> norm_ops;
    bool has_pretok = false; std::vector<Op> pt_ops;
    bool has_post = false;
    // hf_compat (beyond the reference): the post-processor's single-sequence template, parsed but only applied when the caller
    // switches the mode on (tkzh_set_hf_compat); the reference's processors are no-ops (processor.zig:69-74, 147-152)
    bool has_template = false; uint32_t hf_flags = 0;
    std::vector<std::pair<uint32_t, uint32_t>> tpl_prefix, tpl_suffix; uint32_t tpl_seq_type = 0;    // (special id, type id)
    int decoder_kind = 0;
    std::vector<AddedToken> added_tokens;
    SideVocab added_vocab;
    bool has_trunc = false; uint64_t max_length = 512; uint64_t stride = 0;
    bool has_pad = false; bool pad_has_length = false; uint64_t pad_length = 0; uint32_t pad_id = 0, pad_type_id = 0; bool pad_left = false;
    // flattened
    std::vector<uint8_t> vocab_bytes; std::vector<uint64_t> vocab_off;
    uint16_t norm_lut[256]; uint8_t class_lut[256];
    tkz_model_desc desc{};
    std::string decode_buf;
    // device
    tkz_ctx* ctx = nullptr;
    bool dirty = true;
    bool decode_dirty = true;             // decode tables not uploaded yet / special set changed
};

namespace {

using tkzjson::Value;

const std::string* str_field(const Value* obj, const char* key) {        // config.zig:558-565
    const Value* v = obj->get(key);
    return (v && v->kind == Value::String) ? &v->s : nullptr;
}
bool bool_field(const Value* obj, const char* key, bool dflt) {           // config.zig:567-574 + orelse
    const Value* v = obj->get(key);
    return (v && v->kind == Value::Bool) ? v->b : dflt;
}

inline uint8_t ascii_lower(uint8_t c) { return (c >= 'A' && c <= 'Z') ? (uint8_t)(c + 32) : c; }
inline bool is_control(uint8_t c) { return (c < 0x20 && c != '\t' && c != '\n' && c != '\r') || c == 0x7F; }   // normalizer.zig:70-73
inline bool is_ws4(uint8_t c) { return c == ' ' || c == '\t' || c == '\n' || c == '\r'; }
inline bool is_ws6(uint8_t c) { return is_ws4(c) || c == 0x0B || c == 0x0C; }                                  // std.ascii.isWhitespace
inline bool is_punct(uint8_t c) { return (c >= 33 && c <= 47) || (c >= 58 && c <= 64) || (c >= 91 && c <= 96) || (c >= 123 && c <= 126); }

// Composes the op chains into the two tables that cross the ABI.
void build_luts(tkzh_tokenizer* t) {
    for (int b = 0; b < 256; b++) {
        uint16_t cur = (uint16_t)b;
        if (t->has_norm) for (const Op& op : t->norm_ops) {
            if (cur == TKZ_NORM_DROP) break;
            const uint8_t c = (uint8_t)cur;
            switch (op.kind) {
                case TKZH_NORM_CFG_LOWER: case TKZH_NORM_LOWER_STRUCT: cur = ascii_lower(c); break;
                case TKZH_NORM_BERT_STRUCT:
                    if ((op.flags & 1) && is_control(c)) cur = TKZ_NORM_DROP;
                    else if (op.flags & 2) cur = ascii_lower(c);
                    break;
                default: break;
            }
        }
        t->norm_lut[b] = cur;
        // class of a (normalised) byte value b under the pre-tokenizer chain: DELIM is absorbing, ISOLATE survives later
        // splitters unless one of them drops the byte (Sequence re-splits every piece, pretokenizer.zig:212-241)
        uint8_t cls = TKZ_CLS_WORD;
        if (t->has_pretok) for (const Op& op : t->pt_ops) {
            if (cls == TKZ_CLS_DELIM) break;
            const uint8_t c = (uint8_t)b;
            bool drop = false, iso = false;
            switch (op.kind) {
                case TKZH_PT_WS_CFG: case TKZH_PT_WS_STRUCT: case TKZH_PT_BYTELEVEL_STRUCT: drop = is_ws4(c); break;
                case TKZH_PT_BERT_CFG: drop = is_ws6(c); iso = is_punct(c); break;
                case TKZH_PT_BERT_STRUCT: drop = is_ws4(c); iso = is_punct(c); break;
                default: break;
            }
            if (drop) cls = TKZ_CLS_DELIM; else if (iso) cls = TKZ_CLS_ISOLATE;
        }
        t->class_lut[b] = cls;
    }
}

void build_desc(tkzh_tokenizer* t) {
    build_luts(t);
    tkz_model_desc& d = t->desc;
    memset(&d, 0, sizeof d);
    d.model_kind = t->model_kind;
    d.norm_lut = t->has_norm ? t->norm_lut : nullptr;
    d.class_lut = t->has_pretok ? t->class_lut : nullptr;
    d.vocab_bytes = t->vocab_bytes.data(); d.vocab_off = t->vocab_off.data(); d.vocab_ids = t->ids.data(); d.vocab_n = (uint32_t)t->keys.size();
    d.merge_first = t->mf.data(); d.merge_second = t->ms.data(); d.merge_rank = t->mr.data(); d.merge_new = t->mn.data(); d.merges_n = (uint32_t)t->mf.size();
    d.has_unk = 0; d.unk_id = 0;
    if (t->has_unk_token) { auto it = t->vocab.find(t->unk_token); if (it != t->vocab.end()) { d.has_unk = 1; d.unk_id = it->second; } }
    d.prefix = (const uint8_t*)t->prefix.data(); d.prefix_len = (uint32_t)t->prefix.size();
    d.max_input_chars_per_word = t->max_chars;
}

int fail(tkzh_tokenizer* t, int code, const char* msg) { g_load_error = msg; delete t; return code; }

int64_t int_of(const Value* v, int64_t dflt) { return (v && v->kind == Value::Integer) ? v->i : dflt; }
// hf_compat: the single-sequence template  specials* $A specials*  of a post_processor as tokenizers 0.22 serialises it --
// TemplateProcessing {single: [{SpecialToken: {id, type_id}} | {Sequence: {id, type_id}}], special_tokens: {name: {ids}}} or
// BertProcessing {sep: [token, id], cls: [token, id]}.  Anything else (a second sequence, an unknown special token, more than
// TKZ_TPL_MAX ids on a side) leaves has_template false.
void parse_template(tkzh_tokenizer* t, const Value* pp, const std::string& type) {
    std::vector<std::pair<uint32_t, uint32_t>> pre, suf; uint32_t seq_type = 0;
    if (type == "BertProcessing") {
        const Value* cls = pp->get("cls"); const Value* sep = pp->get("sep");
        if (!cls || !sep || cls->kind != Value::Array || sep->kind != Value::Array || cls->arr.size() != 2 || sep->arr.size() != 2) return;
        if (cls->arr[1]->kind != Value::Integer || sep->arr[1]->kind != Value::Integer) return;
        pre.push_back({(uint32_t)cls->arr[1]->i, 0u}); suf.push_back({(uint32_t)sep->arr[1]->i, 0u});
    } else if (type == "TemplateProcessing") {
        const Value* single = pp->get("single"); const Value* specials = pp->get("special_tokens");
        if (!single || single->kind != Value::Array) return;
        bool seen = false;
        for (const auto& piece : single->arr) {
            if (piece->kind != Value::Object) return;
            if (const Value* sq = piece->get("Sequence")) {
                const std::string* id = str_field(sq, "id");
                if (seen || !id || *id != "A") return;
                seen = true; seq_type = (uint32_t)int_of(sq->get("type_id"), 0);
            } else if (const Value* sp = piece->get("SpecialToken")) {
                const std::string* id = str_field(sp, "id");
                const Value* def = (id && specials) ? specials->get(*id) : nullptr;
                const Value* ids = def ? def->get("ids") : nullptr;
                if (!ids || ids->kind != Value::Array) return;
                const uint32_t ty = (uint32_t)int_of(sp->get("type_id"), 0);
                for (const auto& x : ids->arr) { if (x->kind != Value::Integer) return; (seen ? suf : pre).push_back({(uint32_t)x->i, ty}); }
            } else return;
        }
        if (!seen) return;
    } else return;
    if (pre.size() > TKZ_TPL_MAX || suf.size() > TKZ_TPL_MAX) return;
    t->has_template = true; t->tpl_prefix = pre; t->tpl_suffix = suf; t->tpl_seq_type = seq_type;
}

int load(const char* json, uint64_t len, tkzh_tokenizer** out) {
    tkzh_tokenizer* t = new tkzh_tokenizer();
    tkzjson::Parser parser(json, (size_t)len);
    tkzjson::ValuePtr root = parser.parse();
    if (!root || root->kind != Value::Object) return fail(t, TKZ_ERR_INVALID_JSON, "InvalidJson");        // config.zig:60-68
    const Value* model = root->get("model");
    if (!model || model->kind != Value::Object) return fail(t, TKZ_ERR_MISSING_MODEL, "MissingModel");     // :125-128
    const std::string* mt = str_field(model, "type");
    const std::string model_type = mt ? *mt : "WordPiece";                                                 // :130
    if (model_type == "WordPiece") t->model_kind = TKZ_MODEL_WORDPIECE;
    else if (model_type == "BPE") t->model_kind = TKZ_MODEL_BPE;
    else return fail(t, TKZ_ERR_UNSUPPORTED_MODEL, "UnsupportedModelType");                                // :136-138
    const Value* vocab = model->get("vocab");
    if (!vocab || vocab->kind != Value::Object) return fail(t, TKZ_ERR_MISSING_VOCAB, "MissingVocab");     // :143-146, 196-199
    t->vocab_off.push_back(0);
    for (auto& kv : vocab->obj) {
        if (kv.second->kind != Value::Integer) return fail(t, TKZ_ERR_INVALID_VOCAB_ENTRY, "InvalidVocabEntry");   // :162-164
        const uint32_t id = (uint32_t)kv.second->i;                                                         // @intCast
        t->keys.push_back(kv.first); t->ids.push_back(id);
        t->vocab[kv.first] = id; t->vocab_r[id] = kv.first;
        t->vocab_bytes.insert(t->vocab_bytes.end(), kv.first.begin(), kv.first.end());
        t->vocab_off.push_back(t->vocab_bytes.size());
    }
    if (t->vocab_bytes.empty()) t->vocab_bytes.push_back(0);
    if (t->model_kind == TKZ_MODEL_WORDPIECE) {
        const std::string* u = str_field(model, "unk_token");
        t->has_unk_token = true; t->unk_token = u ? *u : "[UNK]";                                           // :172
        const std::string* p = str_field(model, "continuing_subword_prefix");
        t->has_prefix = true; t->prefix = p ? *p : "##";                                                    // :173
        const Value* mc = model->get("max_input_chars_per_word");
        t->max_chars = (mc && mc->kind == Value::Integer) ? (uint64_t)mc->i : 100;                          // :174-177
    } else {
        const Value* merges = model->get("merges");
        if (merges && merges->kind == Value::Array) {                                                       // :228-229
            uint32_t rank = 0;
            for (auto& item : merges->arr) {
                std::string first, second;
                if (item->kind == Value::String) {                                                          // :236-241 splitScalar(' ')
                    const std::string& s = item->s;
                    const size_t a = s.find(' ');
                    if (a == std::string::npos) continue;                                                   // no second part
                    first = s.substr(0, a);
                    const size_t b = s.find(' ', a + 1);
                    second = s.substr(a + 1, b == std::string::npos ? std::string::npos : b - a - 1);
                } else if (item->kind == Value::Array && item->arr.size() == 2) {                           // :242-248
                    if (item->arr[0]->kind != Value::String || item->arr[1]->kind != Value::String) continue;
                    first = item->arr[0]->s; second = item->arr[1]->s;
                } else continue;
                auto fi = t->vocab.find(first); if (fi == t->vocab.end()) continue;                         // :254
                auto si = t->vocab.find(second); if (si == t->vocab.end()) continue;                        // :255
                if (first.size() + second.size() > 512) continue;                                           // :258-260
                auto ni = t->vocab.find(first + second); if (ni == t->vocab.end()) continue;                // :266
                t->mf.push_back(fi->second); t->ms.push_back(si->second); t->mr.push_back(rank); t->mn.push_back(ni->second);
                t->merge_pairs[((uint64_t)fi->second << 32) | si->second] = rank;                           // put :269
                rank++;                                                                                     // :270
            }
        }
        const std::string* u = str_field(model, "unk_token");
        if (u) { t->has_unk_token = true; t->unk_token = *u; }                                              // :276, 281
        const std::string* p = str_field(model, "continuing_subword_prefix");
        if (p) { t->has_prefix = true; t->prefix = *p; }                                                    // stored, unused by encode (bpe.zig:188)
        const std::string* sfx = str_field(model, "end_of_word_suffix");
        if (sfx) { t->has_suffix = true; t->suffix = *sfx; }
    }
    const Value* at = root->get("added_tokens");                                                           // :82-86, 297-337
    if (at && at->kind == Value::Array) {
        for (auto& item : at->arr) {
            if (item->kind != Value::Object) continue;
            const std::string* content = str_field(item.get(), "content");
            if (!content) continue;
            AddedToken a; a.content = *content;
            const Value* idv = item->get("id");
            if (idv && idv->kind == Value::Integer) { a.has_id = true; a.id = (uint32_t)idv->i; }
            a.special = bool_field(item.get(), "special", false);
            a.single_word = bool_field(item.get(), "single_word", false);
            a.lstrip = bool_field(item.get(), "lstrip", false);
            a.rstrip = bool_field(item.get(), "rstrip", false);
            a.normalized = bool_field(item.get(), "normalized", true);
            t->added_tokens.push_back(a);
        }
    }
    const Value* nv = root->get("normalizer");                                                             // :89-93, 339-362
    if (nv && nv->kind == Value::Object) {
        const std::string* ty = str_field(nv, "type");
        if (ty && (*ty == "BertNormalizer" || *ty == "Lowercase")) { t->has_norm = true; t->norm_ops.push_back({TKZH_NORM_CFG_LOWER, 0}); }
    }
    const Value* pv = root->get("pre_tokenizer");                                                          // :96-100, 381-403
    if (pv && pv->kind == Value::Object) {
        const std::string* ty = str_field(pv, "type");
        if (ty && *ty == "BertPreTokenizer") { t->has_pretok = true; t->pt_ops.push_back({TKZH_PT_BERT_CFG, 0}); }
        else if (ty && (*ty == "Whitespace" || *ty == "WhitespaceSplit")) { t->has_pretok = true; t->pt_ops.push_back({TKZH_PT_WS_CFG, 0}); }
    }
    const Value* dv = root->get("decoder");                                                                // :103-107, 459-486
    if (dv && dv->kind == Value::Object) {
        const std::string* ty = str_field(dv, "type");
        if (ty && *ty == "WordPiece") t->decoder_kind = 1; else if (ty && *ty == "ByteLevel") t->decoder_kind = 2; else if (ty && *ty == "BPE") t->decoder_kind = 3;
    }
    const Value* ppv = root->get("post_processor");                                                        // :110-114, 532-549 (a no-op either way)
    if (ppv && ppv->kind == Value::Object) {
        const std::string* ty = str_field(ppv, "type");
        if (ty && (*ty == "TemplateProcessing" || *ty == "BertProcessing")) t->has_post = true;
        if (ty) parse_template(t, ppv, *ty);
    }
    for (const AddedToken& a : t->added_tokens) t->added_vocab.add(a, a.special);                          // lib.zig:66-72
    build_desc(t);
    *out = t;
    return TKZ_OK;
}

int sync_device(tkzh_tokenizer* t) {
    if (!t->ctx) { t->err = "tokenizer was loaded without a device (tokzig_b200 has no CPU fallback)"; return TKZ_ERR_CUDA; }
    if (!t->dirty) return TKZ_OK;
    build_desc(t);
    int rc = tkz_model_upload(t->ctx, &t->desc);
    if (rc != TKZ_OK) { t->err = tkz_last_error(t->ctx); return rc; }
    t->dirty = false;
    return TKZ_OK;
}

}  // namespace

extern "C" int tkzh_from_json(const char* json, uint64_t len, int device, void* stream, tkzh_tokenizer** out) {
    if (!out || !json) return TKZ_ERR_INVALID_ARG;
    *out = nullptr;
    tkzh_tokenizer* t = nullptr;
    int rc = load(json, len, &t);
    if (rc != TKZ_OK) return rc;
    if (device >= 0) {
        rc = tkz_ctx_create(device, stream, 0, &t->ctx);
        if (rc != TKZ_OK) { g_load_error = tkz_last_error(nullptr); delete t; return rc; }
        rc = sync_device(t);
        if (rc != TKZ_OK) { g_load_error = t->err; tkz_ctx_destroy(t->ctx); delete t; return rc; }
    }
    *out = t;
    return TKZ_OK;
}

extern "C" int tkzh_from_file(const char* path, int device, void* stream, tkzh_tokenizer** out) {
    if (!out || !path) return TKZ_ERR_INVALID_ARG;
    *out = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) { g_load_error = std::string("cannot open ") + path; return TKZ_ERR_IO; }
    std::string buf; char tmp[1 << 16]; size_t n;
    while ((n = fread(tmp, 1, sizeof tmp, f)) > 0) {
        buf.append(tmp, n);
        if (buf.size() > 100ull * 1024 * 1024) { fclose(f); g_load_error = "tokenizer.json larger than 100 MiB"; return TKZ_ERR_IO; }   // lib.zig:52
    }
    fclose(f);
    return tkzh_from_json(buf.data(), buf.size(), device, stream, out);
}

extern "C" void tkzh_free(tkzh_tokenizer* t) { if (!t) return; if (t->ctx) tkz_ctx_destroy(t->ctx); delete t; }
extern "C" const char* tkzh_last_error(tkzh_tokenizer* t) { return t ? t->err.c_str() : g_load_error.c_str(); }
extern "C" tkz_ctx* tkzh_ctx(tkzh_tokenizer* t) { return t ? t->ctx : nullptr; }

extern "C" int tkzh_set_truncation(tkzh_tokenizer* t, int has, uint64_t max_length) {
    if (!t) return TKZ_ERR_INVALID_ARG;
    t->has_trunc = has != 0; t->max_length = max_length; return TKZ_OK;
}
extern "C" int tkzh_set_truncation_stride(tkzh_tokenizer* t, uint64_t stride) {
    if (!t) return TKZ_ERR_INVALID_ARG;
    t->stride = stride; return TKZ_OK;
}
extern "C" int tkzh_set_padding(tkzh_tokenizer* t, int has, int has_length, uint64_t length, uint32_t pad_id, uint32_t pad_type_id, int pad_left) {
    if (!t) return TKZ_ERR_INVALID_ARG;
    t->has_pad = has != 0; t->pad_has_length = has_length != 0; t->pad_length = length; t->pad_id = pad_id; t->pad_type_id = pad_type_id; t->pad_left = pad_left != 0;
    return TKZ_OK;
}
extern "C" int tkzh_set_normalizer(tkzh_tokenizer* t, const int32_t* kinds, const int32_t* flags, int32_t n) {
    if (!t || (n > 0 && !kinds)) return TKZ_ERR_INVALID_ARG;
    t->norm_ops.clear(); t->has_norm = n >= 0;
    for (int32_t i = 0; i < n; i++) t->norm_ops.push_back({kinds[i], flags ? flags[i] : 0});
    t->dirty = true; build_desc(t);
    return TKZ_OK;
}
extern "C" int tkzh_set_pretokenizer(tkzh_tokenizer* t, const int32_t* kinds, int32_t n) {
    if (!t || (n > 0 && !kinds)) return TKZ_ERR_INVALID_ARG;
    t->pt_ops.clear(); t->has_pretok = n >= 0;
    for (int32_t i = 0; i < n; i++) t->pt_ops.push_back({kinds[i], 0});
    t->dirty = true; build_desc(t);
    return TKZ_OK;
}

extern "C" int tkzh_encode_batch(tkzh_tokenizer* t, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs, int add_special_tokens,
                                 uint32_t outputs, tkz_batch_result* out) {
    if (!t || !out) return TKZ_ERR_INVALID_ARG;
    // lib.zig:143-147 -> config.zig:551-555: every post-processor is a no-op, add_special_tokens changes nothing -- unless the
    // caller opted into hf_compat (tkzh_set_hf_compat), where it decides whether the template's special tokens go in
    int rc = sync_device(t);
    if (rc != TKZ_OK) return rc;
    tkz_encode_params p{};
    p.has_truncation = t->has_trunc; p.max_length = t->max_length;                // lib.zig:150-152
    p.has_padding = t->has_pad && t->pad_has_length; p.pad_length = t->pad_length; // lib.zig:155-157, encoding.zig:386
    p.pad_id = t->pad_id; p.pad_type_id = t->pad_type_id; p.pad_left = t->pad_left; p.outputs = outputs;
    p.hf_flags = t->hf_flags & (TKZ_HF_DOC_OFFSETS | TKZ_HF_OVERFLOW);
    p.stride = t->stride;
    if ((t->hf_flags & TKZ_HF_TEMPLATE) && t->has_template) {
        p.hf_flags |= TKZ_HF_TEMPLATE; p.tpl_seq_type = t->tpl_seq_type;
        if (add_special_tokens) {
            p.tpl_n_prefix = (uint32_t)t->tpl_prefix.size(); p.tpl_n_suffix = (uint32_t)t->tpl_suffix.size();
            for (size_t i = 0; i < t->tpl_prefix.size(); i++) { p.tpl_prefix_id[i] = t->tpl_prefix[i].first; p.tpl_prefix_type[i] = t->tpl_prefix[i].second; }
            for (size_t i = 0; i < t->tpl_suffix.size(); i++) { p.tpl_suffix_id[i] = t->tpl_suffix[i].first; p.tpl_suffix_type[i] = t->tpl_suffix[i].second; }
        }
    }
    rc = tkz_encode_batch(t->ctx, text, doc_off, n_docs, &p, out);
    if (rc != TKZ_OK) t->err = tkz_last_error(t->ctx);
    return rc;
}
// FastTokenizer.encode (src/lib.zig:356-422) for a batch: same components, arena variants of the models, arena caps; no
// truncation / padding.  One tkz_encode_batch call in fast mode (csrc/tkz_fast.cuh).
extern "C" int tkzh_encode_batch_fast(tkzh_tokenizer* t, const uint8_t* text, const uint64_t* doc_off, uint64_t n_docs,
                                      uint32_t max_sequence_length, uint32_t max_tokens, uint32_t outputs, tkz_batch_result* out) {
    if (!t || !out) return TKZ_ERR_INVALID_ARG;
    int rc = sync_device(t);
    if (rc != TKZ_OK) return rc;
    tkz_encode_params p{};
    p.outputs = outputs;
    p.fast = 1; p.fast_max_sequence_length = max_sequence_length; p.fast_max_tokens = max_tokens;   // FastTokenizerOptions, lib.zig:240-246
    rc = tkz_encode_batch(t->ctx, text, doc_off, n_docs, &p, out);
    if (rc != TKZ_OK) t->err = tkz_last_error(t->ctx);
    return rc;
}

extern "C" int tkzh_decode(tkzh_tokenizer* t, const uint32_t* ids, uint64_t n, int skip_special_tokens, const uint8_t** out, uint64_t* out_len) {
    if (!t || !out || !out_len || (n && !ids)) return TKZ_ERR_INVALID_ARG;
    std::string r;
    for (uint64_t i = 0; i < n; i++) {                                   // lib.zig:167-179
        if (skip_special_tokens) {
            auto a = t->added_vocab.id_to_token.find(ids[i]);
            if (a != t->added_vocab.id_to_token.end() && t->added_vocab.special.count(a->second)) continue;
        }
        auto m = t->vocab_r.find(ids[i]);                                // model_impl.idToToken (not the added vocab)
        if (m != t->vocab_r.end()) r += m->second;
    }
    std::string& o = t->decode_buf;
    o.clear();
    if (t->decoder_kind == 1) {                                          // wordPieceDecodeImpl config.zig:488-505: drops every "##"
        for (size_t i = 0; i < r.size();) { if (i + 1 < r.size() && r[i] == '#' && r[i + 1] == '#') i += 2; else o.push_back(r[i++]); }
    } else if (t->decoder_kind == 3) {                                   // bpeDecodeImpl config.zig:512-530: U+0120 -> space
        for (size_t i = 0; i < r.size();) {
            if (i + 1 < r.size() && (uint8_t)r[i] == 0xC4 && (uint8_t)r[i + 1] == 0xA0) { o.push_back(' '); i += 2; } else o.push_back(r[i++]);
        }
    } else o = r;                                                        // ByteLevel copies (config.zig:507-510); none: lib.zig:188
    *out = (const uint8_t*)o.data(); *out_len = o.size();
    return TKZ_OK;
}

// Tokenizer.decode for a batch on the GPU: same tables as tkzh_decode (model vocabulary by id, special ids of the added
// vocabulary, decoder kind), flattened once and re-uploaded when addSpecialTokens changed the special set.
extern "C" int tkzh_decode_batch(tkzh_tokenizer* t, const uint32_t* ids, const uint64_t* seq_off, uint64_t n_seqs, int skip_special_tokens,
                                 tkz_decode_result* out) {
    if (!t || !out || !seq_off) return TKZ_ERR_INVALID_ARG;
    if (!t->ctx) { t->err = "tokenizer was loaded without a device (tokzig_b200 has no CPU fallback)"; return TKZ_ERR_CUDA; }
    if (t->decode_dirty) {
        uint32_t n_ids = 0;
        for (auto& kv : t->vocab_r) n_ids = std::max(n_ids, kv.first + 1);
        std::vector<uint64_t> off((size_t)n_ids + 1, 0);
        for (auto& kv : t->vocab_r) off[kv.first + 1] = kv.second.size();
        for (uint32_t i = 0; i < n_ids; i++) off[i + 1] += off[i];
        std::vector<uint8_t> bytes((size_t)off[n_ids]);
        for (auto& kv : t->vocab_r) if (!kv.second.empty()) memcpy(bytes.data() + off[kv.first], kv.second.data(), kv.second.size());
        std::vector<uint32_t> special;
        for (auto& kv : t->added_vocab.id_to_token) if (t->added_vocab.special.count(kv.second)) special.push_back(kv.first);
        tkz_decode_desc d{bytes.data(), off.data(), n_ids, special.data(), (uint32_t)special.size(), t->decoder_kind};
        int rc = tkz_decode_upload(t->ctx, &d);
        if (rc != TKZ_OK) { t->err = tkz_last_error(t->ctx); return rc; }
        t->decode_dirty = false;
    }
    int rc = tkz_decode_batch(t->ctx, ids, seq_off, n_seqs, skip_special_tokens, out);
    if (rc != TKZ_OK) t->err = tkz_last_error(t->ctx);
    return rc;
}

extern "C" uint64_t tkzh_get_vocab_size(tkzh_tokenizer* t) { return t->vocab.size() + t->added_vocab.token_to_id.size(); }   // lib.zig:203-205
extern "C" int tkzh_token_to_id(tkzh_tokenizer* t, const uint8_t* token, uint64_t len, uint32_t* id) {                         // lib.zig:208-214
    std::string k((const char*)token, (size_t)len);
    auto a = t->added_vocab.token_to_id.find(k);
    if (a != t->added_vocab.token_to_id.end()) { *id = a->second; return 1; }
    auto m = t->vocab.find(k);
    if (m != t->vocab.end()) { *id = m->second; return 1; }
    return 0;
}
extern "C" int tkzh_id_to_token(tkzh_tokenizer* t, uint32_t id, const uint8_t** token, uint64_t* len) {                         // lib.zig:217-223
    auto a = t->added_vocab.id_to_token.find(id);
    if (a != t->added_vocab.id_to_token.end()) { *token = (const uint8_t*)a->second.data(); *len = a->second.size(); return 1; }
    auto m = t->vocab_r.find(id);
    if (m != t->vocab_r.end()) { *token = (const uint8_t*)m->second.data(); *len = m->second.size(); return 1; }
    return 0;
}
// the MODEL's own id -> token map only: what Tokenizer.encode puts into Encoding.tokens (bpe.zig:258 `vocab_r.get(id) orelse ""`);
// an added token that shares the id does not change it
extern "C" int tkzh_model_id_to_token(tkzh_tokenizer* t, uint32_t id, const uint8_t** token, uint64_t* len) {
    auto m = t->vocab_r.find(id);
    if (m == t->vocab_r.end()) return 0;
    *token = (const uint8_t*)m->second.data(); *len = m->second.size();
    return 1;
}
extern "C" int tkzh_add_special_tokens(tkzh_tokenizer* t, const uint8_t* contents, const uint64_t* off, uint64_t n, uint64_t* added) {   // lib.zig:192-200
    uint64_t c = 0;
    for (uint64_t i = 0; i < n; i++) {
        AddedToken a; a.content.assign((const char*)contents + off[i], (size_t)(off[i + 1] - off[i])); a.special = true;
        if (t->added_vocab.add(a, true)) c++;
    }
    if (added) *added = c;
    if (c) t->decode_dirty = true;
    return TKZ_OK;
}
extern "C" uint64_t tkzh_model_vocab_count(tkzh_tokenizer* t) { return t->vocab.size(); }
extern "C" uint64_t tkzh_merge_count(tkzh_tokenizer* t) { return t->merge_pairs.size(); }
extern "C" int tkzh_has_normalizer(tkzh_tokenizer* t) { return t->has_norm; }
extern "C" int tkzh_has_pretokenizer(tkzh_tokenizer* t) { return t->has_pretok; }
extern "C" int tkzh_has_post_processor(tkzh_tokenizer* t) { return t->has_post; }
// hf_compat switch (TKZ_HF_* flags; 0 = the reference's behaviour, the default).  Returns 1 when the tokenizer.json carried a
// single-sequence template this mode can apply, 0 when TKZ_HF_TEMPLATE will have no effect.
// the parsed single-sequence template (what TKZ_HF_TEMPLATE will apply): ids / type ids into arrays of TKZ_TPL_MAX entries.
// Returns 1 and fills the outputs when the tokenizer.json carried one, 0 otherwise.
extern "C" int tkzh_hf_template(tkzh_tokenizer* t, uint32_t* n_prefix, uint32_t* prefix_id, uint32_t* prefix_type, uint32_t* n_suffix,
                                uint32_t* suffix_id, uint32_t* suffix_type, uint32_t* seq_type) {
    if (!t) return TKZ_ERR_INVALID_ARG;
    if (!t->has_template) return 0;
    if (n_prefix) *n_prefix = (uint32_t)t->tpl_prefix.size();
    if (n_suffix) *n_suffix = (uint32_t)t->tpl_suffix.size();
    for (size_t i = 0; i < t->tpl_prefix.size(); i++) { if (prefix_id) prefix_id[i] = t->tpl_prefix[i].first; if (prefix_type) prefix_type[i] = t->tpl_prefix[i].second; }
    for (size_t i = 0; i < t->tpl_suffix.size(); i++) { if (suffix_id) suffix_id[i] = t->tpl_suffix[i].first; if (suffix_type) suffix_type[i] = t->tpl_suffix[i].second; }
    if (seq_type) *seq_type = t->tpl_seq_type;
    return 1;
}
extern "C" int tkzh_set_hf_compat(tkzh_tokenizer* t, uint32_t flags) {
    if (!t) return TKZ_ERR_INVALID_ARG;
    t->hf_flags = flags & (TKZ_HF_TEMPLATE | TKZ_HF_DOC_OFFSETS | TKZ_HF_OVERFLOW);
    return t->has_template ? 1 : 0;
}
extern "C" uint64_t tkzh_added_token_count(tkzh_tokenizer* t) { return t->added_tokens.size(); }
extern "C" int tkzh_added_token(tkzh_tokenizer* t, uint64_t i, const uint8_t** content, uint64_t* len, int64_t* id, int* special) {
    if (i >= t->added_tokens.size()) return TKZ_ERR_INVALID_ARG;
    const AddedToken& a = t->added_tokens[i];
    *content = (const uint8_t*)a.content.data(); *len = a.content.size(); *id = a.has_id ? (int64_t)a.id : -1; *special = a.special;
    return TKZ_OK;
}
extern "C" int tkzh_model_desc(tkzh_tokenizer* t, tkz_model_desc* out) {
    if (!t || !out) return TKZ_ERR_INVALID_ARG;
    build_desc(t); *out = t->desc; return TKZ_OK;
}
