// tokenizer.cu - token ids -> text for the host side of the path (SURVEY section 8f row 4): the decode half of the reference's
// byte-level BPE tokenizer and WhisperTokenizerWrapper's word splitting, so that word timestamps and segment text work without a
// Swift host, plus text -> ids (pre-tokenizer pattern, byte alphabet, BPE merges; no post-processor: special tokens are the caller's).
// Pure host C++ (no GPU).
//   PreTrainedTokenizer.decode(tokens:skipSpecialTokens:) + cleanUp      Sources/ArgmaxCore/External/Tokenizers/Tokenizer.swift:428-447,510-530
//   ByteLevelDecoder (added tokens verbatim, the rest bytes -> UTF-8)     Sources/ArgmaxCore/External/Tokenizers/Decoder.swift:126-170
//   byteEncoder / byteDecoder (GPT-2 bytes_to_unicode)                   Sources/ArgmaxCore/External/Tokenizers/ByteEncoder.swift
//   WhisperTokenizerWrapper special tokens + defaults                    Sources/WhisperKit/Core/Models.swift:1201-1222,1309-1322
//   splitTokensOnUnicode / splitTokensOnSpaces / splitToWordTokens       Sources/WhisperKit/Core/Models.swift:1224-1306
// Two things the reference takes from Apple frameworks are restated here: CharacterSet.punctuationCharacters = Unicode general
// category P* (unicode_punct.h, generated with:  python -c "import unicodedata; ..." over category(chr(cp)).startswith('P')),
// and NLLanguageRecognizer's dominant language in {zh, ja, th, lo, my, yue} = "most letters are Han / Kana / Thai / Lao / Myanmar".
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <unordered_map>
#include <vector>

#include "kernels.h"
#include "unicode_letters.h"
#include "unicode_punct.h"

using namespace wk;

#define WK_CHECK(expr)                    \
    do {                                  \
        wk_status _s = (expr);            \
        if (_s != WK_OK) return _s;       \
    } while (0)

struct wk_tokenizer {
    std::vector<std::string> id_to_token;   // vocabulary string (byte-level alphabet) or the literal content of an added token
    std::vector<uint8_t> present, added, special;
    std::unordered_map<std::string, int> token_to_id;
    int byte_of_cp[512];                    // GPT-2 byte <-> code point bijection (code points < 0x144)
    std::string cp_of_byte[256];            // the same bijection, byte -> UTF-8 of its alphabet character
    std::unordered_map<std::string, int> merge_rank;   // "left\x01right" -> rank (text -> ids only)
    std::vector<std::string> added_sorted;  // added-token contents, longest first (matched verbatim in the text)
    bool clean_up = true;
};

namespace {

// ---- UTF-8 helpers ------------------------------------------------------------------------------------------------------
void append_utf8(std::string& s, uint32_t cp) {
    if (cp < 0x80) s.push_back((char)cp);
    else if (cp < 0x800) { s.push_back((char)(0xC0 | (cp >> 6))); s.push_back((char)(0x80 | (cp & 0x3F))); }
    else if (cp < 0x10000) { s.push_back((char)(0xE0 | (cp >> 12))); s.push_back((char)(0x80 | ((cp >> 6) & 0x3F))); s.push_back((char)(0x80 | (cp & 0x3F))); }
    else { s.push_back((char)(0xF0 | (cp >> 18))); s.push_back((char)(0x80 | ((cp >> 12) & 0x3F))); s.push_back((char)(0x80 | ((cp >> 6) & 0x3F))); s.push_back((char)(0x80 | (cp & 0x3F))); }
}

// decodes one scalar of VALID UTF-8 at s[i]; returns its length
int next_cp(const std::string& s, size_t i, uint32_t* cp) {
    const unsigned char c = (unsigned char)s[i];
    if (c < 0x80) { *cp = c; return 1; }
    if ((c >> 5) == 6 && i + 1 < s.size()) { *cp = ((c & 0x1F) << 6) | (s[i + 1] & 0x3F); return 2; }
    if ((c >> 4) == 14 && i + 2 < s.size()) { *cp = ((c & 0x0F) << 12) | ((s[i + 1] & 0x3F) << 6) | (s[i + 2] & 0x3F); return 3; }
    if ((c >> 3) == 30 && i + 3 < s.size()) { *cp = ((c & 0x07) << 18) | ((s[i + 1] & 0x3F) << 12) | ((s[i + 2] & 0x3F) << 6) | (s[i + 3] & 0x3F); return 4; }
    *cp = 0xFFFD;
    return 1;
}

// String(decoding: bytes, as: UTF8.self): every maximal invalid subpart becomes one U+FFFD (Unicode 3.9, table 3-7)
std::string utf8_lossy(const std::vector<uint8_t>& b) {
    std::string out;
    size_t i = 0;
    const size_t n = b.size();
    while (i < n) {
        const uint8_t c = b[i];
        if (c < 0x80) { out.push_back((char)c); ++i; continue; }
        int need = 0;
        uint8_t lo = 0x80, hi = 0xBF;
        if (c >= 0xC2 && c <= 0xDF) need = 1;
        else if (c == 0xE0) { need = 2; lo = 0xA0; }
        else if ((c >= 0xE1 && c <= 0xEC) || c == 0xEE || c == 0xEF) need = 2;
        else if (c == 0xED) { need = 2; hi = 0x9F; }
        else if (c == 0xF0) { need = 3; lo = 0x90; }
        else if (c >= 0xF1 && c <= 0xF3) need = 3;
        else if (c == 0xF4) { need = 3; hi = 0x8F; }
        if (need == 0) { out += "\xEF\xBF\xBD"; ++i; continue; }
        size_t j = i + 1;
        int got = 0;
        while (got < need && j < n) {
            const uint8_t d = b[j];
            const uint8_t l = got == 0 ? lo : 0x80, h = got == 0 ? hi : 0xBF;
            if (d < l || d > h) break;
            ++j; ++got;
        }
        if (got == need) out.append((const char*)&b[i], j - i);
        else out += "\xEF\xBF\xBD";
        i = j;
    }
    return out;
}

void build_byte_map(wk_tokenizer* t) {
    // GPT-2 bytes_to_unicode: printable Latin-1 bytes map to themselves, the rest to 256, 257, ... in byte order
    for (int i = 0; i < 512; ++i) t->byte_of_cp[i] = -1;
    int n = 0;
    for (int b = 0; b < 256; ++b) {
        const bool self = (b >= 0x21 && b <= 0x7E) || (b >= 0xA1 && b <= 0xAC) || (b >= 0xAE && b <= 0xFF);
        if (self) t->byte_of_cp[b] = b;
        else t->byte_of_cp[256 + n++] = b;
    }
    for (int cp = 0; cp < 512; ++cp)
        if (t->byte_of_cp[cp] >= 0) { std::string u; append_utf8(u, (uint32_t)cp); t->cp_of_byte[t->byte_of_cp[cp]] = u; }
}

bool in_ranges(const uint32_t (*r)[2], int n, uint32_t cp) {
    int lo = 0, hi = n - 1;
    while (lo <= hi) {
        const int mid = (lo + hi) / 2;
        if (cp < r[mid][0]) hi = mid - 1;
        else if (cp > r[mid][1]) lo = mid + 1;
        else return true;
    }
    return false;
}
bool is_letter(uint32_t cp) { return in_ranges(kLetterRanges, kLetterRangesCount, cp); }
bool is_number(uint32_t cp) { return in_ranges(kNumberRanges, kNumberRangesCount, cp); }
bool is_space(uint32_t cp) {   // \s of the pre-tokenizer pattern = Unicode White_Space
    return (cp >= 0x9 && cp <= 0xD) || cp == 0x20 || cp == 0x85 || cp == 0xA0 || cp == 0x1680 || (cp >= 0x2000 && cp <= 0x200A) || cp == 0x2028 ||
           cp == 0x2029 || cp == 0x202F || cp == 0x205F || cp == 0x3000;
}

// The GPT-2 / Whisper pre-tokenizer (ByteLevel use_regex; BPETokenizer.swift:165):
//   's|'t|'re|'ve|'m|'ll|'d| ?\p{L}+| ?\p{N}+| ?[^\s\p{L}\p{N}]+|\s+(?!\S)|\s+      leftmost, alternatives in order, each greedy
void pre_tokenize(const std::vector<uint32_t>& cps, std::vector<std::pair<size_t, size_t>>& pieces) {
    const size_t n = cps.size();
    size_t i = 0;
    auto other = [&](uint32_t c) { return !is_space(c) && !is_letter(c) && !is_number(c); };
    while (i < n) {
        size_t e = 0;
        if (cps[i] == '\'' && i + 1 < n) {
            const uint32_t a = cps[i + 1], b = i + 2 < n ? cps[i + 2] : 0;
            if (a == 's' || a == 't') e = i + 2;
            else if ((a == 'r' && b == 'e') || (a == 'v' && b == 'e')) e = i + 3;
            else if (a == 'm') e = i + 2;
            else if (a == 'l' && b == 'l') e = i + 3;
            else if (a == 'd') e = i + 2;
        }
        if (!e) {
            const size_t k = (cps[i] == ' ' && i + 1 < n) ? i + 1 : i;
            if (is_letter(cps[k])) { e = k; while (e < n && is_letter(cps[e])) ++e; }
            else if (is_number(cps[k])) { e = k; while (e < n && is_number(cps[e])) ++e; }
            else if (other(cps[k])) { e = k; while (e < n && other(cps[e])) ++e; }
        }
        if (!e && is_space(cps[i])) {
            size_t r = i;
            while (r < n && is_space(cps[r])) ++r;
            if (r == n) e = r;                      // \s+(?!\S) at the end of the text
            else if (r - i >= 2) e = r - 1;         // leave the last blank to the next piece (it becomes its leading space)
            else e = r;                             // \s+
        }
        if (!e) e = i + 1;
        pieces.push_back({i, e});
        i = e;
    }
}

// classic BPE: merge the lowest-rank adjacent pair (all its occurrences, left to right) until none is left
void bpe(const wk_tokenizer* t, std::vector<std::string>& word) {
    while (word.size() > 1) {
        int best = -1;
        size_t where = 0;
        for (size_t k = 0; k + 1 < word.size(); ++k) {
            auto it = t->merge_rank.find(word[k] + '\x01' + word[k + 1]);
            if (it != t->merge_rank.end() && (best < 0 || it->second < best)) { best = it->second; where = k; }
        }
        if (best < 0) break;
        const std::string a = word[where], b = word[where + 1];
        std::vector<std::string> next;
        for (size_t k = 0; k < word.size();) {
            if (k + 1 < word.size() && word[k] == a && word[k + 1] == b) { next.push_back(a + b); k += 2; }
            else { next.push_back(word[k]); ++k; }
        }
        word.swap(next);
    }
}

void finish_added(wk_tokenizer* t) {
    t->added_sorted.clear();
    for (size_t id = 0; id < t->id_to_token.size(); ++id)
        if (t->present[id] && t->added[id] && !t->id_to_token[id].empty()) t->added_sorted.push_back(t->id_to_token[id]);
    std::sort(t->added_sorted.begin(), t->added_sorted.end(), [](const std::string& a, const std::string& b) { return a.size() != b.size() ? a.size() > b.size() : a < b; });
}

void add_merge(wk_tokenizer* t, const std::string& a, const std::string& b) {
    const int rank = (int)t->merge_rank.size();
    t->merge_rank.emplace(a + '\x01' + b, rank);
}

bool is_punct(uint32_t cp) {
    int lo = 0, hi = kNumPunctRanges - 1;
    while (lo <= hi) {
        const int mid = (lo + hi) / 2;
        if (cp < kPunctRanges[mid][0]) hi = mid - 1;
        else if (cp > kPunctRanges[mid][1]) lo = mid + 1;
        else return true;
    }
    return false;
}

bool is_ws_scalar(uint32_t cp) {   // CharacterSet.whitespaces: Zs + TAB
    return cp == 0x20 || cp == 0x09 || cp == 0xA0 || cp == 0x1680 || (cp >= 0x2000 && cp <= 0x200A) || cp == 0x202F || cp == 0x205F || cp == 0x3000;
}

// stand-in for NLLanguageRecognizer.dominantLanguage in {zh, ja, th, lo, my, yue}
bool prefers_unicode_split(const std::string& text) {
    long cjk = 0, other = 0;
    for (size_t i = 0; i < text.size();) {
        uint32_t cp;
        i += next_cp(text, i, &cp);
        const bool target = (cp >= 0x4E00 && cp <= 0x9FFF) || (cp >= 0x3400 && cp <= 0x4DBF) || (cp >= 0x20000 && cp <= 0x2EBEF) ||
                            (cp >= 0x3040 && cp <= 0x30FF) || (cp >= 0x0E00 && cp <= 0x0E7F) || (cp >= 0x0E80 && cp <= 0x0EFF) || (cp >= 0x1000 && cp <= 0x109F);
        const bool letter = (cp >= 'a' && cp <= 'z') || (cp >= 'A' && cp <= 'Z') || (cp >= 0xC0 && !is_punct(cp) && !is_ws_scalar(cp) && cp != 0xFFFD);
        if (target) ++cjk; else if (letter) ++other;
    }
    return cjk > other;
}

std::string decode_ids(const wk_tokenizer* t, const int32_t* ids, int n, bool skip_special) {
    std::string out;
    std::vector<uint8_t> bytes;
    auto flush = [&]() { if (!bytes.empty()) { out += utf8_lossy(bytes); bytes.clear(); } };
    for (int i = 0; i < n; ++i) {
        const int id = ids[i];
        if (id < 0 || id >= (int)t->id_to_token.size() || !t->present[id]) continue;   // convertIdToToken nil -> compactMap drops it
        if (skip_special && t->special[id]) continue;
        const std::string& tok = t->id_to_token[id];
        if (t->added[id]) { flush(); out += tok; continue; }
        for (size_t k = 0; k < tok.size();) {
            uint32_t cp;
            k += next_cp(tok, k, &cp);
            const int b = cp < 512 ? t->byte_of_cp[cp] : -1;
            if (b >= 0) bytes.push_back((uint8_t)b);   // a code point outside the byte alphabet cannot occur in a byte-level vocabulary
        }
    }
    flush();
    if (t->clean_up) {   // PreTrainedTokenizer.cleanUp (Tokenizer.swift:434-447), in this order
        static const char* rules[][2] = {{" .", "."}, {" ?", "?"}, {" !", "!"}, {" ,", ","}, {" ' ", "'"}, {" n't", "n't"}, {" 'm", "'m"},
                                         {" 's", "'s"}, {" 've", "'ve"}, {" 're", "'re"}};
        for (auto& r : rules) {
            const std::string from = r[0], to = r[1];
            size_t pos = 0;
            while ((pos = out.find(from, pos)) != std::string::npos) { out.replace(pos, from.size(), to); pos += to.size(); }
        }
    }
    return out;
}

const char kReplacement[] = "\xEF\xBF\xBD";

void split_on_unicode(const wk_tokenizer* t, const std::vector<int32_t>& tokens, std::vector<std::string>& words, std::vector<std::vector<int32_t>>& groups) {
    const std::string full = decode_ids(t, tokens.data(), (int)tokens.size(), false);
    std::vector<int32_t> cur;
    for (int32_t tok : tokens) {
        cur.push_back(tok);
        const std::string dec = decode_ids(t, cur.data(), (int)cur.size(), false);
        const size_t at = dec.find(kReplacement);
        // Models.swift:1238-1241: the range found in `decoded` is applied to `decodedFull` as is (the running offset the reference
        // computes is never used), i.e. the same UTF-8 offsets from the start of the full text
        bool in_full = false;
        if (at != std::string::npos) in_full = at + 3 <= full.size() && full.compare(at, 3, kReplacement) == 0;
        if (at == std::string::npos || in_full) {
            words.push_back(dec);
            groups.push_back(cur);
            cur.clear();
        }
    }
}

void split_on_spaces(const wk_tokenizer* t, int special_begin, const std::vector<int32_t>& tokens, std::vector<std::string>& words,
                     std::vector<std::vector<int32_t>>& groups) {
    std::vector<std::string> sub;
    std::vector<std::vector<int32_t>> subg;
    split_on_unicode(t, tokens, sub, subg);
    for (size_t i = 0; i < sub.size(); ++i) {
        const std::string& w = sub[i];
        const bool special = subg[i][0] >= special_begin;
        const bool with_space = !w.empty() && w[0] == ' ';
        // UnicodeScalar(trimmed): only a string of exactly one scalar converts
        size_t a = 0, b = w.size();
        for (;;) { if (a >= b) break; uint32_t cp; const int k = next_cp(w, a, &cp); if (!is_ws_scalar(cp)) break; a += k; }
        for (;;) {
            if (b <= a) break;
            size_t s = b - 1;
            while (s > a && ((unsigned char)w[s] & 0xC0) == 0x80) --s;
            uint32_t cp; next_cp(w, s, &cp);
            if (!is_ws_scalar(cp)) break;
            b = s;
        }
        bool punctuation = false;
        if (b > a) {
            uint32_t cp;
            const int k = next_cp(w, a, &cp);
            if (a + k == b) punctuation = is_punct(cp);
        }
        if (special || with_space || punctuation || words.empty()) { words.push_back(w); groups.push_back(subg[i]); }
        else { words.back() += w; groups.back().insert(groups.back().end(), subg[i].begin(), subg[i].end()); }
    }
}

int lookup(const wk_tokenizer* t, const char* s, int fallback) {
    auto it = t->token_to_id.find(s);
    return it == t->token_to_id.end() ? fallback : it->second;
}

// ---- a minimal JSON reader for vocab.json / added_tokens.json / tokenizer.json ---------------------------------------------------
struct Json {
    const char* p; const char* e; bool ok = true;
    void ws() { while (p < e && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) ++p; }
    bool eat(char c) { ws(); if (p < e && *p == c) { ++p; return true; } return false; }
    char peek() { ws(); return p < e ? *p : 0; }
    static int hex4(const char* q) { int v = 0; for (int i = 0; i < 4; ++i) { const char c = q[i]; v <<= 4; if (c >= '0' && c <= '9') v |= c - '0'; else if (c >= 'a' && c <= 'f') v |= c - 'a' + 10; else if (c >= 'A' && c <= 'F') v |= c - 'A' + 10; else return -1; } return v; }
    std::string str() {
        std::string s;
        ws();
        if (p >= e || *p != '"') { ok = false; return s; }
        ++p;
        while (p < e && *p != '"') {
            if (*p != '\\') { s.push_back(*p++); continue; }
            if (++p >= e) break;
            const char c = *p++;
            switch (c) {
                case 'n': s.push_back('\n'); break; case 't': s.push_back('\t'); break; case 'r': s.push_back('\r'); break;
                case 'b': s.push_back('\b'); break; case 'f': s.push_back('\f'); break;
                case 'u': {
                    if (e - p < 4) { ok = false; return s; }
                    int v = hex4(p); p += 4;
                    if (v < 0) { ok = false; return s; }
                    if (v >= 0xD800 && v <= 0xDBFF && e - p >= 6 && p[0] == '\\' && p[1] == 'u') {
                        const int lo = hex4(p + 2);
                        if (lo >= 0xDC00 && lo <= 0xDFFF) { v = 0x10000 + ((v - 0xD800) << 10) + (lo - 0xDC00); p += 6; }
                    }
                    append_utf8(s, (uint32_t)v);
                    break;
                }
                default: s.push_back(c);   // \" \\ \/
            }
        }
        if (p < e) ++p; else ok = false;
        return s;
    }
    double num() { ws(); char* q = nullptr; const double v = strtod(p, &q); if (q == p) ok = false; p = q; return v; }
    void skip() {   // any value
        const char c = peek();
        if (c == '"') { str(); return; }
        if (c == '{' || c == '[') {
            const char close = c == '{' ? '}' : ']';
            ++p;
            if (eat(close)) return;
            do { if (c == '{') { str(); if (!eat(':')) { ok = false; return; } } skip(); } while (ok && eat(','));
            if (!eat(close)) ok = false;
            return;
        }
        while (p < e && *p != ',' && *p != '}' && *p != ']' && *p != ' ' && *p != '\n' && *p != '\r' && *p != '\t') ++p;   // number / true / false / null
    }
};

bool read_file(const std::string& path, std::string& out) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    fseek(f, 0, SEEK_END);
    const long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    out.resize((size_t)std::max(0L, n));
    const size_t got = n > 0 ? fread(&out[0], 1, (size_t)n, f) : 0;
    fclose(f);
    return got == (size_t)std::max(0L, n);
}

void put(wk_tokenizer* t, const std::string& tok, int id, bool added, bool special) {
    if (id < 0 || id > (1 << 22)) return;
    if (id >= (int)t->id_to_token.size()) { t->id_to_token.resize(id + 1); t->present.resize(id + 1, 0); t->added.resize(id + 1, 0); t->special.resize(id + 1, 0); }
    t->id_to_token[id] = tok; t->present[id] = 1; t->added[id] = added; t->special[id] = special;
    t->token_to_id[tok] = id;
}

// {"token": id, ...}
bool parse_flat_vocab(Json& j, wk_tokenizer* t, bool added) {
    if (!j.eat('{')) return false;
    if (j.eat('}')) return true;
    do {
        const std::string k = j.str();
        if (!j.ok || !j.eat(':')) return false;
        const int id = (int)j.num();
        if (!j.ok) return false;
        put(t, k, id, added, added);
    } while (j.eat(','));
    return j.eat('}');
}

// tokenizer.json: {"added_tokens":[{"id":..,"content":"..","special":true,..},..], "model":{"vocab":{..},..}, ..}
bool parse_tokenizer_json(Json& j, wk_tokenizer* t) {
    struct Added { int id = -1; std::string content; bool special = false; };
    std::vector<Added> added;
    if (!j.eat('{')) return false;
    do {
        const std::string key = j.str();
        if (!j.ok || !j.eat(':')) return false;
        if (key == "added_tokens" && j.peek() == '[') {
            j.eat('[');
            if (!j.eat(']')) {
                do {
                    Added a;
                    if (!j.eat('{')) return false;
                    do {
                        const std::string k = j.str();
                        if (!j.ok || !j.eat(':')) return false;
                        if (k == "id") a.id = (int)j.num();
                        else if (k == "content") a.content = j.str();
                        else if (k == "special") { j.ws(); a.special = j.p < j.e && *j.p == 't'; j.skip(); }
                        else j.skip();
                    } while (j.ok && j.eat(','));
                    if (!j.eat('}')) return false;
                    added.push_back(a);
                } while (j.eat(','));
                if (!j.eat(']')) return false;
            }
        } else if (key == "model" && j.peek() == '{') {
            j.eat('{');
            do {
                const std::string k = j.str();
                if (!j.ok || !j.eat(':')) return false;
                if (k == "vocab" && j.peek() == '{') { if (!parse_flat_vocab(j, t, false)) return false; }
                else if (k == "merges" && j.peek() == '[') {
                    // ["a b", ...] (older tokenizers) or [["a", "b"], ...]
                    j.eat('[');
                    if (!j.eat(']')) {
                        do {
                            if (j.peek() == '[') {
                                j.eat('[');
                                const std::string a = j.str();
                                if (!j.eat(',')) return false;
                                const std::string b = j.str();
                                if (!j.ok || !j.eat(']')) return false;
                                add_merge(t, a, b);
                            } else {
                                const std::string m = j.str();
                                const size_t sp = m.find(' ');
                                if (!j.ok || sp == std::string::npos) return false;
                                add_merge(t, m.substr(0, sp), m.substr(sp + 1));
                            }
                        } while (j.eat(','));
                        if (!j.eat(']')) return false;
                    }
                }
                else j.skip();
            } while (j.ok && j.eat(','));
            if (!j.eat('}')) return false;
        } else {
            j.skip();
        }
    } while (j.ok && j.eat(','));
    for (const Added& a : added) put(t, a.content, a.id, true, a.special);
    return j.ok;
}

}  // namespace

extern "C" {

wk_status wk_tokenizer_create(const char* const* tokens, const int32_t* ids, const uint8_t* flags, int32_t n, int32_t clean_up, wk_tokenizer** out) {
    if (!out || n < 0 || (n > 0 && (!tokens || !ids))) { set_error("wk_tokenizer_create: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    wk_tokenizer* t = new wk_tokenizer();
    build_byte_map(t);
    t->clean_up = clean_up != 0;
    for (int i = 0; i < n; ++i) put(t, tokens[i] ? tokens[i] : "", ids[i], flags && (flags[i] & 1), flags && (flags[i] & 2));
    finish_added(t);
    *out = t;
    return WK_OK;
}

wk_status wk_tokenizer_load(const char* path, wk_tokenizer** out) {
    if (!path || !out) { set_error("wk_tokenizer_load: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    wk_tokenizer* t = new wk_tokenizer();
    build_byte_map(t);
    std::string p = path, text;
    auto ends_with = [&](const char* s) { const size_t k = strlen(s); return p.size() >= k && p.compare(p.size() - k, k, s) == 0; };
    bool ok = false;
    if (ends_with(".json")) {
        if (read_file(p, text)) {
            Json j{text.data(), text.data() + text.size()};
            ok = ends_with("tokenizer.json") ? parse_tokenizer_json(j, t) : parse_flat_vocab(j, t, false);
        }
    } else if (read_file(p + "/tokenizer.json", text)) {
        Json j{text.data(), text.data() + text.size()};
        ok = parse_tokenizer_json(j, t);
    } else if (read_file(p + "/vocab.json", text)) {
        Json j{text.data(), text.data() + text.size()};
        ok = parse_flat_vocab(j, t, false);
        std::string extra;
        if (ok && read_file(p + "/added_tokens.json", extra)) {
            Json k{extra.data(), extra.data() + extra.size()};
            ok = parse_flat_vocab(k, t, true);
        }
        std::string merges;
        if (ok && read_file(p + "/merges.txt", merges)) {   // "#version" header line, then "left right" per line
            size_t pos = 0;
            while (pos < merges.size()) {
                size_t eol = merges.find('\n', pos);
                if (eol == std::string::npos) eol = merges.size();
                std::string line = merges.substr(pos, eol - pos);
                if (!line.empty() && line.back() == '\r') line.pop_back();
                const size_t sp = line.find(' ');
                if (!line.empty() && line[0] != '#' && sp != std::string::npos) add_merge(t, line.substr(0, sp), line.substr(sp + 1));
                pos = eol + 1;
            }
        }
    }
    if (!ok || t->id_to_token.empty()) { delete t; set_error("wk_tokenizer_load: no readable tokenizer.json / vocab.json at %s", path); return WK_ERR_MODELS_UNAVAILABLE; }
    finish_added(t);
    *out = t;
    return WK_OK;
}

void wk_tokenizer_free(wk_tokenizer* t) { delete t; }

int32_t wk_tokenizer_vocab_size(const wk_tokenizer* t) { return t ? (int32_t)t->id_to_token.size() : 0; }

int32_t wk_tokenizer_token_to_id(const wk_tokenizer* t, const char* token) { return (t && token) ? lookup(t, token, -1) : -1; }

int32_t wk_tokenizer_decode(const wk_tokenizer* t, const int32_t* tokens, int32_t n, int32_t skip_special_tokens, char* text, int32_t cap) {
    if (!t || n < 0 || (n > 0 && !tokens) || !text || cap < 1) return -1;
    const std::string s = decode_ids(t, tokens, n, skip_special_tokens != 0);
    if ((int64_t)s.size() + 1 > cap) return -(int32_t)(s.size() + 1);   // -(bytes needed)
    memcpy(text, s.c_str(), s.size() + 1);
    return (int32_t)s.size();
}

wk_status wk_tokenizer_set_merges(wk_tokenizer* t, const char* const* left, const char* const* right, int32_t n) {
    if (!t || n < 0 || (n > 0 && (!left || !right))) { set_error("wk_tokenizer_set_merges: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    t->merge_rank.clear();
    for (int i = 0; i < n; ++i) add_merge(t, left[i], right[i]);
    return WK_OK;
}

int32_t wk_tokenizer_encode(const wk_tokenizer* t, const char* text_utf8, int32_t* ids, int32_t cap) {
    if (!t || !text_utf8 || (cap > 0 && !ids)) return -1;
    const std::string text = text_utf8;
    std::vector<int32_t> out;
    auto encode_plain = [&](const std::string& part) -> bool {
        std::vector<uint32_t> cps;
        std::vector<size_t> off;   // byte offset of every code point, plus the end
        for (size_t i = 0; i < part.size();) { uint32_t cp; off.push_back(i); i += next_cp(part, i, &cp); cps.push_back(cp); }
        off.push_back(part.size());
        std::vector<std::pair<size_t, size_t>> pieces;
        pre_tokenize(cps, pieces);
        for (auto& pc : pieces) {
            std::vector<std::string> word;
            for (size_t b = off[pc.first]; b < off[pc.second]; ++b) word.push_back(t->cp_of_byte[(unsigned char)part[b]]);
            bpe(t, word);
            for (const std::string& w : word) {
                auto it = t->token_to_id.find(w);
                if (it == t->token_to_id.end()) return false;   // cannot happen with a byte-level vocabulary
                out.push_back(it->second);
            }
        }
        return true;
    };
    // added tokens are matched verbatim first (Tokenizer.swift:470-481), longest content first
    size_t start = 0, i = 0;
    while (i < text.size()) {
        const std::string* hit = nullptr;
        for (const std::string& a : t->added_sorted)
            if (text.compare(i, a.size(), a) == 0) { hit = &a; break; }
        if (!hit) { ++i; continue; }
        if (i > start && !encode_plain(text.substr(start, i - start))) return -1;
        out.push_back(t->token_to_id.at(*hit));
        i += hit->size();
        start = i;
    }
    if (start < text.size() && !encode_plain(text.substr(start))) return -1;
    if ((int64_t)out.size() > cap) return -(int32_t)out.size();   // -(ids needed)
    if (!out.empty()) memcpy(ids, out.data(), out.size() * 4);
    return (int32_t)out.size();
}

wk_status wk_tokenizer_special_tokens(const wk_tokenizer* t, wk_special_tokens* out) {
    if (!t || !out) { set_error("wk_tokenizer_special_tokens: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    // WhisperTokenizerWrapper.init (Models.swift:1201-1214) with the defaults of Models.swift:1309-1322
    out->end_token = lookup(t, "<|endoftext|>", 50257);
    out->english_token = lookup(t, "<|en|>", 50259);
    out->no_speech_token = lookup(t, "<|nospeech|>", 50362);
    out->no_timestamps_token = lookup(t, "<|notimestamps|>", 50363);
    out->special_token_begin = lookup(t, "<|endoftext|>", 50257);
    out->start_of_previous_token = lookup(t, "<|startofprev|>", 50361);
    out->start_of_transcript_token = lookup(t, "<|startoftranscript|>", 50258);
    out->time_token_begin = lookup(t, "<|0.00|>", 50364);
    out->transcribe_token = lookup(t, "<|transcribe|>", 50359);
    out->translate_token = lookup(t, "<|translate|>", 50358);
    out->whitespace_token = lookup(t, " ", 220);
    return WK_OK;
}

int32_t wk_tokenizer_split_to_word_tokens(const wk_tokenizer* t, const int32_t* tokens, int32_t n, char* text, int32_t text_cap, int32_t* counts, int32_t counts_cap) {
    if (!t || n < 0 || (n > 0 && !tokens) || !text || !counts) return -1;
    const int special_begin = lookup(t, "<|endoftext|>", 50257);
    std::vector<int32_t> all(tokens, tokens + n), plain;
    for (int32_t v : all) if (v < special_begin) plain.push_back(v);
    std::vector<std::string> words;
    std::vector<std::vector<int32_t>> groups;
    if (prefers_unicode_split(decode_ids(t, plain.data(), (int)plain.size(), false))) split_on_unicode(t, all, words, groups);
    else split_on_spaces(t, special_begin, all, words, groups);
    if ((int)words.size() > counts_cap) return -2;
    size_t off = 0;
    for (size_t i = 0; i < words.size(); ++i) {
        // the hook layout is NUL-terminated strings: a NUL byte decoded from the byte alphabet cannot travel and is dropped
        words[i].erase(std::remove(words[i].begin(), words[i].end(), '\0'), words[i].end());
        if (off + words[i].size() + 1 > (size_t)text_cap) return -2;
        memcpy(text + off, words[i].c_str(), words[i].size() + 1);
        off += words[i].size() + 1;
        counts[i] = (int32_t)groups[i].size();
    }
    return (int32_t)words.size();
}

int32_t wk_tokenizer_language_tokens(const wk_tokenizer* t, int32_t* out, int32_t cap) {
    if (!t || cap < 0 || (cap > 0 && !out)) return -1;
    std::vector<int32_t> ids;   // "<|xx|>" / "<|xxx|>": the language codes among the added tokens
    for (size_t id = 0; id < t->id_to_token.size(); ++id) {
        if (!t->present[id] || !t->added[id]) continue;
        const std::string& s = t->id_to_token[id];
        if (s.size() < 6 || s.size() > 7 || s.compare(0, 2, "<|") != 0 || s.compare(s.size() - 2, 2, "|>") != 0) continue;
        bool letters = true;
        for (size_t i = 2; i + 2 < s.size(); ++i) letters &= s[i] >= 'a' && s[i] <= 'z';
        if (letters) ids.push_back((int32_t)id);
    }
    if ((int64_t)ids.size() > cap) return -(int32_t)ids.size();   // -(ids needed)
    if (!ids.empty()) memcpy(out, ids.data(), ids.size() * 4);
    return (int32_t)ids.size();
}

static int32_t hook_split(void* user, const int32_t* tokens, int32_t n, char* text, int32_t text_cap, int32_t* counts, int32_t counts_cap) {
    return wk_tokenizer_split_to_word_tokens((const wk_tokenizer*)user, tokens, n, text, text_cap, counts, counts_cap);
}
static int32_t hook_decode(void* user, const int32_t* tokens, int32_t n, char* text, int32_t text_cap) {
    return wk_tokenizer_decode((const wk_tokenizer*)user, tokens, n, 0, text, text_cap);
}

wk_status wk_tokenizer_hooks_init(wk_tokenizer* t, wk_tokenizer_hooks* out) {
    if (!t || !out) { set_error("wk_tokenizer_hooks_init: bad arguments"); return WK_ERR_INVALID_ARGUMENT; }
    out->split_to_word_tokens = hook_split;
    out->decode = hook_decode;
    out->user = t;
    return WK_OK;
}

}  // extern "C"
