/*
 * stage2_oracle.c -- CPU restatement of the per-primitive half of mojo-simdjson's stage 2 (SURVEY.md section 8(f) rank 3):
 * string unescaping, true / false / null atoms, number syntax.  Plain C, sequential, one primitive at a time.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/ (and tools that check the product) load this library; nothing under
 * mojo_simdjson_b200/ imports, links or executes it.
 *
 * What it follows (paths relative to /root/reference/src/mojo_simdjson/):
 *   parse_string / handle_unicode_codepoint   generic/stage2/string_parsing.mojo:263-386 (escape_map :7-260)
 *   BackslashAndQuote.copy_and_find           include/haswell/stringparsing_defs.mojo:9-48
 *   hex_to_u32_nocheck / codepoint_to_utf8     include/generic/jsoncharutils.mojo:33-81, internal/jsoncharutils_tables.mojo
 *   is_valid_{true,false,null}_atom            include/generic/atom_parsing.mojo:34-80
 *   parse_number                               include/generic/number_parsing.mojo:22-80
 *   the dispatch on the first byte             generic/stage2/json_iterator.mojo:306-329 (visit_primitive)
 *   error codes                                errors.mojo:2-34
 *
 * PARITY STATUS: UNPINNED except for what the reference's own stage-2 tests hold, which is only "stage2() returns SUCCESS"
 * on four fixtures (tests/test_stage_2.mojo:27-63: simple_json, simple_strings, escaping, escaping_very_long); the
 * reference has no golden tape, no golden string buffer and no error-path test for stage 2.  tests/test_stage2_oracle.py
 * checks that every primitive of those four fixtures comes out SUCCESS here, in both string-scanner modes below.
 *
 * Two places where the reference cannot be restated as written, and what this file does instead:
 *  (1) copy_and_find loads 8 bytes (stringparsing_defs.mojo:40) but parse_string advances by BYTES_PROCESSED = 32 when the
 *      window holds neither a quote nor a backslash (string_parsing.mojo:384-385, stringparsing_defs.mojo:10): 24 of every
 *      32 bytes are neither copied nor examined, so a string whose closing quote falls into such a gap is read past its
 *      end (and past the buffer).  `advance` selects the behaviour: 32 = as written, 8 = as intended (upstream simdjson's
 *      loop, every byte examined).  The two agree on every string whose first 8-byte window already contains its first
 *      quote or backslash and so on after every escape -- all strings of the reference's fixtures -- and the product
 *      implements advance = 8.
 *  (2) parse_number hands the token to the Mojo standard library (Int(StringSlice), Float64(StringSlice);
 *      max 25.1.0.dev2025013105, source not vendored).  Restated here: the token syntax the reference's own code decides
 *      (sign, digit run, float iff the run is followed by '.', 'e' or 'E', integer tokens must end at a structural or
 *      whitespace byte, float tokens extend to the next such byte), integer value = the decimal digits accumulated in
 *      64-bit two's complement (no digits: NUMBER_ERROR), float tokens accepted iff they match
 *      -?digits*(.digits*)?([eE][+-]?digits+)? with at least one mantissa digit.  The float VALUE is not restated
 *      (tape_writer.mojo:18-20 stores value.cast[uint64], a numeric cast the reference itself marks "TODO: Is this type cast
 *      correct?").
 */
#include <stdint.h>
#include <string.h>

#define EXPORT __attribute__((visibility("default")))

enum { SUCCESS = 0, TAPE_ERROR = 3, STRING_ERROR = 5, T_ATOM_ERROR = 6, F_ATOM_ERROR = 7, N_ATOM_ERROR = 8, NUMBER_ERROR = 9 };

/* primitive kinds reported per structural */
enum { KIND_NONE = 0, KIND_STRING = 1, KIND_INT = 2, KIND_FLOAT = 3, KIND_TRUE = 4, KIND_FALSE = 5, KIND_NULL = 6, KIND_BAD = 7 };

/* bytes at or beyond the end of the document read as 0x20: stage 1's own tail padding (json_structural_indexer.mojo:103) and
 * what visit_root_number pads its copy with (tape_builder.mojo:139-158) */
static inline uint8_t at(const uint8_t *buf, uint64_t len, uint64_t i) { return i < len ? buf[i] : 0x20; }

/* internal/jsoncharutils_tables.mojo:5-16: 09 0A 0D 20 , : [ ] { } */
static inline int structural_or_whitespace(uint8_t c) {
    return c == 0x09 || c == 0x0A || c == 0x0D || c == 0x20 || c == ',' || c == ':' || c == '[' || c == ']' || c == '{' || c == '}';
}

static inline uint8_t escape_map(uint8_t c) { /* string_parsing.mojo:7-260 */
    switch (c) {
    case '"': return 0x22;
    case '/': return 0x2F;
    case '\\': return 0x5C;
    case 'b': return 0x08;
    case 'f': return 0x0C;
    case 'n': return 0x0A;
    case 'r': return 0x0D;
    case 't': return 0x09;
    default: return 0;
    }
}

/* jsoncharutils.mojo:33-45: 0xFFFFFFFF-ish (high bits set) if any of the four bytes is not a hex digit */
static inline uint32_t hex_digit(uint8_t c) {
    if (c >= '0' && c <= '9') return (uint32_t)(c - '0');
    if (c >= 'a' && c <= 'f') return (uint32_t)(c - 'a' + 10);
    if (c >= 'A' && c <= 'F') return (uint32_t)(c - 'A' + 10);
    return 0xFFFFFFFFu;
}
static inline uint32_t hex_to_u32_nocheck(const uint8_t *buf, uint64_t len, uint64_t i) {
    const uint32_t a = hex_digit(at(buf, len, i)), b = hex_digit(at(buf, len, i + 1)), c = hex_digit(at(buf, len, i + 2)),
                   d = hex_digit(at(buf, len, i + 3));
    if ((a | b | c | d) & 0xFFFF0000u) return 0xFFFFFFFFu;
    return (a << 12) | (b << 8) | (c << 4) | d;
}

/* jsoncharutils.mojo:48-81 */
static inline int codepoint_to_utf8(uint32_t cp, uint8_t *c) {
    if (cp <= 0x7F) {
        if (c) c[0] = (uint8_t)cp;
        return 1;
    }
    if (cp <= 0x7FF) {
        if (c) {
            c[0] = (uint8_t)((cp >> 6) + 192);
            c[1] = (uint8_t)((cp & 63) + 128);
        }
        return 2;
    }
    if (cp <= 0xFFFF) {
        if (c) {
            c[0] = (uint8_t)((cp >> 12) + 224);
            c[1] = (uint8_t)(((cp >> 6) & 63) + 128);
            c[2] = (uint8_t)((cp & 63) + 128);
        }
        return 3;
    }
    if (cp <= 0x10FFFF) {
        if (c) {
            c[0] = (uint8_t)((cp >> 18) + 240);
            c[1] = (uint8_t)(((cp >> 12) & 63) + 128);
            c[2] = (uint8_t)(((cp >> 6) & 63) + 128);
            c[3] = (uint8_t)((cp & 63) + 128);
        }
        return 4;
    }
    return 0;
}

/*
 * parse_string (string_parsing.mojo:334-386), src = index of the byte after the opening quote.  dst may be NULL (length only).
 * Returns the unescaped length, or -1 (STRING_ERROR).  *src_end (if not NULL) = index of the closing quote.
 * advance: 8 = every byte examined (intended / upstream), 32 = BYTES_PROCESSED as written (see the header; bytes the
 * reference neither copies nor examines are left as they are in dst, i.e. whatever the caller put there -- the reference's
 * resize(.., 0) zero fill, dom_parser_implementation.mojo:77-79).
 * limit: scanning stops with an error once src passes len + 64 (the reference would read on; only advance = 32 can get there).
 */
EXPORT int64_t oracle_parse_string(const uint8_t *buf, uint64_t len, uint64_t src, uint8_t *dst, uint32_t advance, uint64_t *src_end) {
    uint64_t d = 0;
    for (;;) {
        if (src > len + 64) return -1;
        /* copy_and_find: 8 bytes copied unconditionally, quote / backslash bits of those 8 bytes */
        uint32_t bs_bits = 0, quote_bits = 0;
        for (int k = 0; k < 8; k++) {
            const uint8_t c = at(buf, len, src + k);
            if (dst) dst[d + k] = c;
            if (c == '\\') bs_bits |= 1u << k;
            if (c == '"') quote_bits |= 1u << k;
        }
        if (((bs_bits - 1u) & quote_bits) != 0) { /* has_quote_first */
            const int q = __builtin_ctz(quote_bits);
            if (src_end) *src_end = src + q;
            return (int64_t)(d + q);
        }
        if (((quote_bits - 1u) & bs_bits) != 0) { /* has_backslash */
            const int bd = __builtin_ctz(bs_bits);
            const uint8_t esc = at(buf, len, src + bd + 1);
            if (esc == 'u') {
                src += bd;
                d += bd;
                /* handle_unicode_codepoint, allow_replacement = False */
                uint32_t cp = hex_to_u32_nocheck(buf, len, src + 2);
                src += 6;
                if (cp >= 0xD800 && cp < 0xDC00) {
                    if (!(at(buf, len, src) == '\\' && at(buf, len, src + 1) == 'u')) return -1;
                    const uint32_t cp2 = hex_to_u32_nocheck(buf, len, src + 2);
                    const uint32_t low = cp2 - 0xDC00u;
                    if (low >> 10) return -1;
                    cp = (((cp - 0xD800u) << 10) | low) + 0x10000u;
                    src += 6;
                } else if (cp >= 0xDC00 && cp <= 0xDFFF) {
                    return -1;
                }
                const int n = codepoint_to_utf8(cp, dst ? dst + d : 0);
                if (n == 0) return -1;
                d += (uint64_t)n;
            } else {
                const uint8_t r = escape_map(esc);
                if (r == 0) return -1;
                if (dst) dst[d + bd] = r;
                src += (uint64_t)bd + 2;
                d += (uint64_t)bd + 1;
            }
        } else {
            src += advance;
            d += advance;
        }
    }
}

/* atom_parsing.mojo:34-80 (the non-root forms: the byte after the atom must be structural or whitespace) */
static inline int atom_is(const uint8_t *buf, uint64_t len, uint64_t i, const char *four) {
    return at(buf, len, i) == (uint8_t)four[0] && at(buf, len, i + 1) == (uint8_t)four[1] && at(buf, len, i + 2) == (uint8_t)four[2] &&
           at(buf, len, i + 3) == (uint8_t)four[3];
}
EXPORT int32_t oracle_is_valid_true_atom(const uint8_t *buf, uint64_t len, uint64_t i) {
    return atom_is(buf, len, i, "true") && structural_or_whitespace(at(buf, len, i + 4));
}
EXPORT int32_t oracle_is_valid_false_atom(const uint8_t *buf, uint64_t len, uint64_t i) {
    return atom_is(buf, len, i + 1, "alse") && structural_or_whitespace(at(buf, len, i + 5));
}
EXPORT int32_t oracle_is_valid_null_atom(const uint8_t *buf, uint64_t len, uint64_t i) {
    return atom_is(buf, len, i, "null") && structural_or_whitespace(at(buf, len, i + 4));
}

/* number_parsing.mojo:22-80.  Returns SUCCESS or NUMBER_ERROR; *is_float, *ivalue (integers), *token_len. */
EXPORT int32_t oracle_parse_number(const uint8_t *buf, uint64_t len, uint64_t i, int32_t *is_float, int64_t *ivalue, uint32_t *token_len) {
    const int neg = at(buf, len, i) == '-';
    uint64_t p = i + (uint64_t)neg;
    uint64_t acc = 0;
    uint64_t digits = 0;
    while (at(buf, len, p) >= '0' && at(buf, len, p) <= '9') {
        acc = acc * 10u + (uint64_t)(at(buf, len, p) - '0');
        digits++;
        p++;
    }
    const uint8_t c = at(buf, len, p);
    *is_float = 0;
    *ivalue = 0;
    if (c == '.' || c == 'e' || c == 'E') {
        *is_float = 1;
        while (!structural_or_whitespace(at(buf, len, p))) p++;
        *token_len = (uint32_t)(p - i);
        /* the token as the standard library's float parser accepts it: -?digits*(.digits*)?([eE][+-]?digits+)?, >= 1 mantissa digit */
        uint64_t q = i + (uint64_t)neg + digits;
        uint64_t mant = digits;
        if (at(buf, len, q) == '.') {
            q++;
            while (at(buf, len, q) >= '0' && at(buf, len, q) <= '9') {
                q++;
                mant++;
            }
        }
        if (mant == 0) return NUMBER_ERROR;
        if (at(buf, len, q) == 'e' || at(buf, len, q) == 'E') {
            q++;
            if (at(buf, len, q) == '+' || at(buf, len, q) == '-') q++;
            uint64_t ed = 0;
            while (at(buf, len, q) >= '0' && at(buf, len, q) <= '9') {
                q++;
                ed++;
            }
            if (ed == 0) return NUMBER_ERROR;
        }
        return q == p ? SUCCESS : NUMBER_ERROR;
    }
    *token_len = (uint32_t)(p - i);
    if (!structural_or_whitespace(c)) return NUMBER_ERROR;
    if (digits == 0) return NUMBER_ERROR; /* Int("") / Int("-") raise */
    *ivalue = (int64_t)(neg ? (uint64_t)0 - acc : acc);
    return SUCCESS;
}

/*
 * Every structural index of a document, in order, as visit_primitive (json_iterator.mojo:306-329) would treat the byte it
 * points at; the structural characters themselves ({ } [ ] : ,) are KIND_NONE.  Outputs, one entry per structural:
 *   kind[k], err[k] (simdjson error code of that primitive, 0 = fine),
 *   value[k]: strings -> unescaped length, integers -> the value, floats -> token length, else 0
 *   str_off[k]: strings -> offset of its record in strbuf, else 0
 * strbuf (may be NULL) receives, for every string in index order, the reference's record: uint32 length, then the bytes
 * (tape_builder.mojo:268-301: no terminator); a string that fails contributes a record of length 0.  *strbuf_len = total.
 * *first_err_index / *first_err: the first primitive (in index order) whose error is non-zero (n / 0 if none).
 */
EXPORT int32_t oracle_stage2_primitives(const uint8_t *buf, uint64_t len, const uint32_t *idx, uint64_t n, uint8_t *kind, uint8_t *err,
                                        int64_t *value, uint64_t *str_off, uint8_t *strbuf, uint64_t *strbuf_len, uint64_t *first_err_index,
                                        int32_t *first_err) {
    uint64_t off = 0;
    *first_err_index = n;
    *first_err = SUCCESS;
    for (uint64_t k = 0; k < n; k++) {
        const uint64_t i = idx[k];
        const uint8_t c = at(buf, len, i);
        uint8_t kd = KIND_NONE, e = SUCCESS;
        int64_t v = 0;
        uint64_t so = 0;
        if (c == '"') {
            kd = KIND_STRING;
            so = off;
            int64_t l = oracle_parse_string(buf, len, i + 1, strbuf ? strbuf + off + 4 : 0, 8, 0);
            if (l < 0) {
                e = STRING_ERROR;
                l = 0;
            }
            if (strbuf) {
                const uint32_t l32 = (uint32_t)l;
                memcpy(strbuf + off, &l32, 4);
            }
            v = l;
            off += 4 + (uint64_t)l;
        } else if (c == '-' || (c >= '0' && c <= '9')) {
            int32_t isf;
            uint32_t tl;
            e = (uint8_t)oracle_parse_number(buf, len, i, &isf, &v, &tl);
            kd = isf ? KIND_FLOAT : KIND_INT;
            if (isf) v = tl;
        } else if (c == 't') {
            kd = KIND_TRUE;
            e = oracle_is_valid_true_atom(buf, len, i) ? SUCCESS : T_ATOM_ERROR;
        } else if (c == 'f') {
            kd = KIND_FALSE;
            e = oracle_is_valid_false_atom(buf, len, i) ? SUCCESS : F_ATOM_ERROR;
        } else if (c == 'n') {
            kd = KIND_NULL;
            e = oracle_is_valid_null_atom(buf, len, i) ? SUCCESS : N_ATOM_ERROR;
        } else if (c == '{' || c == '}' || c == '[' || c == ']' || c == ':' || c == ',') {
            kd = KIND_NONE;
        } else {
            kd = KIND_BAD;
            e = TAPE_ERROR;
        }
        kind[k] = kd;
        err[k] = e;
        value[k] = v;
        str_off[k] = so;
        if (e != SUCCESS && *first_err_index == n) {
            *first_err_index = k;
            *first_err = e;
        }
    }
    *strbuf_len = off;
    return SUCCESS;
}

EXPORT int32_t oracle_stage2_version(void) { return 1; }

/* ------------------------------------------------------------------------------------------------------------------
 * The walk (SURVEY.md section 8(f) rank 4): JsonIterator.walk_document, generic/stage2/json_iterator.mojo:40-254, restated
 * state for state -- the order of every check and therefore the error code it returns are the reference's.  What the walk
 * APPENDS is the tape.  The reference's TapeBuilder is unfinished in three places, so the tape written here is the format
 * its comments describe (upstream simdjson's), not what its code would leave in memory:
 *   - end_container (tape_builder.mojo:227-254) announces "Write the ending tape element" but never appends one;
 *   - next_tape_index (:206-208) is a difference of addresses, i.e. a BYTE offset, which start_container / end_container /
 *     visit_document_end then use as an ELEMENT index (:216-225, :243-251, :100-108): every container start lands 8x too far;
 *   - append_double (tape_writer.mojo:18-20) stores value.cast[uint64], a numeric conversion ("TODO: Is this type cast correct?").
 * Tape words (64 bit, type character in the top byte, tape_type.mojo:1-13), element indexes:
 *   tape[0] = 'r' | N            N = number of tape words (the final root included)
 *   '{' / '[' | count << 32 | index of the word after the matching '}' / ']'     (count saturates at 0xFFFFFF upstream; the
 *                                 reference returns CAPACITY above it, tape_builder.mojo:239-241, restated here)
 *   '}' / ']' | index of the matching start
 *   '"' | offset of the string's record in the string buffer
 *   'l' | 0 followed by the int64 value; 'd' | 0 followed by the IEEE-754 bits (parity UNPINNED for doubles, see (2) above:
 *                                 produced with strtod here, correctly rounded; the tests compare the kernel's
 *                                 payloads with a restatement of its conversion, which is exact only on Clinger's fast path)
 *   't' 'f' 'n' | 0
 *   tape[N-1] = 'r' | 0
 * PARITY: error codes pinned by code reading; the reference's tests only assert SUCCESS on four fixtures.  Tape UNPINNED.
 * ------------------------------------------------------------------------------------------------------------------ */
#include <stdlib.h>

enum { DEPTH_ERROR = 4, CAPACITY_ERROR = 1, EMPTY_ERROR = 13 };
#define MAX_DEPTH 100 /* dom_parser_implementation.mojo:40: _max_depth = 100 */

typedef struct {
    const uint8_t *buf;
    uint64_t len;
    const uint32_t *idx;
    uint64_t n, next; /* next structural */
    uint64_t *tape;
    uint64_t tape_cap, tape_len;
    uint8_t *strbuf;
    uint64_t str_len;
} Walk;

static inline void tape_append(Walk *w, uint64_t value, uint8_t type) {
    if (w->tape && w->tape_len < w->tape_cap) w->tape[w->tape_len] = value | ((uint64_t)type << 56);
    w->tape_len++;
}
static inline void tape_write(Walk *w, uint64_t at_index, uint64_t value, uint8_t type) {
    if (w->tape && at_index < w->tape_cap) w->tape[at_index] = value | ((uint64_t)type << 56);
}

static int32_t walk_primitive(Walk *w, uint64_t i, int root) {
    const uint8_t c = at(w->buf, w->len, i);
    (void)root; /* the root forms differ only in how they guard reads past the end; bytes past the end read as 0x20 here */
    if (c == '"') {
        const uint64_t off = w->str_len;
        int64_t l = oracle_parse_string(w->buf, w->len, i + 1, w->strbuf ? w->strbuf + off + 4 : 0, 8, 0);
        if (l < 0) return STRING_ERROR;
        tape_append(w, off, '"');
        if (w->strbuf) {
            const uint32_t l32 = (uint32_t)l;
            memcpy(w->strbuf + off, &l32, 4);
        }
        w->str_len += 4 + (uint64_t)l;
        return SUCCESS;
    }
    if (c == '-' || (c >= '0' && c <= '9')) { /* visit_primitive tests numbers before atoms (json_iterator.mojo:312-315) */
        int32_t isf;
        int64_t v;
        uint32_t tl;
        const int32_t e = oracle_parse_number(w->buf, w->len, i, &isf, &v, &tl);
        if (e != SUCCESS) return e;
        if (isf) {
            /* a float token can be arbitrarily long (digits and exponent have no length limit): copy it whole */
            char *tmp = (char *)malloc((size_t)tl + 1);
            if (!tmp) return CAPACITY_ERROR;
            for (uint32_t k = 0; k < tl; k++) tmp[k] = (char)at(w->buf, w->len, i + k);
            tmp[tl] = 0;
            const double d = strtod(tmp, 0);
            free(tmp);
            uint64_t bits;
            memcpy(&bits, &d, 8);
            tape_append(w, 0, 'd');
            tape_append(w, bits, 0);
        } else {
            tape_append(w, 0, 'l');
            tape_append(w, (uint64_t)v, 0);
        }
        return SUCCESS;
    }
    if (c == 't') {
        if (!oracle_is_valid_true_atom(w->buf, w->len, i)) return T_ATOM_ERROR;
        tape_append(w, 0, 't');
        return SUCCESS;
    }
    if (c == 'f') {
        if (!oracle_is_valid_false_atom(w->buf, w->len, i)) return F_ATOM_ERROR;
        tape_append(w, 0, 'f');
        return SUCCESS;
    }
    if (c == 'n') {
        if (!oracle_is_valid_null_atom(w->buf, w->len, i)) return N_ATOM_ERROR;
        tape_append(w, 0, 'n');
        return SUCCESS;
    }
    return TAPE_ERROR;
}

EXPORT int32_t oracle_stage2_walk(const uint8_t *buf, uint64_t len, const uint32_t *idx, uint64_t n, uint64_t *tape, uint64_t tape_cap,
                                  uint64_t *tape_len, uint8_t *strbuf, uint64_t *strbuf_len) {
    Walk w = {buf, len, idx, n, 0, tape, tape_cap, 0, strbuf, 0};
    uint32_t start_index[MAX_DEPTH + 2], count[MAX_DEPTH + 2];
    uint8_t is_array[MAX_DEPTH + 2];
    uint32_t depth = 0;
    int32_t e;
#define PEEK() at(buf, len, idx[w.next])   /* idx[n] = len: the trailer reads as padding */
#define ADVANCE() (w.next < n + 2 ? idx[w.next++] : (uint32_t)len)
#define FAIL(code)                 \
    do {                           \
        *tape_len = w.tape_len;    \
        *strbuf_len = w.str_len;   \
        return (code);             \
    } while (0)
    enum { DOC_START, OBJECT_BEGIN, OBJECT_FIELD, OBJECT_CONTINUE, SCOPE_END, ARRAY_BEGIN, ARRAY_VALUE, ARRAY_CONTINUE, DOC_END } state = DOC_START;
    for (;;) {
        switch (state) {
        case DOC_START: {
            if (w.next == n) FAIL(EMPTY_ERROR);                   /* at_eof (:45-46) */
            start_index[0] = (uint32_t)w.tape_len;               /* visit_document_start: start_container at depth 0 */
            count[0] = 0;
            w.tape_len++;                                         /* skip: the root word is written at the end */
            const uint32_t vi = ADVANCE();
            const uint8_t v = at(buf, len, vi);
            const uint8_t last = at(buf, len, idx[n - 1]);       /* last_structural (:283-291) */
            if (v == '{' && last != '}') FAIL(TAPE_ERROR);
            if (v == '[' && last != ']') FAIL(TAPE_ERROR);
            if (v == '{') {
                if (PEEK() == '}') {
                    /* (the reference does not advance past the '}' here, :61-65; the final index check then fails) */
                    const uint64_t s = w.tape_len;
                    tape_append(&w, s + 2, '{');
                    tape_append(&w, s, '}');
                } else {
                    state = OBJECT_BEGIN;
                    continue;
                }
            } else if (v == '[') {
                if (PEEK() == ']') {
                    const uint64_t s = w.tape_len;
                    tape_append(&w, s + 2, '[');
                    tape_append(&w, s, ']');
                } else {
                    state = ARRAY_BEGIN;
                    continue;
                }
            } else {
                e = walk_primitive(&w, vi, 1);
                if (e != SUCCESS) FAIL(e);
            }
            state = DOC_END;
            continue;
        }
        case OBJECT_BEGIN: {
            depth++;
            if (depth > MAX_DEPTH) FAIL(DEPTH_ERROR);             /* :86-88: objects may reach depth == max_depth */
            is_array[depth] = 0;
            start_index[depth] = (uint32_t)w.tape_len;           /* visit_object_start */
            count[depth] = 0;
            w.tape_len++;
            const uint32_t ki = ADVANCE();
            if (at(buf, len, ki) != '"') FAIL(TAPE_ERROR);
            count[depth]++;
            e = walk_primitive(&w, ki, 0);                        /* visit_key = visit_string */
            if (e != SUCCESS) FAIL(e);
            state = OBJECT_FIELD;
            continue;
        }
        case OBJECT_FIELD: {
            if (at(buf, len, ADVANCE()) != ':') FAIL(TAPE_ERROR);
            const uint32_t vi = ADVANCE();
            const uint8_t v = at(buf, len, vi);
            if (v == '{') {
                if (PEEK() == '}') {
                    (void)ADVANCE();
                    const uint64_t s = w.tape_len;
                    tape_append(&w, s + 2, '{');
                    tape_append(&w, s, '}');
                } else {
                    state = OBJECT_BEGIN;
                    continue;
                }
            } else if (v == '[') {
                if (PEEK() == ']') {
                    (void)ADVANCE();
                    const uint64_t s = w.tape_len;
                    tape_append(&w, s + 2, '[');
                    tape_append(&w, s, ']');
                } else {
                    state = ARRAY_BEGIN;
                    continue;
                }
            } else {
                e = walk_primitive(&w, vi, 0);
                if (e != SUCCESS) FAIL(e);
            }
            state = OBJECT_CONTINUE;
            continue;
        }
        case OBJECT_CONTINUE: {
            const uint8_t c = at(buf, len, ADVANCE());
            if (c == ',') {
                count[depth]++;
                const uint32_t ki = ADVANCE();
                if (at(buf, len, ki) != '"') FAIL(TAPE_ERROR);
                e = walk_primitive(&w, ki, 0);
                if (e != SUCCESS) FAIL(e);
                state = OBJECT_FIELD;
                continue;
            } else if (c == '}') {
                if (count[depth] > 0xFFFFFF) FAIL(CAPACITY_ERROR);
                tape_append(&w, start_index[depth], '}');
                tape_write(&w, start_index[depth], w.tape_len | ((uint64_t)count[depth] << 32), '{');
                state = SCOPE_END;
                continue;
            }
            FAIL(TAPE_ERROR);
        }
        case SCOPE_END: {
            depth--;
            if (depth == 0) {
                state = DOC_END;
                continue;
            }
            state = is_array[depth] ? ARRAY_CONTINUE : OBJECT_CONTINUE;
            continue;
        }
        case ARRAY_BEGIN: {
            depth++;
            if (depth >= MAX_DEPTH) FAIL(DEPTH_ERROR);            /* :177-180: arrays fail one level earlier than objects */
            is_array[depth] = 1;
            start_index[depth] = (uint32_t)w.tape_len;
            count[depth] = 0;
            w.tape_len++;
            count[depth]++;
            state = ARRAY_VALUE;
            continue;
        }
        case ARRAY_VALUE: {
            const uint32_t vi = ADVANCE();
            const uint8_t v = at(buf, len, vi);
            if (v == '{') {
                if (PEEK() == '}') {
                    (void)ADVANCE();
                    const uint64_t s = w.tape_len;
                    tape_append(&w, s + 2, '{');
                    tape_append(&w, s, '}');
                } else {
                    state = OBJECT_BEGIN;
                    continue;
                }
            } else if (v == '[') {
                if (PEEK() == ']') {
                    (void)ADVANCE();
                    const uint64_t s = w.tape_len;
                    tape_append(&w, s + 2, '[');
                    tape_append(&w, s, ']');
                } else {
                    state = ARRAY_BEGIN;
                    continue;
                }
            } else {
                e = walk_primitive(&w, vi, 0);
                if (e != SUCCESS) FAIL(e);
            }
            state = ARRAY_CONTINUE;
            continue;
        }
        case ARRAY_CONTINUE: {
            const uint8_t c = at(buf, len, ADVANCE());
            if (c == ',') {
                count[depth]++;
                state = ARRAY_VALUE;
                continue;
            } else if (c == ']') {
                if (count[depth] > 0xFFFFFF) FAIL(CAPACITY_ERROR);
                tape_append(&w, start_index[depth], ']');
                tape_write(&w, start_index[depth], w.tape_len | ((uint64_t)count[depth] << 32), '[');
                state = SCOPE_END;
                continue;
            }
            FAIL(TAPE_ERROR);
        }
        case DOC_END: {
            tape_append(&w, 0, 'r');                              /* visit_document_end (:96-108) */
            tape_write(&w, 0, w.tape_len, 'r');
            *tape_len = w.tape_len;
            *strbuf_len = w.str_len;
            if (w.next != n) return TAPE_ERROR;                   /* more than one value at the root / trailing content (:236-246) */
            return SUCCESS;
        }
        }
    }
#undef PEEK
#undef ADVANCE
#undef FAIL
}
