/*
 * stage2_stream_oracle.c -- CPU restatement of stage 2 over a stream of documents (include/simdjson_b200.h,
 * sjb200_stage2_stream): split the structurals into documents by bracket depth, run the reference's walk
 * (oracle_stage2_walk of oracle/stage2_oracle.c, included unchanged) on every document alone, and lay the tapes out as one
 * stream tape.  TEST INFRASTRUCTURE: only tests/ and tools that check the product load it.
 *
 * Per document d (tokens [doc_first[d], doc_first[d + 1])):
 *   doc_error[d]   what oracle_stage2_walk returns on idx[doc_first[d] ..] + the trailer len, len, 0 (0 = SUCCESS)
 *   doc_tape[d]    where its slice starts: slice length = 2 + words of its tokens (strings, brackets, t f n: 1; numbers: 2;
 *                  ':' ',' and anything else: 0), whatever the verdict
 *   the slice      the walk's tape (relative to the slice, as the walk writes it) with every string word rebased onto the
 *                  stream's one string buffer: the records of all strings in index order, a failing string a record of
 *                  length 0 (the layout of oracle_stage2_primitives).  Meaningful only for successful documents.
 */
#include "../oracle/stage2_oracle.c"

static uint32_t token_words(const uint8_t *buf, uint64_t len, uint32_t i) {
    const uint8_t c = at(buf, len, i);
    if (c == '-' || (c >= '0' && c <= '9')) return 2;
    if (c == '"' || c == '{' || c == '}' || c == '[' || c == ']' || c == 't' || c == 'f' || c == 'n') return 1;
    return 0;
}

/* doc_first / doc_tape: n + 1 entries, doc_error: n.  Returns the number of documents, or -1 if a buffer ran out. */
EXPORT int64_t oracle_stage2_walk_stream(const uint8_t *buf, uint64_t len, const uint32_t *idx, uint64_t n, uint64_t *tape, uint64_t tape_cap,
                                         uint32_t *doc_first, uint64_t *doc_tape, int32_t *doc_error) {
    uint64_t nd = 0;
    int64_t depth = 0;
    for (uint64_t k = 0; k < n; k++) {
        const uint8_t c = at(buf, len, idx[k]);
        if (depth == 0) doc_first[nd++] = (uint32_t)k;
        if (c == '{' || c == '[') depth++;
        if (c == '}' || c == ']') depth--;
    }
    doc_first[nd] = (uint32_t)n;
    doc_tape[0] = 0;
    for (uint64_t d = 0; d < nd; d++) {
        uint64_t w = 2;
        for (uint64_t k = doc_first[d]; k < doc_first[d + 1]; k++) w += token_words(buf, len, idx[k]);
        doc_tape[d + 1] = doc_tape[d] + w;
    }
    if (doc_tape[nd] > tape_cap) return -1;
    uint32_t *sub = (uint32_t *)malloc((size_t)(n + 3) * 4);
    if (!sub) return -1;
    uint64_t str_base = 0;   /* bytes of string records before the current document */
    for (uint64_t d = 0; d < nd; d++) {
        const uint64_t f = doc_first[d], m = doc_first[d + 1] - f;
        memcpy(sub, idx + f, (size_t)m * 4);
        sub[m] = (uint32_t)len;
        sub[m + 1] = (uint32_t)len;
        sub[m + 2] = 0;
        uint64_t *slice = tape + doc_tape[d];
        const uint64_t slice_len = doc_tape[d + 1] - doc_tape[d];
        uint64_t tl = 0, sl = 0;
        doc_error[d] = oracle_stage2_walk(buf, len, sub, m, slice, slice_len, &tl, 0, &sl);
        if (doc_error[d] == SUCCESS) {
            for (uint64_t j = 1; j + 1 < slice_len; j++) {   /* the payload word of a number is skipped, whatever its top byte */
                const uint8_t ty = (uint8_t)(slice[j] >> 56);
                if (ty == '"') slice[j] += str_base;
                if (ty == 'l' || ty == 'd') j++;
            }
        }
        for (uint64_t k = f; k < f + m; k++) {
            const uint32_t i = idx[k];
            if (at(buf, len, i) != '"') continue;
            const int64_t l = oracle_parse_string(buf, len, (uint64_t)i + 1, 0, 8, 0);
            str_base += 4 + (uint64_t)(l < 0 ? 0 : l);
        }
    }
    free(sub);
    return (int64_t)nd;
}
