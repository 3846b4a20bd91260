/*
 * oracle_cs.c -- CPU restatement of minimap2's cs:Z: difference string (--cs, --cs=long) for the oracle's alignments: the
 * reference the GPU's AW_FLAG_CS / AW_FLAG_CS_LONG output is held to.  TEST INFRASTRUCTURE ONLY, built by tests/oracle_cs.py
 * against oracle/liballwave_oracle.so (whose alignments, reverse complement and PAF writer it uses).
 *
 * The tag describes the target against the oriented query, left to right along the CIGAR (WFA2 letters, one per column):
 * a run of M -> ":N" (short) or "=" + the target bases upper-cased (long); every X column -> "*" + target base + query base;
 * a run of D (query bases only, PAF 'I') -> "+" + the query bases; a run of I (target bases only, PAF 'D') -> "-" + the
 * target bases.  "*", "+" and "-" bases are lower-cased; only A-Z change case.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../oracle/aw_oracle.h"

static char lower_c(uint8_t b) { return (char)((b >= 'A' && b <= 'Z') ? b + 32 : b); }
static char upper_c(uint8_t b) { return (char)((b >= 'a' && b <= 'z') ? b - 32 : b); }

/* the tag of the alignment ops[0 .. n) of the oriented query against the target; malloc'ed, NUL-terminated; NULL when the
 * ops do not consume exactly both sequences.  A tag is at most 2 * (qlen + tlen) bytes. */
char* awo_cs_string(const uint8_t* ops, size_t n, const uint8_t* query, size_t qlen, const uint8_t* target, size_t tlen, int long_form) {
    char* s = (char*)malloc(2 * (qlen + tlen) + 24);
    size_t len = 0, q = 0, t = 0, i = 0;
    while (i < n) {
        const uint8_t op = ops[i];
        size_t j = i + 1;
        if (op != 'X')
            while (j < n && ops[j] == op) ++j;
        const size_t run = j - i;
        const size_t dq = (op == 'M' || op == 'X' || op == 'D') ? run : 0, dt = (op == 'M' || op == 'X' || op == 'I') ? run : 0;
        if ((op != 'M' && op != 'X' && op != 'I' && op != 'D') || q + dq > qlen || t + dt > tlen) {
            free(s);
            return NULL;
        }
        if (op == 'M') {
            if (long_form) {
                s[len++] = '=';
                for (size_t k = 0; k < run; ++k) s[len++] = upper_c(target[t + k]);
            } else {
                len += (size_t)sprintf(s + len, ":%zu", run);
            }
        } else if (op == 'X') {
            s[len++] = '*';
            s[len++] = lower_c(target[t]);
            s[len++] = lower_c(query[q]);
        } else if (op == 'I') {
            s[len++] = '-';
            for (size_t k = 0; k < run; ++k) s[len++] = lower_c(target[t + k]);
        } else {
            s[len++] = '+';
            for (size_t k = 0; k < run; ++k) s[len++] = lower_c(query[q + k]);
        }
        q += dq;
        t += dt;
        i = j;
    }
    if (q != qlen || t != tlen) {
        free(s);
        return NULL;
    }
    s[len] = 0;
    return s;
}

/* alignment_to_paf + "\tcs:Z:" + the tag of r's alignment; `query` as given (reverse-complemented here on '-' results);
 * malloc'ed line without trailing newline, NULL when the alignment does not fit the sequences */
char* awo_alignment_to_paf_cs(const awo_result_t* r, const char* qname, const uint8_t* query, size_t qlen, const char* tname,
                              const uint8_t* target, size_t tlen, int long_form) {
    uint8_t* rc = NULL;
    if (r->is_reverse) {
        rc = (uint8_t*)malloc(qlen + 1);
        awo_reverse_complement(query, qlen, rc);
    }
    char* tag = awo_cs_string(r->cigar_bytes, r->cigar_len, rc ? rc : query, qlen, target, tlen, long_form);
    free(rc);
    if (!tag) return NULL;
    char* line = awo_alignment_to_paf(r, qname, qlen, tname, tlen);
    const size_t ll = strlen(line), tl = strlen(tag);
    char* out = (char*)malloc(ll + 6 + tl + 1);
    memcpy(out, line, ll);
    memcpy(out + ll, "\tcs:Z:", 6);
    memcpy(out + ll + 6, tag, tl + 1);
    free(line);
    free(tag);
    return out;
}
