/* oracle/ft8_oracle_codec.c -- CPU restatement, part 2: Costas sync, top-K heap, LLRs,
 * LDPC(174,91) belief propagation, CRC-14, 77-bit unpacking, the daemon's candidate loop,
 * and the encoder used to synthesise inputs.  TEST INFRASTRUCTURE ONLY (see ft8_oracle.h).
 */
#include "ft8_oracle.h"
#include "ft8_tables.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

/* ======================================================================================
 * a7  Costas sync score                                  ref: ft8_lib/ft8/decode.c:35-108
 * ====================================================================================== */
static long wf_index(const orc_waterfall_t *wf, const orc_candidate_t *c) { /* ref: decode.c:35-42 */
    long o = c->time_offset;
    o = o * wf->time_osr + c->time_sub;
    o = o * wf->freq_osr + c->freq_sub;
    o = o * wf->num_bins + c->freq_offset;
    return o;
}

/* ref: ft4_sync_score, decode.c:110-171: four 4-symbol groups at symbols 1, 34, 67, 100, one Costas array each */
static int orc_sync_score_ft4(const orc_waterfall_t *wf, const orc_candidate_t *c) {
    const uint8_t *base = wf->mag + wf_index(wf, c);
    const int stride = wf->block_stride;
    int total = 0, terms = 0;
    for (int grp = 0; grp < 4; ++grp) {
        for (int k = 0; k < 4; ++k) {
            const int rel = 1 + 33 * grp + k;
            const int row = c->time_offset + rel;
            if (row < 0) continue;
            if (row >= wf->num_blocks) break;
            const uint8_t *p = base + (long)rel * stride;
            const int tone = kFt4tCostas[grp][k];
            if (tone > 0) { total += p[tone] - p[tone - 1]; ++terms; }
            if (tone < 3) { total += p[tone] - p[tone + 1]; ++terms; }
            if (k > 0 && row > 0) { total += p[tone] - p[tone - stride]; ++terms; }
            if (k + 1 < 4 && row + 1 < wf->num_blocks) { total += p[tone] - p[tone + stride]; ++terms; }
        }
    }
    if (terms > 0) total /= terms;
    return total;
}

int orc_sync_score(const orc_waterfall_t *wf, const orc_candidate_t *c) {
    if (wf->protocol == 0) return orc_sync_score_ft4(wf, c); /* PROTO_FT4 == 0, constants.h:6-10 */
    const uint8_t *base = wf->mag + wf_index(wf, c);
    const int stride = wf->block_stride;
    int total = 0, terms = 0;
    for (int grp = 0; grp < 3; ++grp) {
        for (int k = 0; k < 7; ++k) {
            const int rel = 36 * grp + k;
            const int row = c->time_offset + rel;
            if (row < 0) continue;
            if (row >= wf->num_blocks) break; /* leaves this Costas group only */
            const uint8_t *p = base + (long)rel * stride;
            const int tone = kFt8tCostas[k];
            if (tone > 0) { total += p[tone] - p[tone - 1]; ++terms; }
            if (tone < 7) { total += p[tone] - p[tone + 1]; ++terms; }
            if (k > 0 && row > 0) { total += p[tone] - p[tone - stride]; ++terms; }
            if (k + 1 < 7 && row + 1 < wf->num_blocks) { total += p[tone] - p[tone + stride]; ++terms; }
        }
    }
    if (terms > 0) total /= terms; /* C division: truncates toward zero */
    return total;
}

/* ======================================================================================
 * a8  candidate search with a size-K min-heap             ref: decode.c:173-234, 388-435
 * ====================================================================================== */
static void sift_down(orc_candidate_t *h, int n) { /* ref: heapify_down, decode.c:388-415 */
    int cur = 0;
    for (;;) {
        int pick = cur;
        const int l = 2 * cur + 1, r = l + 1;
        if (l < n && h[l].score < h[pick].score) pick = l;
        if (r < n && h[r].score < h[pick].score) pick = r;
        if (pick == cur) return;
        const orc_candidate_t t = h[pick]; h[pick] = h[cur]; h[cur] = t;
        cur = pick;
    }
}
static void sift_up(orc_candidate_t *h, int n) { /* ref: heapify_up, decode.c:417-435 */
    int cur = n - 1;
    while (cur > 0) {
        const int par = (cur - 1) / 2;
        if (h[cur].score >= h[par].score) return;
        const orc_candidate_t t = h[par]; h[par] = h[cur]; h[cur] = t;
        cur = par;
    }
}

int orc_find_sync(const orc_waterfall_t *wf, int cap, orc_candidate_t *heap, int min_score) {
    int n = 0;
    orc_candidate_t c;
    for (int ts = 0; ts < wf->time_osr; ++ts) {
        for (int fs = 0; fs < wf->freq_osr; ++fs) {
            for (int to = -12; to < 24; ++to) {
                for (int fo = 0; fo + 7 < wf->num_bins; ++fo) {
                    c.time_sub = (uint8_t)ts; c.freq_sub = (uint8_t)fs;
                    c.time_offset = (int16_t)to; c.freq_offset = (int16_t)fo;
                    c.score = (int16_t)orc_sync_score(wf, &c);
                    if (c.score < min_score) continue;
                    if (n == cap && c.score > heap[0].score) { /* evict the weakest */
                        heap[0] = heap[n - 1];
                        --n;
                        sift_down(heap, n);
                    }
                    if (n < cap) {
                        heap[n++] = c;
                        sift_up(heap, n);
                    }
                }
            }
        }
    }
    for (int rest = n; rest > 1;) { /* in-place heap sort -> descending score */
        const orc_candidate_t t = heap[rest - 1]; heap[rest - 1] = heap[0]; heap[0] = t;
        --rest;
        sift_down(heap, rest);
    }
    return n;
}

/* ======================================================================================
 * a9-a10  LLRs                                 ref: decode.c:265-314, 378-386, 453-466
 * ====================================================================================== */
static inline float fmax2(float a, float b) { return (a >= b) ? a : b; }
static inline float fmax4(float a, float b, float c, float d) { return fmax2(fmax2(a, b), fmax2(c, d)); }

void orc_extract_llr(const orc_waterfall_t *wf, const orc_candidate_t *c, float *llr) {
    const uint8_t *base = wf->mag + wf_index(wf, c);
    if (wf->protocol == 0) { /* ref: ft4_extract_likelihood / ft4_extract_symbol, decode.c:236-263, 438-450 */
        for (int k = 0; k < 87; ++k) {
            const int sym = k + (k < 29 ? 5 : (k < 58 ? 9 : 13));
            const int row = c->time_offset + sym;
            float *o = llr + 2 * k;
            if (row < 0 || row >= wf->num_blocks) { o[0] = o[1] = 0; continue; }
            const uint8_t *p = base + (long)sym * wf->block_stride;
            float s[4];
            for (int j = 0; j < 4; ++j) s[j] = (float)p[kFt4tGray[j]];
            o[0] = fmax2(s[2], s[3]) - fmax2(s[0], s[1]);
            o[1] = fmax2(s[1], s[3]) - fmax2(s[0], s[2]);
        }
        return;
    }
    for (int k = 0; k < 58; ++k) {
        const int sym = k + (k < 29 ? 7 : 14);
        const int row = c->time_offset + sym;
        float *o = llr + 3 * k;
        if (row < 0 || row >= wf->num_blocks) { o[0] = o[1] = o[2] = 0; continue; }
        const uint8_t *p = base + (long)sym * wf->block_stride;
        float s[8];
        for (int j = 0; j < 8; ++j) s[j] = (float)p[kFt8tGray[j]];
        o[0] = fmax4(s[4], s[5], s[6], s[7]) - fmax4(s[0], s[1], s[2], s[3]);
        o[1] = fmax4(s[2], s[3], s[6], s[7]) - fmax4(s[0], s[1], s[4], s[5]);
        o[2] = fmax4(s[1], s[3], s[5], s[7]) - fmax4(s[0], s[2], s[4], s[6]);
    }
}

void orc_normalize_llr(float *llr) { /* ref: ftx_normalize_logl, decode.c:295-314 */
    float s1 = 0, s2 = 0;
    for (int k = 0; k < FT8T_N; ++k) { s1 += llr[k]; s2 += llr[k] * llr[k]; }
    const float inv_n = 1.0f / FT8T_N;
    const float var = (s2 - (s1 * s1 * inv_n)) * inv_n;
    const float g = sqrtf(24.0f / var);
    for (int k = 0; k < FT8T_N; ++k) llr[k] *= g;
}

/* ======================================================================================
 * a11  sum-product LDPC decoder                                  ref: ldpc.c:111-251
 * ====================================================================================== */
static float tanh_pade(float x) { /* ref: fast_tanh, ldpc.c:220-239 */
    if (x < -4.97f) return -1.0f;
    if (x > 4.97f) return 1.0f;
    const float x2 = x * x;
    const float a = x * (945.0f + x2 * (105.0f + x2));
    const float b = 945.0f + x2 * (420.0f + x2 * 15.0f);
    return a / b;
}
static float atanh_pade(float x) { /* ref: fast_atanh, ldpc.c:241-251 */
    const float x2 = x * x;
    const float a = x * (945.0f + x2 * (-735.0f + x2 * 64.0f));
    const float b = (945.0f + x2 * (-1050.0f + x2 * 225.0f));
    return a / b;
}
static int parity_errors(const uint8_t *bits) { /* ref: ldpc_check, ldpc.c:111-128 */
    int bad = 0;
    for (int m = 0; m < FT8T_M; ++m) {
        uint8_t x = 0;
        for (int j = 0; j < kFt8tNumRows[m]; ++j) x ^= bits[kFt8tNm[m][j] - 1];
        if (x) ++bad;
    }
    return bad;
}

void orc_bp_decode(const float *llr, int max_iters, uint8_t *plain, int *errors_out) {
    float v2c_in[FT8T_N][3]; /* "tov": check -> variable messages */
    float c_in[FT8T_M][7];   /* "toc": tanh of variable -> check messages */
    int best = FT8T_M;
    memset(v2c_in, 0, sizeof(v2c_in));
    /* ldpc.c leaves plain[] unwritten when no round runs (max_iters = 0); the kernels report the all-zero word */
    memset(plain, 0, FT8T_N);
    for (int it = 0; it < max_iters; ++it) {
        int ones = 0;
        for (int n = 0; n < FT8T_N; ++n) {
            plain[n] = ((llr[n] + v2c_in[n][0] + v2c_in[n][1] + v2c_in[n][2]) > 0) ? 1 : 0;
            ones += plain[n];
        }
        if (ones == 0) break; /* all-zero word is not a message.  ref: ldpc.c:153-157 */
        const int bad = parity_errors(plain);
        if (bad < best) {
            best = bad;
            if (bad == 0) break;
        }
        for (int m = 0; m < FT8T_M; ++m) {
            for (int j = 0; j < kFt8tNumRows[m]; ++j) {
                const int n = kFt8tNm[m][j] - 1;
                float t = llr[n];
                for (int e = 0; e < 3; ++e)
                    if (kFt8tMn[n][e] - 1 != m) t += v2c_in[n][e];
                c_in[m][j] = tanh_pade(-t / 2);
            }
        }
        for (int n = 0; n < FT8T_N; ++n) {
            for (int e = 0; e < 3; ++e) {
                const int m = kFt8tMn[n][e] - 1;
                float prod = 1.0f;
                for (int j = 0; j < kFt8tNumRows[m]; ++j)
                    if (kFt8tNm[m][j] - 1 != n) prod *= c_in[m][j];
                v2c_in[n][e] = -2 * atanh_pade(prod);
            }
        }
    }
    *errors_out = best;
}

/* ======================================================================================
 * a12  CRC-14                                                         ref: crc.c:10-43
 * ====================================================================================== */
uint16_t orc_crc14(const uint8_t *msg, int num_bits) {
    uint16_t rem = 0;
    for (int b = 0, byte = 0; b < num_bits; ++b) {
        if ((b & 7) == 0) rem ^= (uint16_t)(msg[byte++] << 6);
        rem = (rem & 0x2000u) ? (uint16_t)((rem << 1) ^ 0x2757u) : (uint16_t)(rem << 1);
    }
    return rem & 0x3FFFu;
}

/* ======================================================================================
 * a13  77-bit message -> text                    ref: unpack.c:18-427, text.c:5-253
 * ====================================================================================== */
static char alpha(int c, int table) { /* ref: charn, text.c:172-207 */
    if (table != 2 && table != 3) { if (c == 0) return ' '; c -= 1; }
    if (table != 4) { if (c < 10) return (char)('0' + c); c -= 10; }
    if (table != 3) { if (c < 26) return (char)('A' + c); c -= 26; }
    if (table == 0) { if (c < 5) return "+-./?"[c]; }
    else if (table == 5) { if (c == 0) return '/'; }
    return '_';
}
static char *strip(char *s) { /* ref: trim, text.c:5-33 */
    while (*s == ' ') ++s;
    for (int k = (int)strlen(s) - 1; k >= 0 && s[k] == ' '; --k) s[k] = 0;
    return s;
}
static void put_int(char *dst, int v, int width, int sign) { /* ref: int_to_dd, text.c:138-170 */
    if (v < 0) { *dst++ = '-'; v = -v; } else if (sign) { *dst++ = '+'; }
    int div = 1;
    for (int k = 1; k < width; ++k) div *= 10;
    for (; div >= 1; div /= 10) { const int d = v / div; *dst++ = (char)('0' + d); v -= d * div; }
    *dst = 0;
}

static int unpack_call(uint32_t n28, int ip, int i3, char *out) { /* ref: unpack_callsign, unpack.c:18-116 */
    const uint32_t NTOK = 2063592u, MAX22 = 4194304u;
    if (n28 < NTOK) {
        if (n28 <= 2) { strcpy(out, n28 == 0 ? "DE" : n28 == 1 ? "QRZ" : "CQ"); return 0; }
        if (n28 <= 1002) { strcpy(out, "CQ "); put_int(out + 3, (int)n28 - 3, 3, 0); return 0; }
        if (n28 <= 532443u) {
            uint32_t n = n28 - 1003;
            char a[5]; a[4] = 0;
            for (int k = 3; k >= 0; --k) { a[k] = alpha((int)(n % 27), 4); if (k) n /= 27; }
            const char *t = a; while (*t == ' ') ++t;
            strcpy(out, "CQ "); strcat(out, t);
            return 0;
        }
        return -1;
    }
    n28 -= NTOK;
    if (n28 < MAX22) { strcpy(out, "<...>"); return 0; }
    uint32_t n = n28 - MAX22;
    char cs[7]; cs[6] = 0;
    cs[5] = alpha((int)(n % 27), 4); n /= 27;
    cs[4] = alpha((int)(n % 27), 4); n /= 27;
    cs[3] = alpha((int)(n % 27), 4); n /= 27;
    cs[2] = alpha((int)(n % 10), 3); n /= 10;
    cs[1] = alpha((int)(n % 36), 2); n /= 36;
    cs[0] = alpha((int)(n % 37), 1);
    strcpy(out, strip(cs));
    if (out[0] == 0) return -1;
    if (ip) { if (i3 == 1) strcat(out, "/R"); else if (i3 == 2) strcat(out, "/P"); }
    return 0;
}

static int unpack_std(const uint8_t *a, int i3, char *to, char *de, char *extra) { /* ref: unpack_type1, unpack.c:118-214 */
    uint32_t n28a = ((uint32_t)a[0] << 21) | ((uint32_t)a[1] << 13) | ((uint32_t)a[2] << 5) | (a[3] >> 3);
    uint32_t n28b = ((uint32_t)(a[3] & 7) << 26) | ((uint32_t)a[4] << 18) | ((uint32_t)a[5] << 10) | ((uint32_t)a[6] << 2) | (a[7] >> 6);
    const int ir = (a[7] >> 5) & 1;
    const uint16_t g = (uint16_t)(((a[7] & 0x1F) << 10) | (a[8] << 2) | (a[9] >> 6));
    if (unpack_call(n28a >> 1, n28a & 1, i3, to) < 0) return -1;
    if (unpack_call(n28b >> 1, n28b & 1, i3, de) < 0) return -2;
    char *d = extra;
    if (g <= 32400) {
        if (ir) { *d++ = 'R'; *d++ = ' '; }
        uint16_t n = g;
        d[4] = 0;
        d[3] = (char)('0' + n % 10); n /= 10;
        d[2] = (char)('0' + n % 10); n /= 10;
        d[1] = (char)('A' + n % 18); n /= 18;
        d[0] = (char)('A' + n % 18);
    } else {
        const int rpt = g - 32400;
        switch (rpt) {
        case 1: extra[0] = 0; break;
        case 2: strcpy(d, "RRR"); break;
        case 3: strcpy(d, "RR73"); break;
        case 4: strcpy(d, "73"); break;
        default:
            if (ir) *d++ = 'R';
            put_int(d, rpt - 35, 2, 1);
        }
    }
    return 0;
}

static int unpack_free(const uint8_t *a, char *text) { /* ref: unpack_text, unpack.c:216-246 */
    uint8_t b[9];
    uint8_t carry = 0;
    for (int k = 0; k < 9; ++k) { b[k] = (uint8_t)(carry | (a[k] >> 1)); carry = (a[k] & 1) ? 0x80 : 0; }
    char c[14]; c[13] = 0;
    for (int pos = 12; pos >= 0; --pos) {
        uint16_t rem = 0;
        for (int k = 0; k < 9; ++k) { rem = (uint16_t)((rem << 8) | b[k]); b[k] = (uint8_t)(rem / 42); rem %= 42; }
        c[pos] = alpha(rem, 0);
    }
    strcpy(text, strip(c));
    return 0;
}

static int unpack_telem(const uint8_t *a, char *text) { /* ref: unpack_telemetry, unpack.c:248-274 */
    uint8_t carry = 0;
    for (int k = 0; k < 9; ++k) {
        const uint8_t v = (uint8_t)((carry << 7) | (a[k] >> 1));
        carry = a[k] & 1;
        text[2 * k] = "0123456789ABCDEF"[v >> 4];
        text[2 * k + 1] = "0123456789ABCDEF"[v & 15];
    }
    text[18] = 0;
    return 0;
}

static int unpack_nonstd(const uint8_t *a, char *to, char *de, char *extra) { /* ref: unpack_nonstandard, unpack.c:276-348 */
    uint64_t n58 = ((uint64_t)(a[1] & 0x0F) << 54) | ((uint64_t)a[2] << 46) | ((uint64_t)a[3] << 38) | ((uint64_t)a[4] << 30) |
                   ((uint64_t)a[5] << 22) | ((uint64_t)a[6] << 14) | ((uint64_t)a[7] << 6) | ((uint64_t)a[8] >> 2);
    const int flip = (a[8] >> 1) & 1;
    const int rpt = ((a[8] & 1) << 1) | (a[9] >> 7);
    const int cq = (a[9] >> 6) & 1;
    char c11[12]; c11[11] = 0;
    for (int k = 10; k >= 0; --k) { c11[k] = alpha((int)(n58 % 38), 5); if (k) n58 /= 38; }
    char hashed[8]; strcpy(hashed, "<...>");
    char *first = flip ? c11 : hashed, *second = flip ? hashed : c11;
    if (!cq) {
        strcpy(to, strip(first));
        strcpy(extra, rpt == 1 ? "RRR" : rpt == 2 ? "RR73" : rpt == 3 ? "73" : "");
    } else {
        strcpy(to, "CQ");
        extra[0] = 0;
    }
    strcpy(de, strip(second));
    return 0;
}

int orc_unpack77(const uint8_t *a, char *text) { /* ref: unpack77 + unpack77_fields, unpack.c:350-427 */
    char to[16], de[16], extra[24];
    to[0] = de[0] = extra[0] = 0;
    int rc = -1;
    const int i3 = (a[9] >> 3) & 7;
    if (i3 == 0) {
        const int n3 = ((a[8] << 2) & 4) | ((a[9] >> 6) & 3);
        if (n3 == 0) rc = unpack_free(a, extra);
        else if (n3 == 5) rc = unpack_telem(a, extra);
    } else if (i3 == 1 || i3 == 2) {
        rc = unpack_std(a, i3, to, de, extra);
    } else if (i3 == 4) {
        rc = unpack_nonstd(a, to, de, extra);
    }
    if (rc < 0) return rc;
    char *d = text;
    *d = 0;
    if (to[0]) { d = stpcpy(d, to); *d++ = ' '; }
    if (de[0]) { d = stpcpy(d, de); *d++ = ' '; }
    d = stpcpy(d, extra);
    *d = 0;
    return 0;
}

/* ======================================================================================
 * a14  one candidate end to end                                    ref: decode.c:316-376
 * ====================================================================================== */
int orc_decode(const orc_waterfall_t *wf, const orc_candidate_t *c, int max_iters, orc_message_t *msg, orc_status_t *st,
               float *llr_out, uint8_t *plain_out) {
    float llr[FT8T_N];
    uint8_t plain[FT8T_N];
    orc_extract_llr(wf, c, llr);
    orc_normalize_llr(llr);
    if (llr_out) memcpy(llr_out, llr, sizeof(llr));
    orc_bp_decode(llr, max_iters, plain, &st->ldpc_errors);
    if (plain_out) memcpy(plain_out, plain, sizeof(plain));
    if (st->ldpc_errors > 0) return 0;
    uint8_t a91[12];
    memset(a91, 0, sizeof(a91));
    for (int k = 0; k < FT8T_K; ++k) /* ref: pack_bits, decode.c:527-550 */
        if (plain[k]) a91[k >> 3] |= (uint8_t)(0x80 >> (k & 7));
    st->crc_extracted = (uint16_t)(((a91[9] & 7) << 11) | (a91[10] << 3) | (a91[11] >> 5)); /* ref: crc.c:40-43 */
    a91[9] &= 0xF8;
    a91[10] = 0;
    st->crc_calculated = orc_crc14(a91, 82);
    if (st->crc_extracted != st->crc_calculated) return 0;
    if (wf->protocol == 0) /* FT4 scrambles the 77 message bits before CRC/FEC, decode.c:355-363 */
        for (int k = 0; k < 10; ++k) a91[k] ^= kFt4tXor[k];
    char text[40];
    st->unpack_status = orc_unpack77(a91, text);
    if (st->unpack_status < 0) return 0;
    memset(msg->text, 0, sizeof(msg->text));
    strncpy(msg->text, text, sizeof(msg->text) - 1);
    msg->hash = st->crc_extracted;
    return 1;
}

/* ======================================================================================
 * a15  the daemon's candidate loop, duplicate table and CQ filter
 *                                                       ref: rtlsdr_ft8d.c:1437-1523
 * Deviations, all where the reference's behaviour is undefined:
 *   - a full table (max_messages distinct messages) makes the reference probe forever
 *     (:1490-1502); here the message is dropped after one full cycle;
 *   - strtok() returning NULL for an empty text would crash strncmp (:1509-1510); here it
 *     is treated as "not CQ".  A missing 2nd/3rd token prints as glibc's "(null)" (:1512-1514).
 * ====================================================================================== */
/* The table + filter alone, over an already decoded candidate list (ok[k] != 0: msgs[k] holds candidate k's message):
 * what ft8_subsystem() does after each successful ft8_decode(), rtlsdr_ft8d.c:1467-1522.  Callable with hand-made
 * messages, which is how the edge cases (hash clashes, 2-token CQ, a full table) are pinned to the reference's own loop
 * (oracle/ref_harness.c: ref_subsystem_scripted) and then asked of the CUDA spots kernel. */
int orc_spots(const orc_candidate_t *cand, const uint8_t *ok, const orc_message_t *msgs, int n_cand, int max_messages, int min_score,
              int freq_osr, orc_result_t *results, orc_slot_report_t *rep) {
    orc_message_t *table = (orc_message_t *)calloc((size_t)max_messages, sizeof(orc_message_t));
    uint8_t *used = (uint8_t *)calloc((size_t)max_messages, 1);
    int n_new = 0;
    for (int k = 0; k < n_cand; ++k) {
        const orc_candidate_t *c = &cand[k];
        if (c->score < min_score || !ok[k]) continue;
        const float freq_hz = (c->freq_offset + (float)c->freq_sub / freq_osr) * 6.25f;
        const orc_message_t msg = msgs[k];
        int slot = msg.hash % max_messages, probes = 0, dup = 0, empty = 0;
        while (probes < max_messages) {
            if (!used[slot]) { empty = 1; break; }
            if (table[slot].hash == msg.hash && strcmp(table[slot].text, msg.text) == 0) { dup = 1; break; }
            slot = (slot + 1) % max_messages;
            ++probes;
        }
        if (dup || !empty) continue;
        table[slot] = msg;
        used[slot] = 1;
        if (rep && n_new < 512) { rep->msgs[n_new] = msg; rep->freq_hz[n_new] = freq_hz; rep->score[n_new] = c->score; }
        char work[40];
        memset(work, 0, sizeof(work));
        memcpy(work, msg.text, sizeof(msg.text));   /* 25 bytes, NUL-terminated by the zero fill */
        char *save = NULL;
        const char *tok = strtok_r(work, " ", &save);
        if (tok && strncmp(tok, "CQ", 2) == 0 && n_new < max_messages) {
            const char *call = strtok_r(NULL, " ", &save);
            snprintf(results[n_new].call, sizeof(results[n_new].call), "%.12s", call ? call : "(null)");
            const char *loc = strtok_r(NULL, " ", &save);
            snprintf(results[n_new].loc, sizeof(results[n_new].loc), "%.6s", loc ? loc : "(null)");
            results[n_new].freq = (int32_t)freq_hz;
            results[n_new].snr = (int32_t)c->score;
        }
        ++n_new;
    }
    if (rep) rep->n_unique = n_new;
    free(table); free(used);
    return n_new;
}

int orc_decode_waterfall(const orc_waterfall_t *wf, int max_candidates, int max_messages, int min_score, int ldpc_iters,
                         orc_result_t *results, orc_slot_report_t *rep, orc_candidate_t *cand_out) {
    orc_candidate_t *cand = (orc_candidate_t *)malloc(sizeof(orc_candidate_t) * (size_t)max_candidates);
    const int n_cand = orc_find_sync(wf, max_candidates, cand, min_score);
    if (cand_out) memcpy(cand_out, cand, sizeof(orc_candidate_t) * (size_t)n_cand);
    orc_message_t *msgs = (orc_message_t *)calloc((size_t)(n_cand > 0 ? n_cand : 1), sizeof(orc_message_t));
    uint8_t *ok = (uint8_t *)calloc((size_t)(n_cand > 0 ? n_cand : 1), 1);
    if (rep) memset(rep, 0, sizeof(*rep));
    for (int k = 0; k < n_cand; ++k) {   /* ft8_decode() is a pure function of (waterfall, candidate): decoding first changes nothing */
        orc_status_t st;
        if (cand[k].score < min_score) continue;
        ok[k] = (uint8_t)orc_decode(wf, &cand[k], ldpc_iters, &msgs[k], &st, NULL, NULL);
    }
    const int n_new = orc_spots(cand, ok, msgs, n_cand, max_messages, min_score, 2 /* K_FREQ_OSR, rtlsdr_ft8d.c:1470 */, results, rep);
    if (rep) rep->n_cand = n_cand;
    free(cand); free(msgs); free(ok);
    return n_new;
}

int orc_subsystem(const float *i_s, const float *q_s, int max_candidates, int max_messages, int min_score, int ldpc_iters,
                  orc_result_t *results, orc_slot_report_t *rep, uint8_t *wf_out, orc_candidate_t *cand_out) {
    uint8_t *mag = (uint8_t *)malloc(ORC_WF_BYTES);
    orc_waterfall_daemon(i_s, q_s, mag);
    if (wf_out) memcpy(wf_out, mag, ORC_WF_BYTES);
    orc_waterfall_t wf = { 92, 92, 256, 2, 2, mag, 1024, 1 };
    const int n = orc_decode_waterfall(&wf, max_candidates, max_messages, min_score, ldpc_iters, results, rep, cand_out);
    free(mag);
    return n;
}

/* ======================================================================================
 * encoder (input synthesis only)         ref: pack.c:20-232, crc.c:45-63, encode.c:22-125
 * ====================================================================================== */
static int index_of(const char *set, char c) { const char *p = strchr(set, c); return (p && c) ? (int)(p - set) : -1; }

static int32_t pack_call(const char *call) { /* ref: pack28, pack.c:20-101 (standard calls + DE/QRZ/CQ) */
    if (strcmp(call, "DE") == 0) return 0;
    if (strcmp(call, "QRZ") == 0) return 1;
    if (strcmp(call, "CQ") == 0) return 2;
    const int len = (int)strlen(call);
    char c6[7] = "      ";
    if (len >= 3 && call[2] >= '0' && call[2] <= '9' && len <= 6) memcpy(c6, call, (size_t)len);
    else if (len >= 2 && call[1] >= '0' && call[1] <= '9' && len <= 5) memcpy(c6 + 1, call, (size_t)len);
    else return -1;
    const int i0 = index_of(" 0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[0]);
    const int i1 = index_of("0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[1]);
    const int i2 = index_of("0123456789", c6[2]);
    const int i3 = index_of(" ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[3]);
    const int i4 = index_of(" ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[4]);
    const int i5 = index_of(" ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[5]);
    if (i0 < 0 || i1 < 0 || i2 < 0 || i3 < 0 || i4 < 0 || i5 < 0) return -1;
    int32_t n = i0;
    n = n * 36 + i1; n = n * 10 + i2; n = n * 27 + i3; n = n * 27 + i4; n = n * 27 + i5;
    return 2063592 + 4194304 + n;
}

static uint16_t pack_extra(const char *x) { /* ref: packgrid, pack.c:131-176 */
    if (!x || !x[0]) return 32400 + 1;
    if (strcmp(x, "RRR") == 0) return 32400 + 2;
    if (strcmp(x, "RR73") == 0) return 32400 + 3;
    if (strcmp(x, "73") == 0) return 32400 + 4;
    if (x[0] >= 'A' && x[0] <= 'R' && x[1] >= 'A' && x[1] <= 'R' && x[2] >= '0' && x[2] <= '9' && x[3] >= '0' && x[3] <= '9')
        return (uint16_t)((((x[0] - 'A') * 18 + (x[1] - 'A')) * 10 + (x[2] - '0')) * 10 + (x[3] - '0'));
    if (x[0] == 'R') return (uint16_t)((32400 + 35 + atoi(x + 1)) | 0x8000);
    return (uint16_t)(32400 + 35 + atoi(x));
}

int orc_pack_std(const char *call_to, const char *call_de, const char *extra, uint8_t *b) { /* ref: pack77_1, pack.c:178-232 */
    int32_t a = pack_call(call_to), d = pack_call(call_de);
    if (a < 0 || d < 0) return -1;
    const uint16_t g = pack_extra(extra);
    const uint32_t n28a = (uint32_t)a << 1, n28b = (uint32_t)d << 1;
    b[0] = (uint8_t)(n28a >> 21); b[1] = (uint8_t)(n28a >> 13); b[2] = (uint8_t)(n28a >> 5);
    b[3] = (uint8_t)((uint8_t)(n28a << 3) | (uint8_t)(n28b >> 26));
    b[4] = (uint8_t)(n28b >> 18); b[5] = (uint8_t)(n28b >> 10); b[6] = (uint8_t)(n28b >> 2);
    b[7] = (uint8_t)((uint8_t)(n28b << 6) | (uint8_t)(g >> 10));
    b[8] = (uint8_t)(g >> 2);
    b[9] = (uint8_t)((uint8_t)(g << 6) | (1u << 3));
    return 0;
}

void orc_pack_text(const char *text, uint8_t *b) { /* ref: packtext77, pack.c:234-299 */
    int len = (int)strlen(text);
    while (*text == ' ') { ++text; --len; }
    while (len > 0 && text[len - 1] == ' ') --len;
    memset(b, 0, 10);
    for (int j = 0; j < 13; ++j) {
        uint16_t x = 0;
        for (int k = 8; k >= 0; --k) { x = (uint16_t)(x + b[k] * 42u); b[k] = (uint8_t)x; x >>= 8; }
        int q = (j < len) ? index_of(" 0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ+-./?", text[j]) : 0;
        x = (uint16_t)((q > 0 ? q : 0) << 1);
        for (int k = 8; k >= 0 && x; --k) { x = (uint16_t)(x + b[k]); b[k] = (uint8_t)x; x >>= 8; }
    }
    b[8] &= 0xFE;
    b[9] = 0;
}

/* ---- pack77(): whole message text -> payload.  ref: pack77, pack.c:284-301 = pack77_1 (:167-218) else packtext77 (:220-282) ---- */
/* The fields are NOT separate strings in the reference: pack28() is handed a pointer into the message and looks at what follows. */
static int begins(const char *s, const char *prefix) { return strncmp(s, prefix, strlen(prefix)) == 0; }

static int32_t msg_pack28(const char *cs) { /* ref: pack28, pack.c:22-98 */
    if (begins(cs, "DE ")) return 0;
    if (begins(cs, "QRZ ")) return 1;
    if (begins(cs, "CQ ")) return 2;
    int length = 0;
    while (cs[length] != ' ' && cs[length] != 0) ++length;
    /* characters the reference tests beyond a short field: cs[length] is the delimiter, nothing further is ever decisive */
    const char c1 = length >= 1 ? cs[1] : 0, c2 = length >= 2 ? cs[2] : 0;
    char c6[6] = { ' ', ' ', ' ', ' ', ' ', ' ' };
    if (begins(cs, "3DA0") && length <= 7) { /* :45-49 */
        memcpy(c6, "3D0", 3);
        memcpy(c6 + 3, cs + 4, (size_t)(length - 4));
    } else if (begins(cs, "3X") && ((c2 >= 'A' && c2 <= 'Z') || (c2 >= 'a' && c2 <= 'z')) && length <= 7) { /* :50-55 */
        memcpy(c6, "Q", 1);
        memcpy(c6 + 1, cs + 2, (size_t)(length - 2));
    } else if (c2 >= '0' && c2 <= '9' && length <= 6) { /* :58-62 */
        memcpy(c6, cs, (size_t)length);
    } else if (c1 >= '0' && c1 <= '9' && length <= 5) { /* :63-67 */
        memcpy(c6 + 1, cs, (size_t)length);
    }
    const int i0 = index_of(" 0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[0]);
    const int i1 = index_of("0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[1]);
    const int i2 = index_of("0123456789", c6[2]);
    const int i3 = index_of(" ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[3]);
    const int i4 = index_of(" ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[4]);
    const int i5 = index_of(" ABCDEFGHIJKLMNOPQRSTUVWXYZ", c6[5]);
    if (i0 < 0 || i1 < 0 || i2 < 0 || i3 < 0 || i4 < 0 || i5 < 0) return -1;
    int32_t n = i0;
    n = n * 36 + i1; n = n * 10 + i2; n = n * 27 + i3; n = n * 27 + i4; n = n * 27 + i5;
    return 2063592 + 4194304 + n;
}

static int msg_dd_to_int(const char *str, int length) { /* ref: dd_to_int, text.c:103-131 */
    int result = 0, i, negative = 0;
    if (str[0] == '-') { negative = 1; i = 1; }
    else i = (str[0] == '+') ? 1 : 0;
    while (i < length && str[i] != 0 && str[i] >= '0' && str[i] <= '9') { result = result * 10 + (str[i] - '0'); ++i; }
    return negative ? -result : result;
}

static uint16_t msg_packgrid(const char *g) { /* ref: packgrid, pack.c:122-164; g = the text behind the second blank, or NULL */
    if (g == 0) return 32400 + 1;
    if (strcmp(g, "RRR") == 0) return 32400 + 2;
    if (strcmp(g, "RR73") == 0) return 32400 + 3;
    if (strcmp(g, "73") == 0) return 32400 + 4;
    if (g[0] >= 'A' && g[0] <= 'R' && g[1] >= 'A' && g[1] <= 'R' && g[2] >= '0' && g[2] <= '9' && g[3] >= '0' && g[3] <= '9') {
        uint16_t v = (uint16_t)(g[0] - 'A');
        v = (uint16_t)(v * 18 + (g[1] - 'A'));
        v = (uint16_t)(v * 10 + (g[2] - '0'));
        v = (uint16_t)(v * 10 + (g[3] - '0'));
        return v;
    }
    if (g[0] == 'R') {
        const uint16_t irpt = (uint16_t)(35 + msg_dd_to_int(g + 1, 3));
        return (uint16_t)((32400 + irpt) | 0x8000);
    }
    const uint16_t irpt = (uint16_t)(35 + msg_dd_to_int(g, 3));
    return (uint16_t)(32400 + irpt);
}

int orc_pack77(const char *msg, uint8_t *b) { /* returns 0 = standard message, 1 = free text (the reference returns 0 for both) */
    const char *s1 = strchr(msg, ' ');
    if (s1 != 0) {
        const int32_t a = msg_pack28(msg), d = msg_pack28(s1 + 1);
        if (a >= 0 && d >= 0) {
            const char *s2 = strchr(s1 + 1, ' ');
            const uint16_t g = msg_packgrid(s2 ? s2 + 1 : 0);
            const uint32_t n28a = (uint32_t)a << 1, n28b = (uint32_t)d << 1;
            b[0] = (uint8_t)(n28a >> 21); b[1] = (uint8_t)(n28a >> 13); b[2] = (uint8_t)(n28a >> 5);
            b[3] = (uint8_t)((uint8_t)(n28a << 3) | (uint8_t)(n28b >> 26));
            b[4] = (uint8_t)(n28b >> 18); b[5] = (uint8_t)(n28b >> 10); b[6] = (uint8_t)(n28b >> 2);
            b[7] = (uint8_t)((uint8_t)(n28b << 6) | (uint8_t)(g >> 10));
            b[8] = (uint8_t)(g >> 2);
            b[9] = (uint8_t)((uint8_t)(g << 6) | (1u << 3));
            return 0;
        }
    }
    orc_pack_text(msg, b);
    return 1;
}

void orc_encode174(const uint8_t *payload, uint8_t *bits) {
    uint8_t a91[12];
    memcpy(a91, payload, 10);
    a91[9] &= 0xF8; a91[10] = 0; a91[11] = 0;
    const uint16_t crc = orc_crc14(a91, 82);
    a91[9] |= (uint8_t)(crc >> 11);
    a91[10] = (uint8_t)(crc >> 3);
    a91[11] = (uint8_t)(crc << 5);
    for (int k = 0; k < FT8T_K; ++k) bits[k] = (a91[k >> 3] >> (7 - (k & 7))) & 1;
    for (int r = 0; r < FT8T_M; ++r) {
        int acc = 0;
        for (int k = 0; k < FT8T_K; ++k) acc ^= bits[k] & ((kFt8tGen[r][k >> 3] >> (7 - (k & 7))) & 1);
        bits[FT8T_K + r] = (uint8_t)acc;
    }
}

void orc_encode_tones_ft4(const uint8_t *payload, uint8_t *tones) { /* ref: ft4_encode, encode.c:126-195; 105 tones */
    uint8_t scrambled[10], bits[FT8T_N];
    for (int k = 0; k < 10; ++k) scrambled[k] = payload[k] ^ kFt4tXor[k];
    orc_encode174(scrambled, bits);
    int k = 0;
    for (int s = 0; s < 105; ++s) {
        if (s == 0 || s == 104) tones[s] = 0; /* ramp symbols */
        else if (s < 5) tones[s] = kFt4tCostas[0][s - 1];
        else if (s >= 34 && s < 38) tones[s] = kFt4tCostas[1][s - 34];
        else if (s >= 67 && s < 71) tones[s] = kFt4tCostas[2][s - 67];
        else if (s >= 100) tones[s] = kFt4tCostas[3][s - 100];
        else { tones[s] = kFt4tGray[(bits[k] << 1) | bits[k + 1]]; k += 2; }
    }
}

void orc_encode_tones(const uint8_t *payload, uint8_t *tones) { /* ref: ft8_encode, encode.c:66-125 */
    uint8_t bits[FT8T_N];
    orc_encode174(payload, bits);
    int k = 0;
    for (int s = 0; s < 79; ++s) {
        if (s < 7) tones[s] = kFt8tCostas[s];
        else if (s >= 36 && s < 43) tones[s] = kFt8tCostas[s - 36];
        else if (s >= 72) tones[s] = kFt8tCostas[s - 72];
        else { tones[s] = kFt8tGray[(bits[k] << 2) | (bits[k + 1] << 1) | bits[k + 2]]; k += 3; }
    }
}
