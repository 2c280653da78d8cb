/* tests/support/osd_oracle.c -- CPU restatement of ordered-statistics decoding (OSD) after belief propagation, the definition of
 * DESIGN.md section 2.4.1.  TEST INFRASTRUCTURE ONLY: compiled by tests/test_osd.py together with the unchanged sources of the
 * oracle library (oracle/ft8_oracle*.c, same flags as oracle/Makefile), whose public functions it composes.  The reference has no
 * OSD, so orc_osd is pinned by tests/test_osd.py against an independent numpy implementation of the definition; the GPU kernel is
 * then held to it byte for byte (tests/test_gpu_osd.py).
 *
 * orc_osd: one candidate's normalised LLRs, order 1 or 2, hard-distance cap, protocol as in orc_waterfall_t (0 = FT4).
 * -1 = not attempted (order 0 or a non-finite LLR), 0 = winner rejected, 1 = winner accepted; cw174 / *hard / *dist = the winner,
 * its hard-decision distance and its metric D whenever it is attempted.
 * The _osd forms of orc_decode, orc_decode_waterfall and orc_subsystem equal them at order 0; osd_out: 0 not attempted,
 * 1 rejected, 2 decoded by OSD. */
#include "ft8_oracle.h"
#include "ft8_tables.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

int orc_osd(const float *llr174, int order, int max_hard, int protocol, uint8_t *cw174, int *hard, uint32_t *dist);
int orc_decode_osd(const orc_waterfall_t *wf, const orc_candidate_t *c, int max_iters, int order, int max_hard, orc_message_t *msg,
                   orc_status_t *st, float *llr_out, uint8_t *plain_out, uint8_t *osd_out, int *osd_hard_out);
int orc_decode_waterfall_osd(const orc_waterfall_t *wf, int max_candidates, int max_messages, int min_score, int ldpc_iters, int osd_order,
                             int osd_max_hard, orc_result_t *results, orc_slot_report_t *rep, orc_candidate_t *cand_out);
int orc_subsystem_osd(const float *i_s, const float *q_s, int max_candidates, int max_messages, int min_score, int ldpc_iters, int osd_order,
                      int osd_max_hard, orc_result_t *results, orc_slot_report_t *rep, uint8_t *wf_out, orc_candidate_t *cand_out);

/* a12-a13 on a codeword whose parity checks hold: CRC-14 of the 91 message bits, FT4 descrambling, unpack77.  1 = msg holds the
 * message; st gets the fields the reference would have written. */
static int finish_codeword(const uint8_t *plain, int protocol, orc_message_t *msg, orc_status_t *st) {
    uint8_t a91[12];
    memset(a91, 0, sizeof(a91));
    for (int k = 0; k < FT8T_K; ++k) /* ref: pack_bits, decode.c:527-550 */
        if (plain[k]) a91[k >> 3] |= (uint8_t)(0x80 >> (k & 7));
    st->crc_extracted = (uint16_t)(((a91[9] & 7) << 11) | (a91[10] << 3) | (a91[11] >> 5)); /* ref: crc.c:40-43 */
    a91[9] &= 0xF8;
    a91[10] = 0;
    st->crc_calculated = orc_crc14(a91, 82);
    if (st->crc_extracted != st->crc_calculated) return 0;
    if (protocol == 0) /* FT4 scrambles the 77 message bits before CRC/FEC, decode.c:355-363 */
        for (int k = 0; k < 10; ++k) a91[k] ^= kFt4tXor[k];
    char text[40];
    st->unpack_status = orc_unpack77(a91, text);
    if (st->unpack_status < 0) return 0;
    memset(msg->text, 0, sizeof(msg->text));
    strncpy(msg->text, text, sizeof(msg->text) - 1);
    msg->hash = st->crc_extracted;
    return 1;
}

int orc_osd(const float *llr, int order, int max_hard, int protocol, uint8_t *cw, int *hard_out, uint32_t *dist_out) {
    if (order < 1 || order > 2) return -1;
    for (int k = 0; k < FT8T_N; ++k)
        if (!isfinite(llr[k])) return -1;
    uint8_t h[FT8T_N];
    uint32_t q[FT8T_N], mag[FT8T_N];
    int perm[FT8T_N];
    for (int k = 0; k < FT8T_N; ++k) {
        uint32_t b;
        memcpy(&b, &llr[k], 4);
        mag[k] = b & 0x7fffffffu;
        h[k] = llr[k] > 0.0f;
        q[k] = (uint32_t)(fminf(fabsf(llr[k]), 255.0f) * 256.0f);
    }
    for (int k = 0; k < FT8T_N; ++k) {  /* stable insertion sort, |llr| descending: ties keep the lower index first */
        int j = k;
        while (j > 0 && mag[perm[j - 1]] < mag[k]) { perm[j] = perm[j - 1]; --j; }
        perm[j] = k;
    }
    /* G = [I_91 | P], row k = the codeword of message bit k; Gauss-Jordan over the columns in reliability order */
    static const int R = FT8T_K;
    uint8_t g[FT8T_K][FT8T_N];
    memset(g, 0, sizeof(g));
    for (int k = 0; k < R; ++k) {
        g[k][k] = 1;
        for (int r = 0; r < FT8T_M; ++r) g[k][FT8T_K + r] = (kFt8tGen[r][k >> 3] >> (7 - (k & 7))) & 1;
    }
    uint8_t used[FT8T_K];
    int pivrow[FT8T_K], mrb[FT8T_K], rank = 0;
    memset(used, 0, sizeof(used));
    for (int p = 0; p < FT8T_N && rank < R; ++p) {
        const int col = perm[p];
        int r = 0;
        while (r < R && (used[r] || !g[r][col])) ++r;
        if (r == R) continue;  /* dependent on the columns already taken */
        used[r] = 1;
        pivrow[rank] = r;
        mrb[rank++] = col;
        for (int r2 = 0; r2 < R; ++r2)
            if (r2 != r && g[r2][col])
                for (int n = 0; n < FT8T_N; ++n) g[r2][n] ^= g[r][n];
    }
    uint8_t base[FT8T_N];
    memset(base, 0, sizeof(base));
    for (int t = 0; t < R; ++t)
        if (h[mrb[t]])
            for (int n = 0; n < FT8T_N; ++n) base[n] ^= g[pivrow[t]][n];
    const int n_pat = order == 1 ? 1 + R : 1 + R + 32 * 31 / 2;
    uint32_t best = 0xffffffffu;
    int best_idx = -1;
    for (int idx = 0; idx < n_pat; ++idx) {
        int fa = -1, fb = -1;
        if (idx >= 1 && idx <= R) fa = idx - 1;
        else if (idx > R) {  /* pair number idx - 92 of the 32 least reliable basis positions, lexicographic */
            int p = idx - 1 - R;
            fa = 0;
            while (p >= 31 - fa) { p -= 31 - fa; ++fa; }
            fb = R - 32 + fa + 1 + p;
            fa += R - 32;
        }
        uint32_t d = 0;
        for (int n = 0; n < FT8T_N; ++n) {
            uint8_t c = base[n];
            if (fa >= 0) c ^= g[pivrow[fa]][n];
            if (fb >= 0) c ^= g[pivrow[fb]][n];
            if (c != h[n]) d += q[n];
        }
        if (d < best) { best = d; best_idx = idx; }
    }
    /* the winner again, bit by bit */
    int fa = -1, fb = -1;
    if (best_idx >= 1 && best_idx <= R) fa = best_idx - 1;
    else if (best_idx > R) {
        int p = best_idx - 1 - R;
        fa = 0;
        while (p >= 31 - fa) { p -= 31 - fa; ++fa; }
        fb = R - 32 + fa + 1 + p;
        fa += R - 32;
    }
    int hard = 0;
    for (int n = 0; n < FT8T_N; ++n) {
        uint8_t c = base[n];
        if (fa >= 0) c ^= g[pivrow[fa]][n];
        if (fb >= 0) c ^= g[pivrow[fb]][n];
        cw[n] = c;
        hard += c != h[n];
    }
    *hard_out = hard;
    *dist_out = best;
    orc_message_t msg;
    orc_status_t st;
    return (hard <= max_hard && finish_codeword(cw, protocol, &msg, &st)) ? 1 : 0;
}

int orc_decode_osd(const orc_waterfall_t *wf, const orc_candidate_t *c, int max_iters, int order, int max_hard, orc_message_t *msg,
                   orc_status_t *st, float *llr_out, uint8_t *plain_out, uint8_t *osd_out, int *osd_hard_out) {
    float llr[FT8T_N];
    uint8_t plain[FT8T_N];
    if (osd_out) *osd_out = 0;
    if (osd_hard_out) *osd_hard_out = -1;
    const int ok = orc_decode(wf, c, max_iters, msg, st, llr, plain);
    if (llr_out) memcpy(llr_out, llr, sizeof(llr));
    if (plain_out) memcpy(plain_out, plain, sizeof(plain));
    /* OSD only where BP stopped at the parity check or the CRC (stage 1 or 2) */
    if (ok || (st->ldpc_errors == 0 && st->crc_extracted == st->crc_calculated)) return ok;
    uint8_t cw[FT8T_N];
    int hard = 0;
    uint32_t dist = 0;
    const int acc = orc_osd(llr, order, max_hard, wf->protocol, cw, &hard, &dist);
    if (acc < 0) return 0;
    if (osd_out) *osd_out = (uint8_t)(acc ? 2 : 1);
    if (osd_hard_out) *osd_hard_out = hard;
    if (!acc) return 0;
    st->ldpc_errors = 0;
    finish_codeword(cw, wf->protocol, msg, st);
    if (plain_out) memcpy(plain_out, cw, sizeof(cw));
    return 1;
}

/* orc_decode_waterfall with OSD: the daemon's candidate loop, duplicate table and CQ filter (oracle/ft8_oracle_codec.c) */
int orc_decode_waterfall_osd(const orc_waterfall_t *wf, int max_candidates, int max_messages, int min_score, int ldpc_iters, int osd_order,
                             int osd_max_hard, orc_result_t *results, orc_slot_report_t *rep, orc_candidate_t *cand_out) {
    orc_candidate_t *cand = (orc_candidate_t *)malloc(sizeof(orc_candidate_t) * (size_t)max_candidates);
    const int n_cand = orc_find_sync(wf, max_candidates, cand, min_score);
    if (cand_out) memcpy(cand_out, cand, sizeof(orc_candidate_t) * (size_t)n_cand);
    orc_message_t *msgs = (orc_message_t *)calloc((size_t)(n_cand > 0 ? n_cand : 1), sizeof(orc_message_t));
    uint8_t *ok = (uint8_t *)calloc((size_t)(n_cand > 0 ? n_cand : 1), 1);
    if (rep) memset(rep, 0, sizeof(*rep));
    for (int k = 0; k < n_cand; ++k) {   /* ft8_decode() is a pure function of (waterfall, candidate): decoding first changes nothing */
        orc_status_t st;
        if (cand[k].score < min_score) continue;
        ok[k] = (uint8_t)orc_decode_osd(wf, &cand[k], ldpc_iters, osd_order, osd_max_hard, &msgs[k], &st, NULL, NULL, NULL, NULL);
    }
    const int n_new = orc_spots(cand, ok, msgs, n_cand, max_messages, min_score, 2 /* K_FREQ_OSR, rtlsdr_ft8d.c:1470 */, results, rep);
    if (rep) rep->n_cand = n_cand;
    free(cand); free(msgs); free(ok);
    return n_new;
}

int orc_subsystem_osd(const float *i_s, const float *q_s, int max_candidates, int max_messages, int min_score, int ldpc_iters, int osd_order,
                      int osd_max_hard, orc_result_t *results, orc_slot_report_t *rep, uint8_t *wf_out, orc_candidate_t *cand_out) {
    uint8_t *mag = (uint8_t *)malloc(ORC_WF_BYTES);
    orc_waterfall_daemon(i_s, q_s, mag);
    if (wf_out) memcpy(wf_out, mag, ORC_WF_BYTES);
    orc_waterfall_t wf = { 92, 92, 256, 2, 2, mag, 1024, 1 };
    const int n = orc_decode_waterfall_osd(&wf, max_candidates, max_messages, min_score, ldpc_iters, osd_order, osd_max_hard, results, rep, cand_out);
    free(mag);
    return n;
}
