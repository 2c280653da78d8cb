/* tests/support/ap_oracle.c -- CPU restatement of a-priori (AP) decoding of "CQ ??? ???" after belief propagation and OSD, the
 * definition of DESIGN.md section 2.4.3.  TEST INFRASTRUCTURE ONLY: compiled by tests/test_ap.py together with the unchanged sources of
 * the oracle library (oracle/ft8_oracle*.c, same flags as oracle/Makefile).  It includes tests/support/osd_oracle.c, whose _osd forms
 * it extends, and composes the oracle's public orc_bp_decode, which tests/test_gpu_bp.py already pins.  The reference has no AP, so
 * orc_ap is pinned by tests/test_ap.py against an independent numpy implementation of the definition's other steps; the GPU kernel is
 * then held to it byte for byte (tests/test_gpu_ap.py).
 *
 * orc_ap: one candidate's normalised LLRs, BP iteration limit, hard-distance cap, protocol as in orc_waterfall_t (0 = FT4).
 * -1 = not attempted (a non-finite LLR), 0 = rejected, 1 = accepted; whenever it is attempted, cw174 = BP's final word and *hard its
 * distance from the hard decision of the unforced LLRs.
 * The _ap forms of orc_decode_osd, orc_decode_waterfall_osd and orc_subsystem_osd equal them with ap_on = 0; ap_out: 0 not attempted,
 * 1 rejected, 2 decoded by AP. */
#include "osd_oracle.c"

int orc_ap_hypothesis(int protocol, uint8_t *mask174, uint8_t *val174);
int orc_ap(const float *llr174, int max_iters, int max_hard, int protocol, uint8_t *cw174, int *hard);
int orc_decode_ap(const orc_waterfall_t *wf, const orc_candidate_t *c, int max_iters, int osd_order, int osd_max_hard, int ap_on, int ap_max_hard,
                  orc_message_t *msg, orc_status_t *st, float *llr_out, uint8_t *plain_out, uint8_t *osd_out, int *osd_hard_out, uint8_t *ap_out,
                  int *ap_hard_out);
int orc_decode_waterfall_ap(const orc_waterfall_t *wf, int max_candidates, int max_messages, int min_score, int ldpc_iters, int osd_order,
                            int osd_max_hard, int ap_on, int ap_max_hard, orc_result_t *results, orc_slot_report_t *rep, orc_candidate_t *cand_out);
int orc_subsystem_ap(const float *i_s, const float *q_s, int max_candidates, int max_messages, int min_score, int ldpc_iters, int osd_order,
                     int osd_max_hard, int ap_on, int ap_max_hard, orc_result_t *results, orc_slot_report_t *rep, uint8_t *wf_out,
                     orc_candidate_t *cand_out);

/* the hypothesis as codeword bits: mask174[n] = 1 at the 32 known positions, val174[n] their values (FT4: scrambled) */
int orc_ap_hypothesis(int protocol, uint8_t *mask, uint8_t *val) {
    memset(mask, 0, FT8T_N);
    memset(val, 0, FT8T_N);
    for (int n = 0; n < 77; ++n) {
        if (n > 28 && n < 74) continue;
        mask[n] = 1;
        val[n] = (n == 26 || n == 76);  /* bits 0-28: c28 << 1 | r1 = 4, big-endian; bits 74-76: i3 = 1 */
        if (protocol == 0) val[n] ^= (kFt4tXor[n >> 3] >> (7 - (n & 7))) & 1;
    }
    return 32;
}

/* message bits [first, first + len) of a codeword, descrambled for FT4, big-endian */
static uint32_t ap_field(const uint8_t *cw, int protocol, int first, int len) {
    uint32_t v = 0;
    for (int n = first; n < first + len; ++n) {
        uint32_t b = cw[n];
        if (protocol == 0) b ^= (kFt4tXor[n >> 3] >> (7 - (n & 7))) & 1;
        v = (v << 1) | b;
    }
    return v;
}

int orc_ap(const float *llr, int max_iters, int max_hard, int protocol, uint8_t *cw, int *hard_out) {
    for (int n = 0; n < FT8T_N; ++n)
        if (!isfinite(llr[n])) return -1;
    uint8_t mask[FT8T_N], val[FT8T_N];
    orc_ap_hypothesis(protocol, mask, val);
    float amax = 0.0f;
    for (int n = 0; n < FT8T_N; ++n) amax = fmaxf(amax, fabsf(llr[n]));
    const float apmag = amax * 1.01f;
    float forced[FT8T_N];
    for (int n = 0; n < FT8T_N; ++n) forced[n] = mask[n] ? (val[n] ? apmag : -apmag) : llr[n];
    int errors = 0;
    orc_bp_decode(forced, max_iters, cw, &errors);
    int hard = 0, kept = 1;
    for (int n = 0; n < FT8T_N; ++n) {
        hard += cw[n] != (llr[n] > 0.0f);
        if (mask[n] && cw[n] != val[n]) kept = 0;
    }
    *hard_out = hard;
    if (errors != 0 || !kept || hard > max_hard) return 0;
    /* plausibility of "CQ call_2 [grid]": call_2 a standard callsign (n28 >= NTOK + MAX22 of unpack_callsign), R1 = 0, a locator
     * (g15 <= 32400) or none (32401) */
    const uint32_t n28b = ap_field(cw, protocol, 29, 29) >> 1, g15 = ap_field(cw, protocol, 59, 15);
    if (n28b < 2063592u + 4194304u || ap_field(cw, protocol, 58, 1) != 0 || (g15 > 32400u && g15 != 32401u)) return 0;
    orc_message_t msg;
    orc_status_t st;
    return finish_codeword(cw, protocol, &msg, &st);
}

int orc_decode_ap(const orc_waterfall_t *wf, const orc_candidate_t *c, int max_iters, int osd_order, int osd_max_hard, int ap_on, int ap_max_hard,
                  orc_message_t *msg, orc_status_t *st, float *llr_out, uint8_t *plain_out, uint8_t *osd_out, int *osd_hard_out, uint8_t *ap_out,
                  int *ap_hard_out) {
    float llr[FT8T_N];
    uint8_t plain[FT8T_N];
    if (ap_out) *ap_out = 0;
    if (ap_hard_out) *ap_hard_out = -1;
    const int ok = orc_decode_osd(wf, c, max_iters, osd_order, osd_max_hard, msg, st, llr, plain, osd_out, osd_hard_out);
    if (llr_out) memcpy(llr_out, llr, sizeof(llr));
    if (plain_out) memcpy(plain_out, plain, sizeof(plain));
    /* AP only where BP and OSD left the candidate at the parity check or the CRC (stage 1 or 2) */
    if (!ap_on || ok || (st->ldpc_errors == 0 && st->crc_extracted == st->crc_calculated)) return ok;
    uint8_t cw[FT8T_N];
    int hard = 0;
    const int acc = orc_ap(llr, max_iters, ap_max_hard, wf->protocol, cw, &hard);
    if (acc < 0) return 0;
    if (ap_out) *ap_out = (uint8_t)(acc ? 2 : 1);
    if (ap_hard_out) *ap_hard_out = hard;
    if (!acc) return 0;
    st->ldpc_errors = 0;
    finish_codeword(cw, wf->protocol, msg, st);
    if (plain_out) memcpy(plain_out, cw, sizeof(cw));
    return 1;
}

/* orc_decode_waterfall_osd with AP: the daemon's candidate loop, duplicate table and CQ filter (oracle/ft8_oracle_codec.c) */
int orc_decode_waterfall_ap(const orc_waterfall_t *wf, int max_candidates, int max_messages, int min_score, int ldpc_iters, int osd_order,
                            int osd_max_hard, int ap_on, int ap_max_hard, orc_result_t *results, orc_slot_report_t *rep, orc_candidate_t *cand_out) {
    orc_candidate_t *cand = (orc_candidate_t *)malloc(sizeof(orc_candidate_t) * (size_t)max_candidates);
    const int n_cand = orc_find_sync(wf, max_candidates, cand, min_score);
    if (cand_out) memcpy(cand_out, cand, sizeof(orc_candidate_t) * (size_t)n_cand);
    orc_message_t *msgs = (orc_message_t *)calloc((size_t)(n_cand > 0 ? n_cand : 1), sizeof(orc_message_t));
    uint8_t *ok = (uint8_t *)calloc((size_t)(n_cand > 0 ? n_cand : 1), 1);
    if (rep) memset(rep, 0, sizeof(*rep));
    for (int k = 0; k < n_cand; ++k) {
        orc_status_t st;
        if (cand[k].score < min_score) continue;
        ok[k] = (uint8_t)orc_decode_ap(wf, &cand[k], ldpc_iters, osd_order, osd_max_hard, ap_on, ap_max_hard, &msgs[k], &st, NULL, NULL, NULL, NULL,
                                       NULL, NULL);
    }
    const int n_new = orc_spots(cand, ok, msgs, n_cand, max_messages, min_score, 2 /* K_FREQ_OSR, rtlsdr_ft8d.c:1470 */, results, rep);
    if (rep) rep->n_cand = n_cand;
    free(cand); free(msgs); free(ok);
    return n_new;
}

int orc_subsystem_ap(const float *i_s, const float *q_s, int max_candidates, int max_messages, int min_score, int ldpc_iters, int osd_order,
                     int osd_max_hard, int ap_on, int ap_max_hard, orc_result_t *results, orc_slot_report_t *rep, uint8_t *wf_out,
                     orc_candidate_t *cand_out) {
    uint8_t *mag = (uint8_t *)malloc(ORC_WF_BYTES);
    orc_waterfall_daemon(i_s, q_s, mag);
    if (wf_out) memcpy(wf_out, mag, ORC_WF_BYTES);
    orc_waterfall_t wf = { 92, 92, 256, 2, 2, mag, 1024, 1 };
    const int n = orc_decode_waterfall_ap(&wf, max_candidates, max_messages, min_score, ldpc_iters, osd_order, osd_max_hard, ap_on, ap_max_hard, results,
                                          rep, cand_out);
    free(mag);
    return n;
}
