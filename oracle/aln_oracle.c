/*
 * aln_oracle.c -- CPU restatement of the step that turns an alignment region into an alignment record: CIGAR, NM, MD,
 * the strand and the leftmost position (SURVEY.md 8(f)).
 *
 * TEST INFRASTRUCTURE ONLY (same rule as ksw_oracle.c: nothing under genomicsbench_b200/ may link, import or call
 * this file).
 *
 * What it restates (bwa 0.7.17, paths relative to /root/reference/tools/bwa):
 *   bwamem.c  infer_bw            the band from the region and its local score
 *   bwamem.c  mem_reg2aln         the band-doubling loop (three tries), bns_depos, the squeeze of ONE end D, the clips
 *   bwa.c     bwa_gen_cigar2      reversal of both sequences on the reverse strand, the no-DP fast path, the band of
 *                                 ksw_global2, the NM / MD walk
 * ksw_global2 itself is global_oracle.c's restatement, which the golden vectors pin.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>

typedef struct {
    int32_t o_del, e_del, o_ins, e_ins, zdrop, end_bonus;
    int32_t match, mismatch, ambig;
    int32_t zdrop_mode;
} oracle_params;                                   /* ksw_oracle.c */

int bsw_oracle_global(const oracle_params *p, const uint8_t *query, int qlen, const uint8_t *target, int tlen,
                      int w, uint32_t *cigar, int *n_cigar);                          /* global_oracle.c */

static int infer_bw(int l1, int l2, int score, int a, int q, int r)                   /* bwamem.c: infer_bw */
{
    int w;
    if (l1 == l2 && l1 * a - score < (q + r - a * 2) * 2) return 0;      /* (q + r - (a<<1))<<1 */
    w = (int)((double)((l1 < l2 ? l1 : l2) * a - score - q) / r + 2.);
    if (w < abs(l1 - l2)) w = abs(l1 - l2);
    return w;
}

static int col_score(const oracle_params *p, int t, int q)                             /* bwa_fill_scmat */
{
    if (t >= 4 || q >= 4) return p->ambig;
    return t == q ? p->match : -p->mismatch;
}

/* bwa.c: bwa_gen_cigar2 on the (already reversed) sequences.  cigar holds l_query + rlen entries, md 4 l_query + rlen + 2
 * bytes.  Returns the score; *n_cigar, *nm, *l_md receive the counts. */
static int gen_cigar2(const oracle_params *p, int w_, const uint8_t *query, int l_query, const uint8_t *rseq, int rlen,
                      int is_rev, uint32_t *cigar, int *n_cigar, int *nm, char *md, int *l_md)
{
    int score, i, k, x, y, u, n_mm = 0, n_gap = 0, l = 0;
    const char *int2base = is_rev ? "TGCAN" : "ACGTN";
    if (l_query == rlen && w_ == 0) {                                                  /* no DP */
        cigar[0] = (uint32_t)l_query << 4;
        *n_cigar = 1;
        for (i = 0, score = 0; i < l_query; ++i) score += col_score(p, rseq[i], query[i]);
    } else {
        const int a = p->match;
        int w, max_gap, max_ins, max_del, min_w;
        max_ins = (int)((double)(((l_query + 1) >> 1) * a - p->o_ins) / p->e_ins + 1.);
        max_del = (int)((double)(((l_query + 1) >> 1) * a - p->o_del) / p->e_del + 1.);
        max_gap = max_ins > max_del ? max_ins : max_del;
        max_gap = max_gap > 1 ? max_gap : 1;
        w = (max_gap + abs(rlen - l_query) + 1) >> 1;
        w = w < w_ ? w : w_;
        min_w = abs(rlen - l_query) + 3;
        w = w > min_w ? w : min_w;
        score = bsw_oracle_global(p, query, l_query, rseq, rlen, w, cigar, n_cigar);
    }
    for (k = 0, x = y = u = 0; k < *n_cigar; ++k) {                                    /* NM and MD */
        const int op = (int)(cigar[k] & 0xf), len = (int)(cigar[k] >> 4);
        if (op == 0) {
            for (i = 0; i < len; ++i) {
                if (query[x + i] != rseq[y + i]) {
                    l += sprintf(md + l, "%d", u);
                    md[l++] = int2base[rseq[y + i] < 4 ? rseq[y + i] : 4];
                    ++n_mm; u = 0;
                } else ++u;
            }
            x += len; y += len;
        } else if (op == 2) {
            if (k > 0 && k < *n_cigar - 1) {                                           /* not the first or the last op */
                l += sprintf(md + l, "%d", u);
                md[l++] = '^';
                for (i = 0; i < len; ++i) md[l++] = int2base[rseq[y + i] < 4 ? rseq[y + i] : 4];
                u = 0; n_gap += len;
            }
            y += len;
        } else if (op == 1) { x += len; n_gap += len; }                               /* I: u is not reset */
    }
    l += sprintf(md + l, "%d", u);
    *l_md = l;
    *nm = n_mm + n_gap;
    return score;
}

/* One region of mem_reg2aln.  read = the whole read (l_query codes), rseq = bns_get_seq(rb, re) (re - rb bytes).
 * rec = {is_rev, n_cigar, NM, gscore, w}; info = {tries, exit, fast}: exit 1 score == last_sc, 2 w2 == w << 2,
 * 3 three tries, 4 score >= truesc - a; fast = 1 when the first try took the no-DP path.  cigar holds
 * (qe - qb) + (re - rb) + 2 entries, md 4 (qe - qb) + (re - rb) + 1 bytes.  Returns the MD length (no NUL), or -2 for a
 * region bwa_gen_cigar2 rejects. */
int bsw_oracle_reg2aln(const oracle_params *p, int w, int64_t l_pac, const uint8_t *read, int l_query, int64_t rb,
                       int64_t re, int qb, int qe, int truesc, int reg_w, const uint8_t *rseq_in, int64_t *pos_out,
                       int32_t *rec, uint32_t *cigar, char *md, int32_t *info)
{
    const int a = p->match;
    int i, w2, tmp, score = 0, last_sc = -(1 << 30), n_cigar = 0, nm = 0, l_md = 0, tries = 0, why = 0, is_rev, lo = 0,
        wl = 0, clip5, clip3, j;
    const int lq = qe - qb, rlen = (int)(re - rb);
    int64_t pos;
    uint8_t *q, *r;
    uint32_t *cg;
    char *mdb;
    memset(rec, 0, 5 * sizeof(int32_t));
    info[0] = info[1] = info[2] = 0;
    if (rb < 0 || re < 0) { *pos_out = -1; return 0; }                                   /* unmapped record */
    if (lq <= 0 || rb >= re || (rb < l_pac && re > l_pac)) return -2;
    is_rev = rb >= l_pac;
    q = (uint8_t *)malloc((size_t)lq + 1); r = (uint8_t *)malloc((size_t)rlen + 1);
    cg = (uint32_t *)malloc(((size_t)lq + rlen + 2) * 4); mdb = (char *)malloc(4 * (size_t)lq + rlen + 32);
    for (i = 0; i < lq; ++i) q[i] = is_rev ? read[qe - 1 - i] : read[qb + i];           /* bwa.c: reverse both */
    for (i = 0; i < rlen; ++i) r[i] = is_rev ? rseq_in[rlen - 1 - i] : rseq_in[i];
    tmp = infer_bw(lq, rlen, truesc, a, p->o_del, p->e_del);
    w2 = infer_bw(lq, rlen, truesc, a, p->o_ins, p->e_ins);
    w2 = w2 > tmp ? w2 : tmp;
    if (w2 > w) w2 = w2 < reg_w ? w2 : reg_w;
    i = 0;
    do {
        w2 = w2 < w << 2 ? w2 : w << 2;
        if (tries == 0) info[2] = lq == rlen && w2 == 0;
        score = gen_cigar2(p, w2, q, lq, r, rlen, is_rev, cg, &n_cigar, &nm, mdb, &l_md);
        wl = w2; ++tries;
        if (score == last_sc) { why = 1; break; }
        if (w2 == w << 2) { why = 2; break; }
        last_sc = score;
        w2 <<= 1;
    } while (++i < 3 && score < truesc - a);
    if (why == 0) why = i == 3 ? 3 : 4;
    pos = is_rev ? 2 * l_pac - 1 - (re - 1) : rb;                                      /* bns_depos */
    if (n_cigar > 0) {                                                                 /* squeeze ONE end: the else */
        if ((cg[0] & 0xf) == 2) { pos += cg[0] >> 4; lo = 1; }
        else if ((cg[n_cigar - 1] & 0xf) == 2) --n_cigar;
    }
    clip5 = is_rev ? l_query - qe : qb; clip3 = is_rev ? qb : l_query - qe;
    j = 0;
    if (clip5) cigar[j++] = (uint32_t)clip5 << 4 | 3;
    for (i = lo; i < n_cigar; ++i) cigar[j++] = cg[i];
    if (clip3) cigar[j++] = (uint32_t)clip3 << 4 | 3;
    memcpy(md, mdb, (size_t)l_md);
    *pos_out = pos;
    rec[0] = is_rev; rec[1] = j; rec[2] = nm; rec[3] = score; rec[4] = wl;
    info[0] = tries; info[1] = why;
    free(q); free(r); free(cg); free(mdb);
    return l_md;
}

/* bsw_oracle_reg2aln over n regions on nthreads threads.  regs: bsw_reg_in records (include/bsw.h, 72 bytes: rb re qb
 * qe score truesc w ... at the bsw_alnreg offsets, query_off at 48, ref_off at 56, l_query at 64).  cigar_room /
 * md_room: per-region start offsets into cigar / md (capacity bounds).  pos: 1 int64, rec: 5 int32, info: 3 int32,
 * l_md: 1 int32 per region.  Returns 0, or -2 if a region was rejected. */
int bsw_oracle_reg2aln_batch(const oracle_params *p, int w, int64_t l_pac, const uint8_t *regs, int64_t n,
                             const uint8_t *query, const uint8_t *ref, int64_t *pos, int32_t *rec, uint32_t *cigar,
                             const int64_t *cigar_room, char *md, const int64_t *md_room, int32_t *l_md, int32_t *info,
                             int nthreads)
{
    int bad = 0;
    int64_t k;
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads) reduction(|: bad)
    for (k = 0; k < n; ++k) {
        const uint8_t *g = regs + 72 * k;
        int64_t rb, re, qoff, roff;
        int32_t qb, qe, truesc, rw, lq;
        memcpy(&rb, g, 8); memcpy(&re, g + 8, 8); memcpy(&qb, g + 16, 4); memcpy(&qe, g + 20, 4);
        memcpy(&truesc, g + 28, 4); memcpy(&rw, g + 32, 4); memcpy(&qoff, g + 48, 8); memcpy(&roff, g + 56, 8);
        memcpy(&lq, g + 64, 4);
        l_md[k] = bsw_oracle_reg2aln(p, w, l_pac, query + qoff, lq, rb, re, qb, qe, truesc, rw,
                                     rb < 0 || re < 0 ? ref : ref + roff, pos + k, rec + 5 * k, cigar + cigar_room[k],
                                     md + md_room[k], info + 3 * k);
        if (l_md[k] < 0) bad = 1;
    }
    return bad ? -2 : 0;
}
