/*
 * TEST INFRASTRUCTURE -- counts per index row (bulk locus mode) by the C restatement of the bulk loop, for checking
 * full-size device results bit for bit.  It reuses the bucket hash of oracle/te_oracle_c.c (included, unchanged) and
 * runs the same loop with two additions (tests/locus_oracle.py restates them in Python):
 *   - a unit whose hit rows include a gene, TE or snRNA type adds 1 to every row it hits, once per row;
 *   - strand (optional): the bulk --strand rule of oracle/te_oracle_ext.py, a feature on '+' / '-' is a candidate only
 *     for units whose first record is on that strand.
 * Per-thread counters, summed.  Built by tests/locus_oracle.py into a temporary directory.
 */
#include "../oracle/te_oracle_c.c"

#define LO_F_REVERSE 8u

typedef struct {
    const teo_index* ix;
    int paired, qual;
    int64_t u0, u1;
    const int32_t *start, *end;
    const uint16_t* chrom;
    const uint8_t *mapq, *flag, *strand;
    int64_t *counts, *loci;
    int64_t stats[6];                        /* assigned, lowq, badchrom, qcfail, crash_enhancer, crash_name */
    uint32_t* estamp;
} lo_job;

static void* lo_worker(void* arg) {
    lo_job* j = (lo_job*)arg;
    const teo_index* ix = j->ix;
    const int bs = ix->bs;
    uint32_t tick = 0;
    int32_t hits[4096];
    for (int64_t u = j->u0; u < j->u1; ++u) {
        int64_t c, loc1, loc2, r1;
        if (j->paired) {
            r1 = 2 * u;
            const int64_t r2 = 2 * u + 1;
            if (j->flag[r1] & F_REJECT) { j->stats[3]++; continue; }            /* te_count.py:81 */
            if (j->flag[r2] & F_REJECT) { j->stats[3]++; continue; }            /* :84 */
            if ((int)j->mapq[r1] < j->qual) { j->stats[1]++; continue; }        /* :88 */
            if (j->flag[r1] & F_NAME_MISMATCH) { j->stats[5]++; continue; }     /* :92-94 */
            c = j->chrom[r1]; loc1 = j->start[r1]; loc2 = j->start[r2];         /* :96-98 */
        } else {
            r1 = u;
            if (j->flag[u] & F_REJECT) { j->stats[3]++; continue; }             /* :204 */
            if ((int)j->mapq[u] < j->qual) { j->stats[1]++; continue; }         /* :208 */
            c = j->chrom[u]; loc1 = j->start[u]; loc2 = j->end[u];              /* :212-214 */
        }
        if (c >= ix->n_chrom || !ix->has[c]) { j->stats[2]++; continue; }       /* :100 / :216 */
        const int64_t b1 = floordiv64(loc1 - 1, bs), b2 = floordiv64(loc2 + 1, bs);
        if (++tick == 0) { memset(j->estamp, 0, (size_t)ix->n_ensg * 4); tick = 1; }
        int nh = 0, overflow = 0;
        unsigned types = 0;
        int64_t ta = 0, ea = 0, tb = 0, eb = 0;                                 /* union of the two buckets: merge walk */
        if (b1 >= 0 && b1 < ix->n_buck[c]) { ta = ix->list_off[ix->buck_off[c] + b1]; ea = ix->list_off[ix->buck_off[c] + b1 + 1]; }
        if (b2 != b1 && b2 >= 0 && b2 < ix->n_buck[c]) { tb = ix->list_off[ix->buck_off[c] + b2]; eb = ix->list_off[ix->buck_off[c] + b2 + 1]; }
        while (ta < ea || tb < eb) {
            int32_t i;
            if (tb >= eb || (ta < ea && ix->ids[ta] <= ix->ids[tb])) {
                i = ix->ids[ta++];
                if (tb < eb && ix->ids[tb] == i) ++tb;
            } else i = ix->ids[tb++];
            if (j->strand) {
                const unsigned fs = j->strand[i], us = (j->flag[r1] & LO_F_REVERSE) ? 1u : 0u;
                if (fs <= 1u && fs != us) continue;
            }
            const int a = loc1 >= ix->L[i] && loc1 + 1 <= ix->R[i];            /* :122 */
            const int bq = loc2 - 1 >= ix->L[i] && loc2 <= ix->R[i];           /* :125 */
            if (a || bq) {
                types |= 1u << ix->type[i];
                if (nh < 4096) hits[nh++] = i; else overflow = 1;
            }
        }
        if (!nh) continue;                                                      /* :128 */
        j->stats[0]++;                                                          /* :149 */
        if (overflow) abort();
        if (!(types & ((1u << T_GENE) | (1u << T_TE) | (1u << T_SNRNA)))) {
            if (types & (1u << T_ENH)) j->stats[4]++;
            continue;
        }
        for (int h = 0; h < nh; ++h) {                                          /* one per distinct ensg */
            const int32_t e = ix->ensg[hits[h]];
            if (j->estamp[e] == tick) continue;
            j->estamp[e] = tick;
            j->counts[e]++;
        }
        for (int h = 0; h < nh; ++h) j->loci[hits[h]]++;                        /* the merge walk lists each row once */
    }
    return 0;
}

/* counts[n_ensg], stats[7] (include/tecount.h order, as teo_bulk_count), loci[n_feat] in linearData order.
 * strand: feature strand codes for the bulk --strand rule, or NULL.  At most 32 threads. */
int lo_bulk_count_loci(void* index, int paired, int qual, int64_t n_rec, const int32_t* start, const int32_t* end,
                       const uint16_t* chrom, const uint8_t* mapq, const uint8_t* flag, const uint8_t* strand,
                       int64_t* counts, int64_t* stats, int64_t* loci, int n_threads) {
    const teo_index* ix = (const teo_index*)index;
    const int64_t n_units = paired ? n_rec / 2 : n_rec;
    if (n_threads < 1) n_threads = 1;
    if (n_threads > 32) n_threads = 32;
    lo_job* jobs = (lo_job*)calloc((size_t)n_threads, sizeof(lo_job));
    pthread_t* th = (pthread_t*)calloc((size_t)n_threads, sizeof(pthread_t));
    for (int t = 0; t < n_threads; ++t) {
        lo_job* j = &jobs[t];
        j->ix = ix; j->paired = paired; j->qual = qual;
        j->u0 = n_units * t / n_threads; j->u1 = n_units * (t + 1) / n_threads;
        j->start = start; j->end = end; j->chrom = chrom; j->mapq = mapq; j->flag = flag; j->strand = strand;
        j->counts = (int64_t*)calloc((size_t)ix->n_ensg + 1, 8);
        j->loci = (int64_t*)calloc((size_t)ix->n_feat + 1, 8);
        j->estamp = (uint32_t*)calloc((size_t)ix->n_ensg + 1, 4);
        pthread_create(&th[t], 0, lo_worker, j);
    }
    memset(counts, 0, (size_t)ix->n_ensg * 8);
    memset(loci, 0, (size_t)ix->n_feat * 8);
    memset(stats, 0, 7 * 8);
    stats[0] = n_units;
    for (int t = 0; t < n_threads; ++t) {
        pthread_join(th[t], 0);
        for (int e = 0; e < ix->n_ensg; ++e) counts[e] += jobs[t].counts[e];
        for (int64_t f = 0; f < ix->n_feat; ++f) loci[f] += jobs[t].loci[f];
        for (int k = 0; k < 6; ++k) stats[1 + k] += jobs[t].stats[k];
        free(jobs[t].counts); free(jobs[t].loci); free(jobs[t].estamp);
    }
    free(jobs); free(th);
    return 0;
}
