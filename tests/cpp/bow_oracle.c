/* TEST INFRASTRUCTURE ONLY -- the CPU oracle of the BoW database (sfe_bowdb_*).  Never linked by the product path; the
 * tests and tools/bow_bench.py compile it with tests/bow_oracle.py (gcc -O2 -ffp-contract=off into a temporary directory)
 * and use it as the checker and the reported host baseline.
 *
 * Dependency-free C restatement of DBoW2's L1 scoring (thirdparty/DBoW2/DBoW2: L1Scoring::score in GeneralScoring.cpp,
 * TemplatedDatabase::queryL1).  Vectors are BowVectors: ids ascending and unique, IEEE double values.
 * orc_bow_score_l1: the sum of fabs(v - w) - fabs(v) - fabs(w) over the common words from 0.0 in ascending word order,
 * returned as -sum / 2.0 (-0.0 when no word is shared).
 * orc_bow_query_l1: the database as its inverted file (if_off[n_words + 1]; row w = the entries holding word w in ascending
 * entry id, with their values).  For each query word in ascending order and each entry e of its row with
 * (e < max_id || max_id == -1), value = fabs(q - d) - fabs(q) - fabs(d) starts entry e's sum or is added to it; the entries
 * that share a word are sorted by that raw sum, cut to max_results when max_results > 0 and scored -sum / 2.0.
 * T8 (canonical, next to T1-T7 of oracle/orb_oracle.h): std::sort on DBoW2's Result compares scores only, so the order of
 * equal raw sums is unspecified in the reference; here equal raw sums are ordered by ascending entry id, and the cut
 * follows that order.
 * Writes at most cap results, returns how many.  dense (optional, n_entries): the score of the query against every entry
 * whatever max_id, -0.0 where no word is shared. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

double orc_bow_score_l1(const int32_t *a_ids, const double *a_v, int na, const int32_t *b_ids, const double *b_v, int nb);
int orc_bow_query_l1(const int64_t *if_off, const int32_t *if_entry, const double *if_val, int n_words, int n_entries,
                     const int32_t *q_ids, const double *q_v, int nq, int max_id, int max_results, int32_t *out_entry,
                     double *out_score, int cap, double *dense);

double orc_bow_score_l1(const int32_t *a_ids, const double *a_v, int na, const int32_t *b_ids, const double *b_v, int nb) {
    double score = 0;
    int i = 0, j = 0;
    while (i < na && j < nb) {
        if (a_ids[i] == b_ids[j]) {
            const double vi = a_v[i], wi = b_v[j];
            score += fabs(vi - wi) - fabs(vi) - fabs(wi);
            ++i;
            ++j;
        } else if (a_ids[i] < b_ids[j]) {
            ++i;
        } else {
            ++j;
        }
    }
    score = -score / 2.0;
    return score;
}

typedef struct {
    int32_t id;
    double score;
} orc_bow_result;

/* T8: equal raw sums keep ascending entry id (std::sort compares the scores only) */
static int bow_result_cmp(const void *pa, const void *pb) {
    const orc_bow_result *a = (const orc_bow_result *)pa, *b = (const orc_bow_result *)pb;
    if (a->score < b->score) return -1;
    if (b->score < a->score) return 1;
    return a->id < b->id ? -1 : (a->id > b->id ? 1 : 0);
}

int orc_bow_query_l1(const int64_t *if_off, const int32_t *if_entry, const double *if_val, int n_words, int n_entries,
                     const int32_t *q_ids, const double *q_v, int nq, int max_id, int max_results, int32_t *out_entry,
                     double *out_score, int cap, double *dense) {
    double *pairs = (double *)calloc((size_t)n_entries + 1, sizeof(double));
    uint8_t *present = (uint8_t *)calloc((size_t)n_entries + 1, 1);
    int32_t *order = (int32_t *)malloc(((size_t)n_entries + 1) * sizeof(int32_t));
    int touched = 0;
    for (int k = 0; k < nq; k++) {
        const int w = q_ids[k];
        if (w < 0 || w >= n_words) continue;
        const double qvalue = q_v[k];
        for (int64_t r = if_off[w]; r < if_off[w + 1]; r++) {
            const int e = if_entry[r];
            if (!dense && !(e < max_id || max_id == -1)) continue;  /* dense: every entry, max_id applies to ret */
            const double dvalue = if_val[r];
            const double value = fabs(qvalue - dvalue) - fabs(qvalue) - fabs(dvalue);
            if (present[e]) {
                pairs[e] += value;
            } else {
                pairs[e] = value;
                present[e] = 1;
                order[touched++] = e;
            }
        }
    }
    if (dense) {
        for (int e = 0; e < n_entries; e++) dense[e] = -0.0;
        for (int t = 0; t < touched; t++) dense[order[t]] = -pairs[order[t]] / 2.0;
    }
    orc_bow_result *ret = (orc_bow_result *)malloc(((size_t)touched + 1) * sizeof(orc_bow_result));
    int n = 0;
    for (int t = 0; t < touched; t++) {
        const int e = order[t];
        if (e < max_id || max_id == -1) {
            ret[n].id = e;
            ret[n].score = pairs[e];
            n++;
        }
    }
    qsort(ret, (size_t)n, sizeof(orc_bow_result), bow_result_cmp);
    if (max_results > 0 && n > max_results) n = max_results;
    if (n > cap) n = cap;
    for (int t = 0; t < n; t++) {
        out_entry[t] = ret[t].id;
        out_score[t] = -ret[t].score / 2.0;
    }
    free(ret); free(order); free(present); free(pairs);
    return n;
}
