/* distance_oracle.c -- the CPU oracle of `mash dist` (DESIGN.md §5 "mash dist"). TEST INFRASTRUCTURE.
 *
 * Mash 2.3 CommandDistance restated on top of the screen oracle: this file includes
 * oracle/mash_screen_oracle.c whole (its .msh reader, orc_db and the long-double incomplete-beta
 * p-value) and adds, per pair, Mash's serial merge loop -- deliberately not the closed form the tests
 * also check against, and not the way the CUDA kernels work.  Built by tests/_distance_ref.py:
 *   _build/libdistoracle.so   orc_distance, orc_distance_write, orc_dist_pvalue, orc_dist_distance (+ the screen oracle)
 *   _build/distance_oracle    `distance_oracle dist [-p N] [-t] [-C] [-v P] [-d D] ref.msh q.msh [q.msh..]`,
 *                             the timed CPU baseline
 */
#include "../../oracle/mash_screen_oracle.c"

/* ------------------------------------------------------------------------ */
/* `mash dist` (DESIGN.md §5 "mash dist"): Mash 2.3 CommandDistance restated, one pair   */
/* at a time with its serial merge loop (not a closed form).                  */
/* ------------------------------------------------------------------------ */
static void dist_merge(const uint64_t *A, uint64_t na, const uint64_t *B, uint64_t nb, uint64_t s,
                       uint64_t *common, uint64_t *denom)
{
    uint64_t i = 0, j = 0, c = 0, d = 0;
    while (d < s && i < na && j < nb) {
        if (A[i] < B[j]) i++;
        else if (A[i] > B[j]) j++;
        else { i++; j++; c++; }
        d++;
    }
    if (d < s) {
        if (i < na) d += na - i;
        if (j < nb) d += nb - j;
        if (d > s) d = s;
    }
    *common = c;
    *denom = d;
}

ORC_API double orc_dist_distance(uint64_t common, uint64_t denom, uint32_t k)
{
    if (common == denom) return 0.0;
    if (common == 0) return 1.0;
    double jaccard = (double)common / denom;
    double distance = -log(2 * jaccard / (1. + jaccard)) / k;
    return distance > 1 ? 1 : distance;
}

/* P[Binomial(denom, r) >= x] with r from both genome lengths (Mash's pValue) */
ORC_API double orc_dist_pvalue(uint64_t x, uint64_t len_ref, uint64_t len_qry, uint32_t k, uint64_t denom)
{
    if (x == 0) return 1.0;
    double kmer_space = pow(4.0, (double)k);
    double px = 1. / (1. + kmer_space / len_ref);
    double py = 1. / (1. + kmer_space / len_qry);
    double r = px * py / (px + py - px * py);
    if (x > denom) return 0.0;
    return (double)betai_l((long double)x, (long double)(denom - x + 1), (long double)r);
}

typedef struct {
    const orc_db *ref, *qry;
    const uint64_t *q_idx;
    uint64_t q_begin, q_end;
    uint32_t s_p;
    uint64_t *common, *denom;
    double *pvalue;
} dist_job;

static void *dist_worker(void *arg)
{
    const dist_job *j = (const dist_job *)arg;
    const uint64_t N = j->ref->n_refs;
    for (uint64_t x = j->q_begin; x < j->q_end; x++) {
        const uint64_t q = j->q_idx ? j->q_idx[x] : x;
        const uint64_t *B = orc_db_hashes(j->qry, q), nb = orc_db_size(j->qry, q);
        for (uint64_t r = 0; r < N; r++) {
            uint64_t c, d;
            dist_merge(orc_db_hashes(j->ref, r), orc_db_size(j->ref, r), B, nb, j->s_p, &c, &d);
            j->common[x * N + r] = c;
            j->denom[x * N + r] = d;
            j->pvalue[x * N + r] = orc_dist_pvalue(c, j->ref->lengths[r], j->qry->lengths[q], j->ref->k, d);
        }
    }
    return NULL;
}

/* every pair of queries q_idx[0..n_q) (NULL: 0..n_q-1) x all references, q-major: common, denom, p-value */
ORC_API int orc_distance(const orc_db *ref, const orc_db *qry, const uint64_t *q_idx, uint64_t n_q, uint32_t s_p,
                         int threads, uint64_t *common, uint64_t *denom, double *pvalue)
{
    if (threads < 1) threads = 1;
    if ((uint64_t)threads > n_q) threads = n_q ? (int)n_q : 1;
    pthread_t *th = (pthread_t *)calloc((size_t)threads, sizeof *th);
    dist_job *jobs = (dist_job *)calloc((size_t)threads, sizeof *jobs);
    if (!th || !jobs) { free(th); free(jobs); return -1; }
    for (int t = 0; t < threads; t++) {
        dist_job j = {ref, qry, q_idx, n_q * (uint64_t)t / threads, n_q * (uint64_t)(t + 1) / threads, s_p, common, denom, pvalue};
        jobs[t] = j;
        if (t) pthread_create(&th[t], NULL, dist_worker, &jobs[t]);
    }
    dist_worker(&jobs[0]);
    for (int t = 1; t < threads; t++) pthread_join(th[t], NULL);
    free(th); free(jobs);
    return 0;
}

static void dist_name(FILE *f, const orc_db *db, uint64_t i, int comments)
{
    fputs(orc_db_name(db, i), f);
    if (comments) { fputc(':', f); fputs(orc_db_comment(db, i), f); }
}

/* `mash dist` output of one query file (queries outer, references inner) to fd; -t header when asked */
ORC_API int orc_distance_write(const orc_db *ref, const orc_db *qry, uint32_t s_p, int threads, double max_d, double max_p,
                               int table, int comments, int header, int fd)
{
    FILE *f = fdopen(dup(fd), "w");
    if (!f) return -1;
    const uint64_t N = ref->n_refs, Q = qry->n_refs, chunk = 256;
    uint64_t *common = (uint64_t *)malloc(chunk * (N + 1) * 8), *denom = (uint64_t *)malloc(chunk * (N + 1) * 8);
    double *pv = (double *)malloc(chunk * (N + 1) * 8);
    uint64_t *idx = (uint64_t *)malloc(chunk * 8);
    if (!common || !denom || !pv || !idx) { free(common); free(denom); free(pv); free(idx); fclose(f); return -1; }
    if (table && header) {
        fputs("#query", f);
        for (uint64_t r = 0; r < N; r++) { fputc('\t', f); dist_name(f, ref, r, comments); }
        fputc('\n', f);
    }
    for (uint64_t q0 = 0; q0 < Q; q0 += chunk) {
        const uint64_t n = Q - q0 < chunk ? Q - q0 : chunk;
        for (uint64_t x = 0; x < n; x++) idx[x] = q0 + x;
        orc_distance(ref, qry, idx, n, s_p, threads, common, denom, pv);
        for (uint64_t x = 0; x < n; x++) {
            if (table) dist_name(f, qry, q0 + x, comments);
            for (uint64_t r = 0; r < N; r++) {
                const uint64_t c = common[x * N + r], d = denom[x * N + r];
                const double dist = orc_dist_distance(c, d, ref->k), p = pv[x * N + r];
                const int pass = !(dist > max_d) && !(p > max_p);
                if (table) {
                    fputc('\t', f);
                    if (pass) fprintf(f, "%g", dist);
                    continue;
                }
                if (!pass) continue;
                dist_name(f, ref, r, comments);
                fputc('\t', f);
                dist_name(f, qry, q0 + x, comments);
                fprintf(f, "\t%g\t%g\t%llu/%llu\n", dist, p, (unsigned long long)c, (unsigned long long)d);
            }
            if (table) fputc('\n', f);
        }
    }
    free(common); free(denom); free(pv); free(idx);
    return fclose(f) == 0 ? 0 : -1;
}

#ifdef DIST_ORACLE_MAIN
static int dist_main(int argc, char **argv)
{
    int threads = 1, table = 0, comments = 0;
    double max_d = 1.0, max_p = 1.0;
    int a = 2;
    for (; a < argc && argv[a][0] == '-' && argv[a][1]; a++) {
        if (!strcmp(argv[a], "-t")) table = 1;
        else if (!strcmp(argv[a], "-C")) comments = 1;
        else if (a + 1 < argc && !strcmp(argv[a], "-p")) threads = atoi(argv[++a]);
        else if (a + 1 < argc && !strcmp(argv[a], "-d")) max_d = atof(argv[++a]);
        else if (a + 1 < argc && !strcmp(argv[a], "-v")) max_p = atof(argv[++a]);
        else { fprintf(stderr, "ERROR: unknown option %s\n", argv[a]); return 1; }
    }
    if (argc - a < 2) {
        fprintf(stderr, "usage: distance_oracle dist [-p N] [-t] [-C] [-v P] [-d D] <reference>.msh <query>.msh [<query>.msh] ...\n");
        return 0;
    }
    char err[512];
    double t0 = now_s();
    orc_db *ref = orc_db_load_msh(argv[a], err, sizeof err);
    if (!ref) { fprintf(stderr, "ERROR: %s\n", err); return 1; }
    double t_dist = 0;
    uint64_t pairs = 0;
    for (int i = a + 1; i < argc; i++) {
        orc_db *qry = orc_db_load_msh(argv[i], err, sizeof err);
        if (!qry) { fprintf(stderr, "ERROR: %s\n", err); orc_db_free(ref); return 1; }
        if (qry->k != ref->k || qry->seed != ref->seed) {
            fprintf(stderr, "ERROR: %s differs from the reference in k-mer size or seed\n", argv[i]);
            orc_db_free(qry); orc_db_free(ref); return 1;
        }
        const uint32_t s_p = qry->s < ref->s ? qry->s : ref->s;
        double t1 = now_s();
        fflush(stdout);
        int rc = orc_distance_write(ref, qry, s_p, threads, max_d, max_p, table, comments, i == a + 1, 1);
        t_dist += now_s() - t1;
        pairs += ref->n_refs * qry->n_refs;
        orc_db_free(qry);
        if (rc) { fprintf(stderr, "ERROR: writing the output\n"); orc_db_free(ref); return 1; }
    }
    fprintf(stderr, "[oracle timing] total %.3f s, pairs %.3f s (%llu pairs, %d threads)\n", now_s() - t0, t_dist,
            (unsigned long long)pairs, threads);
    orc_db_free(ref);
    return 0;
}

int main(int argc, char **argv)
{
    if (argc >= 2 && strcmp(argv[1], "dist") == 0) return dist_main(argc, argv);
    fprintf(stderr, "usage: distance_oracle dist [-p N] [-t] [-C] [-v P] [-d D] <reference>.msh <query>.msh [<query>.msh] ...\n");
    return argc < 2 ? 0 : 2;
}
#endif
