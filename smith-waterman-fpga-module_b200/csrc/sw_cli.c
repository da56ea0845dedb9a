/*
 * sw_cli.c -- command-line front end, the B200 counterpart of the reference host program
 * `main_test -q <query> -l <library> -t <timeout>` (main_test.c:231-279, 528).
 *
 *   sw_b200_cli -q query.fa -l library.fa [-t seconds] [-o out.txt] [-R score.txt]
 *               [-m match] [-x mismatch] [-g gap_open] [-e gap_extend] [-w score_width] [-G ngpus]
 *               [-T min_score]
 *
 * Without -o / -R it prints, like main_test, "result: %d, biased: %d" for every pair
 * (biased = score + 2048, the RTL's ZERO offset).  -T scores in hit-list mode (sw_set_hits) and prints
 * those lines only for the pairs scoring at least min_score; -o / -R list every subject, so they do
 * not combine with it.
 */
#include "../../include/sw_b200.h"

#include <getopt.h>
#include <stdlib.h>
#include <string.h>

static void usage(const char *n)
{
    fprintf(stderr, "Usage: %s -q <query.fa> -l <library.fa> [-t timeout_s] [-o out.txt] [-R score.txt]\n"
                    "          [-m match] [-x mismatch] [-g gap_open] [-e gap_extend] [-w score_width] [-G ngpus]\n"
                    "          [-T min_score]\n", n);
}

int main(int argc, char **argv)
{
    const char *qf = NULL, *lf = NULL, *of = NULL, *rf = NULL;
    int timeout_s = 10, ngpus = 1, opt, rc, i, min_score = 0;
    sw_params_t p;
    sw_handle_t *h = NULL;
    sw_seqset_t *q = NULL, *db = NULL;
    int32_t *scores = NULL, *hscore = NULL;
    uint32_t *hrow = NULL;
    uint64_t *hindex = NULL;
    size_t nhits = 0;
    int gpu_ids[64];
    static struct option lo[] = {{"timeout", required_argument, 0, 't'}, {"query", required_argument, 0, 'q'},
                                 {"library", required_argument, 0, 'l'}, {"help", no_argument, 0, 'h'}, {0, 0, 0, 0}};
    sw_default_params(&p);
    while ((opt = getopt_long(argc, argv, "ht:q:l:o:R:m:x:g:e:w:G:T:", lo, NULL)) >= 0) {
        switch (opt) {
            case 'q': qf = optarg; break;
            case 'l': lf = optarg; break;
            case 't': timeout_s = (int)strtoul(optarg, NULL, 0); break;
            case 'o': of = optarg; break;
            case 'R': rf = optarg; break;
            case 'm': p.match = (int16_t)atoi(optarg); break;
            case 'x': p.mismatch = (int16_t)atoi(optarg); break;
            case 'g': p.gap_open = (int16_t)atoi(optarg); break;
            case 'e': p.gap_extend = (int16_t)atoi(optarg); break;
            case 'w': p.score_width = atoi(optarg); break;
            case 'G': ngpus = atoi(optarg); break;
            case 'T': min_score = atoi(optarg); break;
            case 'h': usage(argv[0]); return 0;
            default: usage(argv[0]); return -1;
        }
    }
    if (!qf || !lf) { printf("Input files missing\n"); usage(argv[0]); return -1; }
    if (min_score < 0 || (min_score > 0 && (of || rf))) {
        printf("-T takes a score >= 1 and prints hits only: it does not combine with -o / -R\n");
        usage(argv[0]);
        return -1;
    }
    if (ngpus < 1 || ngpus > 64) ngpus = 1;
    for (i = 0; i < ngpus; ++i) gpu_ids[i] = i;

    if ((rc = sw_read_fasta(qf, &q)) != SW_OK) { printf("Query file error! (%s)\n", sw_strerror(rc)); return -1; }
    if ((rc = sw_read_fasta(lf, &db)) != SW_OK) { printf("Database file error! (%s)\n", sw_strerror(rc)); return -1; }
    if ((rc = sw_init(&h, &p, gpu_ids, ngpus)) != SW_OK) { printf("sw_init: %s\n", sw_strerror(rc)); return -1; }
    if (min_score > 0) {
        /* a GPU's list never needs more entries than pairs */
        size_t max_hits = q->n * db->n;
        if (max_hits > ((size_t)1 << 26)) max_hits = (size_t)1 << 26;
        if ((rc = sw_set_hits(h, min_score, max_hits ? max_hits : 1)) != SW_OK) goto fail;
    }
    if ((rc = sw_set_queries(h, q->packed, q->len, q->off, (int)q->n)) != SW_OK) goto fail;
    if ((rc = sw_score_batch(h, db->packed, db->len, db->off, NULL, db->n)) != SW_OK) goto fail;
    if (min_score > 0) {
        rc = sw_fetch_hits(h, NULL, NULL, NULL, 0, &nhits, timeout_s * 1000);       /* size query */
        if (rc == SW_ECAPACITY) {
            hrow = (uint32_t *)malloc(nhits * sizeof *hrow);
            hindex = (uint64_t *)malloc(nhits * sizeof *hindex);
            hscore = (int32_t *)malloc(nhits * sizeof *hscore);
            if (!hrow || !hindex || !hscore) { rc = SW_ENOMEM; goto fail; }
            rc = sw_fetch_hits(h, hrow, hindex, hscore, nhits, &nhits, timeout_s * 1000);
        }
        if (rc != SW_OK) goto fail;
        for (i = 0; (size_t)i < nhits; ++i)
            printf("%s x %s result: %d, biased: %d(0x%04x)\n", q->name[hrow[i]], db->name[hindex[i]],
                   (int)hscore[i], (int)hscore[i] + 2048, (unsigned)(hscore[i] + 2048));
        free(hrow); free(hindex); free(hscore); sw_destroy(h); sw_seqset_free(q); sw_seqset_free(db);
        return 0;
    }
    scores = (int32_t *)calloc(q->n * db->n + 1, sizeof(int32_t));
    if (!scores) { rc = SW_ENOMEM; goto fail; }
    if ((rc = sw_fetch(h, scores, q->n * db->n, timeout_s * 1000)) != SW_OK) goto fail;

    if (of) {
        FILE *f = fopen(of, "w");
        if (!f) { rc = SW_EIO; goto fail; }
        rc = sw_write_out_txt(f, db, scores, NULL);
        fclose(f);
        if (rc != SW_OK) goto fail;
    }
    if (rf) {
        FILE *f = fopen(rf, "w");
        if (!f) { rc = SW_EIO; goto fail; }
        rc = sw_write_ssearch_R(f, qf, lf, q, db, scores);
        fclose(f);
        if (rc != SW_OK) goto fail;
    }
    if (!of && !rf) {
        size_t a, b;
        for (a = 0; a < q->n; ++a)
            for (b = 0; b < db->n; ++b)
                printf("%s x %s result: %d, biased: %d(0x%04x)\n", q->name[a], db->name[b],
                       (int)scores[a * db->n + b], (int)scores[a * db->n + b] + 2048,
                       (unsigned)(scores[a * db->n + b] + 2048));
    }
    free(scores); sw_destroy(h); sw_seqset_free(q); sw_seqset_free(db);
    return 0;
fail:
    printf("error: %s", sw_strerror(rc));
    if (rc == SW_ECUDA) printf(" [%s]", sw_last_cuda_error_string(h));
    printf("\n");
    free(scores); free(hrow); free(hindex); free(hscore); sw_destroy(h); sw_seqset_free(q); sw_seqset_free(db);
    return -1;
}
