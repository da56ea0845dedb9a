/*
 * sw_cli.c -- command-line front end, the B200 counterpart of the reference host program
 * `main_test -q <query> -l <library> -t <timeout>` (main_test.c:231-279, 528).
 *
 *   sw_b200_cli -q query.fa -l library.fa [-t seconds] [-o out.txt] [-R score.txt]
 *               [-m match] [-x mismatch] [-g gap_open] [-e gap_extend] [-w score_width] [-G ngpus]
 *               [-T min_score] [-B] [-L] [-A]
 *
 * Without -o / -R it prints, like main_test, "result: %d, biased: %d" for every pair
 * (biased = score + 2048, the RTL's ZERO offset).  -T scores in hit-list mode (sw_set_hits) and prints
 * those lines only for the pairs scoring at least min_score; -o / -R list every subject, so they do
 * not combine with it.  -B scores in subject-best mode (sw_set_subject_best) and prints one line per
 * subject, "<subject> best <query> result: %d, second: %d" (second = -1 with one query); it combines
 * with none of -o / -R / -T.  -L (with -T or -B only) scores the library as a resident database
 * (sw_load_db, sw_score_db) and appends to each of those lines where the best alignment of the pair lies
 * (sw_locate_db), 1-based and inclusive like ssearch36 prints it: " query %u-%u subject %u-%u"
 * (0-0 for a score of 0).  -A (with -T or -B only; implies -L) also appends how it aligns (sw_align_db):
 * " cigar <CIGAR>" in SAM's text with the query as the read, "*" for a score of 0.
 */
#include "../../include/sw_b200.h"

#include <getopt.h>
#include <stdlib.h>
#include <string.h>

static void usage(const char *n)
{
    fprintf(stderr, "Usage: %s -q <query.fa> -l <library.fa> [-t timeout_s] [-o out.txt] [-R score.txt]\n"
                    "          [-m match] [-x mismatch] [-g gap_open] [-e gap_extend] [-w score_width] [-G ngpus]\n"
                    "          [-T min_score] [-B] [-L] [-A]\n", n);
}

/* " query b-e subject b-e" of a located pair: 1-based, inclusive; 0-0 for a score of 0 */
static void print_span(int32_t score, const uint32_t *c)
{
    if (score > 0) printf(" query %u-%u subject %u-%u", c[0] + 1, c[1], c[2] + 1, c[3]);
    else printf(" query 0-0 subject 0-0");
}

/* sw_locate_db; with -A sw_align_db, its CIGAR buffer sized by sum(query + subject length), which always suffices */
static int locate_pairs(sw_handle_t *h, const sw_seqset_t *q, const sw_seqset_t *db, const uint32_t *row,
                        const uint64_t *index, size_t n, int align, int32_t *score, uint32_t *coord, uint64_t **off,
                        uint32_t **ops)
{
    size_t cap = 0, count = 0, i;
    if (!align) return sw_locate_db(h, row, index, n, score, coord);
    for (i = 0; i < n; ++i) cap += (size_t)q->len[row[i]] + db->len[index[i]];
    *off = (uint64_t *)malloc((n + 1) * sizeof **off);
    *ops = (uint32_t *)malloc((cap + 1) * sizeof **ops);
    if (!*off || !*ops) return SW_ENOMEM;
    return sw_align_db(h, row, index, n, score, coord, *off, *ops, cap, &count);
}

/* " cigar <CIGAR>" of aligned pair i: SAM text of its BAM ops, "*" for none */
static void print_cigar(const uint64_t *off, const uint32_t *ops, size_t i)
{
    uint64_t k;
    printf(" cigar ");
    if (off[i] == off[i + 1]) printf("*");
    for (k = off[i]; k < off[i + 1]; ++k) printf("%u%c", ops[k] >> 4, "MIDNSHP=X"[ops[k] & 15]);
}

int main(int argc, char **argv)
{
    const char *qf = NULL, *lf = NULL, *of = NULL, *rf = NULL;
    int timeout_s = 10, ngpus = 1, opt, rc, i, min_score = 0, subject_best = 0, locate = 0, align = 0;
    sw_params_t p;
    sw_handle_t *h = NULL;
    sw_seqset_t *q = NULL, *db = NULL;
    int32_t *scores = NULL, *hscore = NULL, *bscore = NULL, *bsecond = NULL, *lscore = NULL;
    uint32_t *hrow = NULL, *brow = NULL, *lcoord = NULL, *aops = NULL;
    uint64_t *hindex = NULL, *bindex = NULL, *aoff = NULL;
    size_t nhits = 0;
    int gpu_ids[64];
    static struct option lo[] = {{"timeout", required_argument, 0, 't'}, {"query", required_argument, 0, 'q'},
                                 {"library", required_argument, 0, 'l'}, {"help", no_argument, 0, 'h'}, {0, 0, 0, 0}};
    sw_default_params(&p);
    while ((opt = getopt_long(argc, argv, "ht:q:l:o:R:m:x:g:e:w:G:T:BLA", lo, NULL)) >= 0) {
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
            case 'B': subject_best = 1; break;
            case 'L': locate = 1; break;
            case 'A': align = locate = 1; break;
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
    if (subject_best && (of || rf || min_score > 0)) {
        printf("-B prints each subject's best query only: it does not combine with -o / -R / -T\n");
        usage(argv[0]);
        return -1;
    }
    if (locate && min_score <= 0 && !subject_best) {
        printf(align ? "-A aligns the pairs -T or -B prints: it needs one of them\n"
                     : "-L locates the pairs -T or -B prints: it needs one of them\n");
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
    if (subject_best && (rc = sw_set_subject_best(h, 1)) != SW_OK) goto fail;
    if ((rc = sw_set_queries(h, q->packed, q->len, q->off, (int)q->n)) != SW_OK) goto fail;
    if (locate) {
        /* sw_locate_db reads the resident database */
        if ((rc = sw_load_db(h, db->packed, db->len, db->off, NULL, db->n)) != SW_OK) goto fail;
        if ((rc = sw_score_db(h)) != SW_OK) goto fail;
        if ((rc = sw_wait(h, timeout_s * 1000)) != SW_OK) goto fail;
    } else if ((rc = sw_score_batch(h, db->packed, db->len, db->off, NULL, db->n)) != SW_OK) goto fail;
    if (min_score > 0) {
        /* size query */
        rc = locate ? sw_fetch_db_hits(h, NULL, NULL, NULL, 0, &nhits) : sw_fetch_hits(h, NULL, NULL, NULL, 0, &nhits, timeout_s * 1000);
        if (rc == SW_ECAPACITY) {
            hrow = (uint32_t *)malloc(nhits * sizeof *hrow);
            hindex = (uint64_t *)malloc(nhits * sizeof *hindex);
            hscore = (int32_t *)malloc(nhits * sizeof *hscore);
            if (!hrow || !hindex || !hscore) { rc = SW_ENOMEM; goto fail; }
            rc = locate ? sw_fetch_db_hits(h, hrow, hindex, hscore, nhits, &nhits)
                        : sw_fetch_hits(h, hrow, hindex, hscore, nhits, &nhits, timeout_s * 1000);
        }
        if (rc != SW_OK) goto fail;
        if (locate) {
            lscore = (int32_t *)malloc((nhits + 1) * sizeof *lscore);
            lcoord = (uint32_t *)malloc((nhits + 1) * 4 * sizeof *lcoord);
            if (!lscore || !lcoord) { rc = SW_ENOMEM; goto fail; }
            if ((rc = locate_pairs(h, q, db, hrow, hindex, nhits, align, lscore, lcoord, &aoff, &aops)) != SW_OK) goto fail;
        }
        for (i = 0; (size_t)i < nhits; ++i) {
            printf("%s x %s result: %d, biased: %d(0x%04x)", q->name[hrow[i]], db->name[hindex[i]],
                   (int)hscore[i], (int)hscore[i] + 2048, (unsigned)(hscore[i] + 2048));
            if (locate) print_span(lscore[i], lcoord + 4 * (size_t)i);
            if (align) print_cigar(aoff, aops, (size_t)i);
            printf("\n");
        }
        free(hrow); free(hindex); free(hscore); free(lscore); free(lcoord); free(aoff); free(aops); sw_destroy(h); sw_seqset_free(q); sw_seqset_free(db);
        return 0;
    }
    if (subject_best) {
        bscore = (int32_t *)malloc((db->n + 1) * sizeof *bscore);
        bsecond = (int32_t *)malloc((db->n + 1) * sizeof *bsecond);
        brow = (uint32_t *)malloc((db->n + 1) * sizeof *brow);
        if (!bscore || !bsecond || !brow) { rc = SW_ENOMEM; goto fail; }
        rc = locate ? sw_fetch_db_subject_best(h, bscore, brow, bsecond, db->n)
                    : sw_fetch_subject_best(h, bscore, brow, bsecond, db->n, timeout_s * 1000);
        if (rc != SW_OK) goto fail;
        if (locate) {
            bindex = (uint64_t *)malloc((db->n + 1) * sizeof *bindex);
            lscore = (int32_t *)malloc((db->n + 1) * sizeof *lscore);
            lcoord = (uint32_t *)malloc((db->n + 1) * 4 * sizeof *lcoord);
            if (!bindex || !lscore || !lcoord) { rc = SW_ENOMEM; goto fail; }
            for (i = 0; (size_t)i < db->n; ++i) bindex[i] = (uint64_t)i;
            if ((rc = locate_pairs(h, q, db, brow, bindex, db->n, align, lscore, lcoord, &aoff, &aops)) != SW_OK) goto fail;
        }
        for (i = 0; (size_t)i < db->n; ++i) {
            printf("%s best %s result: %d, second: %d", db->name[i], q->name[brow[i]], (int)bscore[i], (int)bsecond[i]);
            if (locate) print_span(lscore[i], lcoord + 4 * (size_t)i);
            if (align) print_cigar(aoff, aops, (size_t)i);
            printf("\n");
        }
        free(bscore); free(bsecond); free(brow); free(bindex); free(lscore); free(lcoord); free(aoff); free(aops); sw_destroy(h); sw_seqset_free(q); sw_seqset_free(db);
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
    free(scores); free(hrow); free(hindex); free(hscore); free(bscore); free(bsecond); free(brow); free(bindex); free(lscore); free(lcoord);
    free(aoff); free(aops); sw_destroy(h); sw_seqset_free(q); sw_seqset_free(db);
    return -1;
}
