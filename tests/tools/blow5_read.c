/* blow5_read.c -- test driver of cli/blow5.c: `blow5_read FILE [READ_ID...]` reads every record in file order, or
 * the given read ids through the index, and writes per record to stdout
 *   uint32 id_len | id | uint64 n | double digitisation, offset, range | int16 samples[n]
 * and the experiment_type of read groups 0 and 1 to stderr. Exit codes: 1 open, 2 index, 3 fetch, 4 decode,
 * 5 read error. */
#include <stdlib.h>
#include <string.h>

#include "blow5.h"

static void put(const blow5_rec_t *r) {
    const uint32_t l = (uint32_t)strlen(r->read_id);
    fwrite(&l, 4, 1, stdout);
    fwrite(r->read_id, 1, l, stdout);
    fwrite(&r->len_raw_signal, 8, 1, stdout);
    fwrite(&r->digitisation, 8, 1, stdout);
    fwrite(&r->offset, 8, 1, stdout);
    fwrite(&r->range, 8, 1, stdout);
    fwrite(r->raw_signal, 2, (size_t)r->len_raw_signal, stdout);
}

int main(int argc, char **argv) {
    blow5_file_t *f = argc > 1 ? blow5_open(argv[1]) : NULL;
    if (!f) return 1;
    for (uint32_t g = 0; g < 2; g++) {
        const char *v = blow5_hdr_get(f, "experiment_type", g);
        fprintf(stderr, "experiment_type[%u]=%s\n", g, v ? v : "(none)");
    }
    blow5_rec_t *rec = NULL;
    int rc = 0;
    if (argc > 2) {
        if (blow5_idx_load(f) < 0) rc = 2;
        for (int i = 2; i < argc && !rc; i++) {
            if (blow5_get(f, argv[i], &rec) < 0) rc = 3;
            else put(rec);
        }
    } else {
        char *mem;
        size_t n;
        int got;
        while (!rc && (got = blow5_next_bytes(f, &mem, &n)) == 0) {
            if (blow5_decode(f, &mem, &n, &rec) < 0) rc = 4;
            else put(rec);
        }
        if (!rc && got != BLOW5_EOF) rc = 5;
    }
    blow5_rec_free(rec);
    blow5_close(f);
    return rc;
}
