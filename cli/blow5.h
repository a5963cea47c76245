/* blow5.h -- the part of the SLOW5 / BLOW5 format (slow5lib file format 0.2.0 and 1.0.0) that `sigtk` reads.
 *
 * SLOW5 (ASCII, *.slow5) and BLOW5 (binary, *.blow5) files, told apart by the name's extension as slow5lib does:
 * header attributes per read group, records read in file order or by read id, record compression none or zlib,
 * signal compression none or svb-zd. Files with zstd records or ex-zd signals are refused when opened. Only the primary columns the raw-signal commands use (read_id,
 * digitisation, offset, range, raw_signal) are parsed; auxiliary columns are skipped.
 *
 * Record bytes returned by blow5_next_bytes are what the file stores (BLOW5: possibly compressed); blow5_inflate
 * and blow5_decode turn them into a record and are thread safe for different records. */
#ifndef SIGTK_BLOW5_H
#define SIGTK_BLOW5_H

#include <stddef.h>
#include <stdint.h>
#include <stdio.h>

enum { BLOW5_PRESS_NONE = 0, BLOW5_PRESS_ZLIB = 1 };   /* record compression */
enum { BLOW5_SIGNAL_NONE = 0, BLOW5_SIGNAL_SVB_ZD = 1 }; /* signal compression */

#define BLOW5_EOF (-1)       /* no more records */
#define BLOW5_ERR_IO (-2)    /* read error or truncated file */
#define BLOW5_ERR_PRESS (-3) /* record or signal cannot be decompressed */
#define BLOW5_ERR_PARSE (-4) /* malformed record */
#define BLOW5_ERR_NOID (-5)  /* read id not in the file */

typedef struct {
    char *name;
    char **val; /* one per read group; NULL where the group has no value ('.') */
} blow5_attr_t;

typedef struct {
    char *read_id;
    uint64_t off;   /* file offset of the record (BLOW5: of its size field) */
} blow5_idx_t;

typedef struct {
    FILE *fp;
    char *path;
    int ascii;
    int record_press;
    int signal_press;
    uint32_t num_read_groups;
    blow5_attr_t *attr;
    int n_attr;
    blow5_idx_t *idx; /* sorted by read id; built by blow5_idx_load */
    uint64_t n_idx;
} blow5_file_t;

typedef struct {
    char *read_id;
    double digitisation, offset, range;
    uint64_t len_raw_signal;
    int16_t *raw_signal;
} blow5_rec_t;

/* the primary columns of an uncompressed BLOW5 record, pointing into its bytes */
typedef struct {
    const char *read_id;      /* not NUL terminated */
    size_t read_id_len;
    double digitisation, offset, range;
    const uint8_t *signal;    /* raw_signal as stored: int16 samples, or an svb-zd stream */
    uint64_t signal_bytes;
    uint64_t len_raw_signal;  /* samples (for svb-zd: the count in the stream's header) */
} blow5_view_t;

/* opens and reads the header; NULL (with a message on stderr) when the file cannot be read or is not supported */
blow5_file_t *blow5_open(const char *path);
void blow5_close(blow5_file_t *f);

/* value of header attribute `attr` for read group `rg`, or NULL */
const char *blow5_hdr_get(const blow5_file_t *f, const char *attr, uint32_t rg);

/* the next record as stored (malloc'd into *mem, *bytes long); 0, BLOW5_EOF or another BLOW5_ERR_* */
int blow5_next_bytes(blow5_file_t *f, char **mem, size_t *bytes);

/* BLOW5: undoes the record compression of *mem in place (it may be replaced); 0 or BLOW5_ERR_PRESS */
int blow5_inflate(const blow5_file_t *f, char **mem, size_t *bytes);

/* BLOW5: the primary columns of a record blow5_inflate has decompressed; 0 or BLOW5_ERR_PARSE */
int blow5_view(const blow5_file_t *f, const char *mem, size_t bytes, blow5_view_t *v);

/* a stored record -> *rec (allocated on first use, reused after); frees *mem. 0 or BLOW5_ERR_* */
int blow5_decode(const blow5_file_t *f, char **mem, size_t *bytes, blow5_rec_t **rec);
void blow5_rec_free(blow5_rec_t *rec);

/* random access by read id: the index is built by reading the file once */
int blow5_idx_load(blow5_file_t *f);
int blow5_get(blow5_file_t *f, const char *read_id, blow5_rec_t **rec);
void blow5_idx_unload(blow5_file_t *f);

/* svb-zd stream (uint32 count | key bytes | data bytes) -> count samples into out (cap samples);
 * the count, or -1 when the stream is malformed */
int64_t blow5_svbzd_decode(const uint8_t *in, uint64_t n_bytes, int16_t *out, uint64_t cap);

#endif
