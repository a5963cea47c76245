/* blow5.c -- SLOW5 / BLOW5 reading for `sigtk` (see blow5.h).
 *
 * BLOW5 layout (little endian):
 *   header   "BLOW5\1" | uint8 version[3] | uint8 record_press | uint32 num_read_groups | uint8 signal_press
 *            (version >= 0.2.0) | zero padding to 64 bytes | uint32 text_len | header text (text_len bytes)
 *   records  uint64 size | size bytes, compressed as a whole by record_press; uncompressed:
 *            uint16 read_id_len | read_id | uint32 read_group | double digitisation, offset, range, sampling_rate |
 *            uint64 len_raw_signal | raw_signal | auxiliary columns
 *            where raw_signal is len_raw_signal int16 samples, or with svb-zd a stream of len_raw_signal bytes
 *   end      "5WOLB"
 * SLOW5 is the same header as text ("#slow5_version", "#num_read_groups", "@attr\tvalue per read group" lines,
 * then the column types and names) followed by one tab-separated line per record, samples separated by commas.
 * Header text lines "@name\tv0\tv1..." hold one value per read group, '.' for none. */
#define _POSIX_C_SOURCE 200809L
#define _FILE_OFFSET_BITS 64
#include "blow5.h"

#include <stdlib.h>
#include <string.h>
#include <sys/types.h>
#include <zlib.h>

#define BLOW5_HDR_FIXED 64

static int ends_with(const char *s, const char *suffix) {
    const size_t n = strlen(s), m = strlen(suffix);
    return n >= m && strcmp(s + n - m, suffix) == 0;
}

/* one header text line; "@name\tv0\tv1..." lines become attributes, "#num_read_groups\tN" sets the count */
static int hdr_line(blow5_file_t *f, char *line) {
    if (strncmp(line, "#num_read_groups\t", 17) == 0) {
        f->num_read_groups = (uint32_t)strtoul(line + 17, NULL, 10);
        return 0;
    }
    if (line[0] != '@') return 0;
    blow5_attr_t *a = (blow5_attr_t *)realloc(f->attr, (size_t)(f->n_attr + 1) * sizeof *a);
    if (!a) return -1;
    f->attr = a;
    a = &f->attr[f->n_attr++];
    a->val = (char **)calloc(f->num_read_groups ? f->num_read_groups : 1, sizeof(char *));
    char *save = NULL, *tok = strtok_r(line + 1, "\t", &save);
    a->name = strdup(tok ? tok : "");
    if (!a->val || !a->name) return -1;
    for (uint32_t g = 0; g < f->num_read_groups && (tok = strtok_r(NULL, "\t", &save)) != NULL; g++)
        if (strcmp(tok, ".") != 0 && !(a->val[g] = strdup(tok))) return -1;
    return 0;
}

static int hdr_text(blow5_file_t *f, char *text) {
    char *save = NULL;
    for (char *line = strtok_r(text, "\n", &save); line; line = strtok_r(NULL, "\n", &save))
        if (hdr_line(f, line) < 0) return -1;
    return 0;
}

static int open_binary(blow5_file_t *f) {
    uint8_t h[BLOW5_HDR_FIXED];
    uint32_t text_len;
    if (fread(h, 1, sizeof h, f->fp) != sizeof h || memcmp(h, "BLOW5\1", 6) != 0) {
        fprintf(stderr, "[blow5_open] %s is not a BLOW5 file\n", f->path);
        return -1;
    }
    f->record_press = h[9];
    memcpy(&f->num_read_groups, h + 10, 4);
    f->signal_press = (h[6] > 0 || h[7] >= 2) ? h[14] : BLOW5_SIGNAL_NONE;
    if (f->record_press != BLOW5_PRESS_NONE && f->record_press != BLOW5_PRESS_ZLIB) {
        fprintf(stderr, "[blow5_open] %s: record compression %d is not supported (none or zlib)\n", f->path,
                f->record_press);
        return -1;
    }
    if (f->signal_press != BLOW5_SIGNAL_NONE && f->signal_press != BLOW5_SIGNAL_SVB_ZD) {
        fprintf(stderr, "[blow5_open] %s: signal compression %d is not supported (none or svb-zd)\n", f->path,
                f->signal_press);
        return -1;
    }
    if (f->num_read_groups == 0 || fread(&text_len, 4, 1, f->fp) != 1) return -1;
    char *text = (char *)malloc((size_t)text_len + 1);
    if (!text) return -1;
    if (fread(text, 1, text_len, f->fp) != text_len) { free(text); return -1; }
    text[text_len] = '\0';
    const int rc = hdr_text(f, text);
    free(text);
    return rc;
}

static int open_ascii(blow5_file_t *f) {
    char *line = NULL;
    size_t cap = 0;
    ssize_t n;
    f->num_read_groups = 1;
    while ((n = getline(&line, &cap, f->fp)) > 0) {
        if (line[n - 1] == '\n') line[--n] = '\0';
        if (strncmp(line, "#read_id", 8) == 0) { free(line); return 0; } /* the last header line */
        if (line[0] != '#' && line[0] != '@') break;
        if (hdr_line(f, line) < 0) break;
    }
    free(line);
    fprintf(stderr, "[blow5_open] %s: malformed SLOW5 header\n", f->path);
    return -1;
}

blow5_file_t *blow5_open(const char *path) {
    blow5_file_t *f = (blow5_file_t *)calloc(1, sizeof *f);
    if (!f) return NULL;
    f->path = strdup(path);
    f->ascii = ends_with(path, ".slow5");
    if (!f->ascii && !ends_with(path, ".blow5")) {
        fprintf(stderr, "[blow5_open] %s: unknown file format (expected a .slow5 or .blow5 extension)\n", path);
        blow5_close(f);
        return NULL;
    }
    if (!f->path || !(f->fp = fopen(path, "rb")) || (f->ascii ? open_ascii(f) : open_binary(f)) < 0) {
        blow5_close(f);
        return NULL;
    }
    return f;
}

void blow5_close(blow5_file_t *f) {
    if (!f) return;
    blow5_idx_unload(f);
    for (int k = 0; k < f->n_attr; k++) {
        for (uint32_t g = 0; g < f->num_read_groups && f->attr[k].val; g++) free(f->attr[k].val[g]);
        free(f->attr[k].val);
        free(f->attr[k].name);
    }
    free(f->attr);
    if (f->fp) fclose(f->fp);
    free(f->path);
    free(f);
}

const char *blow5_hdr_get(const blow5_file_t *f, const char *attr, uint32_t rg) {
    if (rg >= f->num_read_groups) return NULL;
    for (int k = 0; k < f->n_attr; k++)
        if (strcmp(f->attr[k].name, attr) == 0) return f->attr[k].val[rg];
    return NULL;
}

int blow5_next_bytes(blow5_file_t *f, char **mem, size_t *bytes) {
    *mem = NULL;
    *bytes = 0;
    if (f->ascii) {
        size_t cap = 0;
        ssize_t n = getline(mem, &cap, f->fp);
        if (n <= 0) { free(*mem); *mem = NULL; return feof(f->fp) ? BLOW5_EOF : BLOW5_ERR_IO; }
        if ((*mem)[n - 1] == '\n') (*mem)[--n] = '\0';
        *bytes = (size_t)n;
        return 0;
    }
    uint8_t sz[8];
    const size_t got = fread(sz, 1, sizeof sz, f->fp);
    if (got == 5 && memcmp(sz, "5WOLB", 5) == 0) return BLOW5_EOF;
    if (got != sizeof sz) return BLOW5_ERR_IO;
    uint64_t n;
    memcpy(&n, sz, 8);
    if (n == 0 || n > ((uint64_t)1 << 40) || !(*mem = (char *)malloc((size_t)n))) return BLOW5_ERR_IO;
    if (fread(*mem, 1, (size_t)n, f->fp) != n) { free(*mem); *mem = NULL; return BLOW5_ERR_IO; }
    *bytes = (size_t)n;
    return 0;
}

int blow5_inflate(const blow5_file_t *f, char **mem, size_t *bytes) {
    if (f->ascii || f->record_press == BLOW5_PRESS_NONE) return 0;
    z_stream s;
    memset(&s, 0, sizeof s);
    if (inflateInit(&s) != Z_OK) return BLOW5_ERR_PRESS;
    size_t cap = *bytes * 4 + 4096, len = 0;
    char *out = (char *)malloc(cap);
    int rc = Z_OK;
    s.next_in = (Bytef *)*mem;
    s.avail_in = (uInt)*bytes; /* records are far below 4 GB */
    while (out && rc == Z_OK) {
        if (len == cap) {
            char *grown = (char *)realloc(out, cap *= 2);
            if (!grown) { free(out); out = NULL; break; }
            out = grown;
        }
        s.next_out = (Bytef *)(out + len);
        s.avail_out = (uInt)(cap - len);
        rc = inflate(&s, Z_NO_FLUSH);
        len = cap - s.avail_out;
        if (rc == Z_BUF_ERROR && s.avail_out == 0) rc = Z_OK; /* the output buffer was full: grow it */
    }
    inflateEnd(&s);
    if (!out || rc != Z_STREAM_END || len == 0) { free(out); return BLOW5_ERR_PRESS; }
    free(*mem);
    *mem = out;
    *bytes = len;
    return 0;
}

static int rec_prepare(blow5_rec_t **rec, size_t id_len, uint64_t n_samples) {
    if (!*rec && !(*rec = (blow5_rec_t *)calloc(1, sizeof **rec))) return BLOW5_ERR_PARSE;
    blow5_rec_t *r = *rec;
    char *id = (char *)realloc(r->read_id, id_len + 1);
    int16_t *raw = (int16_t *)realloc(r->raw_signal, (size_t)(n_samples ? n_samples : 1) * sizeof(int16_t));
    if (id) r->read_id = id;
    if (raw) r->raw_signal = raw;
    return id && raw ? 0 : BLOW5_ERR_PARSE;
}

int blow5_view(const blow5_file_t *f, const char *m, size_t nb, blow5_view_t *v) {
    uint16_t idl;
    double d[4];
    if (nb < 2) return BLOW5_ERR_PARSE;
    memcpy(&idl, m, 2);
    size_t at = 2;
    if (nb < at + idl + 4u + sizeof d + 8u) return BLOW5_ERR_PARSE;
    v->read_id = m + at;
    v->read_id_len = idl;
    at += idl + 4u; /* read_group */
    memcpy(d, m + at, sizeof d); /* digitisation, offset, range, sampling_rate */
    at += sizeof d;
    v->digitisation = d[0];
    v->offset = d[1];
    v->range = d[2];
    memcpy(&v->signal_bytes, m + at, 8); /* len_raw_signal: bytes of the stream with svb-zd, samples without */
    at += 8;
    v->signal = (const uint8_t *)m + at;
    if (f->signal_press == BLOW5_SIGNAL_SVB_ZD) {
        uint32_t count;
        if (v->signal_bytes < 4 || v->signal_bytes > nb - at) return BLOW5_ERR_PARSE;
        memcpy(&count, v->signal, 4);
        v->len_raw_signal = count;
    } else {
        if (v->signal_bytes > (nb - at) / 2) return BLOW5_ERR_PARSE;
        v->len_raw_signal = v->signal_bytes;
        v->signal_bytes *= 2;
    }
    return 0;
}

static int decode_binary(const blow5_file_t *f, const char *m, size_t nb, blow5_rec_t **rec) {
    blow5_view_t v;
    if (blow5_view(f, m, nb, &v) < 0 || rec_prepare(rec, v.read_id_len, v.len_raw_signal) < 0) return BLOW5_ERR_PARSE;
    blow5_rec_t *r = *rec;
    memcpy(r->read_id, v.read_id, v.read_id_len);
    r->read_id[v.read_id_len] = '\0';
    r->digitisation = v.digitisation;
    r->offset = v.offset;
    r->range = v.range;
    r->len_raw_signal = v.len_raw_signal;
    if (f->signal_press == BLOW5_SIGNAL_SVB_ZD) {
        if (blow5_svbzd_decode(v.signal, v.signal_bytes, r->raw_signal, v.len_raw_signal) != (int64_t)v.len_raw_signal)
            return BLOW5_ERR_PRESS;
    } else {
        memcpy(r->raw_signal, v.signal, (size_t)v.signal_bytes);
    }
    return 0;
}

/* a whole field as a double; 0 or BLOW5_ERR_PARSE */
static int field_double(const char *s, double *x) {
    char *end;
    *x = strtod(s, &end);
    return end == s || *end ? BLOW5_ERR_PARSE : 0;
}

/* read_id \t read_group \t digitisation \t offset \t range \t sampling_rate \t len_raw_signal \t s0,s1,... [\t aux] */
static int decode_ascii(char *line, blow5_rec_t **rec) {
    char *col[8], *save = NULL, *end;
    for (int k = 0; k < 8; k++)
        if (!(col[k] = strtok_r(k ? NULL : line, "\t", &save))) return BLOW5_ERR_PARSE;
    const uint64_t n = strtoull(col[6], &end, 10);
    if (*end || rec_prepare(rec, strlen(col[0]), n) < 0) return BLOW5_ERR_PARSE;
    blow5_rec_t *r = *rec;
    strcpy(r->read_id, col[0]);
    if (field_double(col[2], &r->digitisation) < 0 || field_double(col[3], &r->offset) < 0 ||
        field_double(col[4], &r->range) < 0)
        return BLOW5_ERR_PARSE;
    r->len_raw_signal = n;
    const char *p = col[7];
    for (uint64_t i = 0; i < n; i++) {
        const long s = strtol(p, &end, 10);
        if (end == p || s < INT16_MIN || s > INT16_MAX || (i + 1 < n ? *end != ',' : *end != '\0'))
            return BLOW5_ERR_PARSE;
        r->raw_signal[i] = (int16_t)s;
        p = end + 1;
    }
    return 0;
}

int blow5_decode(const blow5_file_t *f, char **mem, size_t *bytes, blow5_rec_t **rec) {
    int rc = blow5_inflate(f, mem, bytes);
    if (rc == 0) rc = f->ascii ? decode_ascii(*mem, rec) : decode_binary(f, *mem, *bytes, rec);
    free(*mem);
    *mem = NULL;
    return rc;
}

void blow5_rec_free(blow5_rec_t *rec) {
    if (!rec) return;
    free(rec->read_id);
    free(rec->raw_signal);
    free(rec);
}

static int idx_cmp(const void *a, const void *b) {
    return strcmp(((const blow5_idx_t *)a)->read_id, ((const blow5_idx_t *)b)->read_id);
}

int blow5_idx_load(blow5_file_t *f) {
    if (f->idx) return 0;
    const off_t start = ftello(f->fp);
    uint64_t cap = 0;
    char *mem;
    size_t nb;
    int rc;
    for (;;) {
        const off_t at = ftello(f->fp);
        if ((rc = blow5_next_bytes(f, &mem, &nb)) < 0) break;
        if ((rc = blow5_inflate(f, &mem, &nb)) < 0) { free(mem); break; }
        char *id;
        if (f->ascii) {
            id = strndup(mem, strcspn(mem, "\t"));
        } else {
            uint16_t idl = 0;
            if (nb >= 2) memcpy(&idl, mem, 2);
            id = nb >= 2u + idl ? strndup(mem + 2, idl) : NULL;
        }
        free(mem);
        if (f->n_idx == cap) {
            blow5_idx_t *grown = (blow5_idx_t *)realloc(f->idx, (size_t)(cap = cap * 2 + 1024) * sizeof *grown);
            if (!grown) { free(id); rc = BLOW5_ERR_PARSE; break; }
            f->idx = grown;
        }
        if (!id) { rc = BLOW5_ERR_PARSE; break; }
        f->idx[f->n_idx].read_id = id;
        f->idx[f->n_idx++].off = (uint64_t)at;
    }
    if (rc != BLOW5_EOF || fseeko(f->fp, start, SEEK_SET) != 0) {
        blow5_idx_unload(f);
        return rc == BLOW5_EOF ? BLOW5_ERR_IO : rc;
    }
    if (!f->idx) f->idx = (blow5_idx_t *)malloc(sizeof *f->idx); /* an empty file is indexed too */
    qsort(f->idx, (size_t)f->n_idx, sizeof *f->idx, idx_cmp);
    return f->idx ? 0 : BLOW5_ERR_IO;
}

int blow5_get(blow5_file_t *f, const char *read_id, blow5_rec_t **rec) {
    const blow5_idx_t key = {(char *)read_id, 0};
    const blow5_idx_t *hit =
        f->idx ? (const blow5_idx_t *)bsearch(&key, f->idx, (size_t)f->n_idx, sizeof key, idx_cmp) : NULL;
    if (!hit) return BLOW5_ERR_NOID;
    char *mem;
    size_t nb;
    if (fseeko(f->fp, (off_t)hit->off, SEEK_SET) != 0) return BLOW5_ERR_IO;
    const int rc = blow5_next_bytes(f, &mem, &nb);
    if (rc < 0) return rc == BLOW5_EOF ? BLOW5_ERR_IO : rc;
    return blow5_decode(f, &mem, &nb, rec);
}

void blow5_idx_unload(blow5_file_t *f) {
    for (uint64_t i = 0; i < f->n_idx; i++) free(f->idx[i].read_id);
    free(f->idx);
    f->idx = NULL;
    f->n_idx = 0;
}

/* svb-zd: value i = zigzag(raw[i] - raw[i-1]) (raw[-1] = 0, 32-bit arithmetic) stored in code+1 little-endian data
 * bytes, the 2-bit codes packed four to a key byte, lowest bits first (streamvbyte with zigzag deltas) */
int64_t blow5_svbzd_decode(const uint8_t *in, uint64_t n_bytes, int16_t *out, uint64_t cap) {
    if (n_bytes < 4) return -1;
    uint32_t count;
    memcpy(&count, in, 4);
    const uint64_t key_len = ((uint64_t)count + 3u) / 4u;
    if (count > cap || 4u + key_len > n_bytes) return -1;
    const uint8_t *keys = in + 4, *data = keys + key_len, *end = in + n_bytes;
    int32_t prev = 0;
    for (uint64_t i = 0; i < count; i++) {
        const uint32_t code = (keys[i >> 2] >> (2u * (i & 3u))) & 3u;
        if (data + code + 1u > end) return -1;
        uint32_t z = 0;
        for (uint32_t b = 0; b <= code; b++) z |= (uint32_t)data[b] << (8u * b);
        data += code + 1u;
        const int32_t d = (int32_t)((z >> 1) ^ (0u - (z & 1u)));
        prev = (int32_t)((uint32_t)prev + (uint32_t)d);
        out[i] = (int16_t)prev;
    }
    return data == end ? (int64_t)count : -1;
}
