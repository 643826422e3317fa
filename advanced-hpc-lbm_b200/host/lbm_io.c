/* lbm_io.c -- parsers and writers of the d2q9-bgk file contract (see lbm_io.h). */
#define _POSIX_C_SOURCE 200809L
#include "lbm_io.h"

#include <ctype.h>
#include <errno.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/types.h>
#include <unistd.h>

void die(const char* message, const int line, const char* file)
{
  fprintf(stderr, "Error at line %d of file %s:\n", line, file);
  fprintf(stderr, "%s\n", message);
  fflush(stderr);
  exit(EXIT_FAILURE);
}

static int read_int(FILE* fp, int* out)
{
  return fscanf(fp, "%d\n", out) == 1;
}

/* one real value, kept as text so it can be converted the way %f and %lf would */
static int read_real(FILE* fp, float* f, double* d)
{
  char tok[128];
  if (fscanf(fp, "%127s", tok) != 1) return 0;
  char* end = NULL;
  errno = 0;
  *d = strtod(tok, &end);
  if (end == tok) return 0;
  *f = strtof(tok, NULL);
  return 1;
}

void lbm_read_params(const char* paramfile, lbm_param* pf, lbm_param_f64* pd)
{
  char message[1024];
  FILE* fp = fopen(paramfile, "r");
  if (fp == NULL) {
    snprintf(message, sizeof message, "could not open input parameter file: %s", paramfile);
    die(message, __LINE__, __FILE__);
  }
  if (!read_int(fp, &pf->nx)) die("could not read param file: nx", __LINE__, __FILE__);
  if (!read_int(fp, &pf->ny)) die("could not read param file: ny", __LINE__, __FILE__);
  if (!read_int(fp, &pf->maxIters)) die("could not read param file: maxIters", __LINE__, __FILE__);
  if (!read_int(fp, &pf->reynolds_dim)) die("could not read param file: reynolds_dim", __LINE__, __FILE__);
  if (!read_real(fp, &pf->density, &pd->density)) die("could not read param file: density", __LINE__, __FILE__);
  if (!read_real(fp, &pf->accel, &pd->accel)) die("could not read param file: accel", __LINE__, __FILE__);
  if (!read_real(fp, &pf->omega, &pd->omega)) die("could not read param file: omega", __LINE__, __FILE__);
  fclose(fp);
  pd->nx = pf->nx; pd->ny = pf->ny; pd->maxIters = pf->maxIters; pd->reynolds_dim = pf->reynolds_dim;
}

/* Obstacle list -> bit mask.  The reference reads "%d %d %d\n" triples until EOF and
 * dies on a short triple, an out-of-range coordinate or a third value other than 1
 * (d2q9-bgk.c:2844-2853).  Synthetic grids have millions of lines, so the file is read
 * in blocks and tokenised by hand instead of one fscanf per line. */
uint32_t* lbm_read_obstacle_bits(const char* obstaclefile, int nx, int ny)
{
  char message[1024];
  FILE* fp = fopen(obstaclefile, "r");
  if (fp == NULL) {
    snprintf(message, sizeof message, "could not open input obstacles file: %s", obstaclefile);
    die(message, __LINE__, __FILE__);
  }
  const size_t wpr = (size_t)((nx + 31) / 32);
  uint32_t* bits = (uint32_t*)calloc(wpr * (size_t)ny, sizeof(uint32_t));
  if (bits == NULL) die("cannot allocate column memory for obstacles", __LINE__, __FILE__);

  enum { BUF = 1 << 20 };
  char* buf = (char*)malloc(BUF);
  if (buf == NULL) die("cannot allocate column memory for obstacles", __LINE__, __FILE__);
  long long vals[3];
  int nvals = 0;          /* values of the current triple already parsed */
  int in_tok = 0, neg = 0, digits = 0;
  long long cur = 0;
  size_t got;
  int eof = 0;
  while (!eof) {
    got = fread(buf, 1, BUF, fp);
    if (got < BUF) { eof = 1; buf[got++] = '\n'; }   /* sentinel ends a last token */
    for (size_t i = 0; i < got; i++) {
      const char c = buf[i];
      if (c >= '0' && c <= '9') {
        if (!in_tok) { in_tok = 1; neg = 0; cur = 0; digits = 0; }
        if (cur < (1LL << 40)) cur = cur * 10 + (c - '0');
        digits++;
      } else if ((c == '-' || c == '+') && !in_tok) {
        in_tok = 1; neg = (c == '-'); cur = 0; digits = 0;
      } else if (isspace((unsigned char)c)) {
        if (in_tok) {
          if (digits == 0) die("expected 3 values per line in obstacle file", __LINE__, __FILE__);
          vals[nvals++] = neg ? -cur : cur;
          in_tok = 0;
          if (nvals == 3) {
            if (vals[0] < 0 || vals[0] > nx - 1) die("obstacle x-coord out of range", __LINE__, __FILE__);
            if (vals[1] < 0 || vals[1] > ny - 1) die("obstacle y-coord out of range", __LINE__, __FILE__);
            if (vals[2] != 1) die("obstacle blocked value should be 1", __LINE__, __FILE__);
            bits[(size_t)vals[1] * wpr + (size_t)(vals[0] >> 5)] |= 1u << (vals[0] & 31);
            nvals = 0;
          }
        }
      } else {
        die("expected 3 values per line in obstacle file", __LINE__, __FILE__);
      }
    }
  }
  if (nvals != 0) die("expected 3 values per line in obstacle file", __LINE__, __FILE__);
  free(buf);
  fclose(fp);
  return bits;
}

/* ---------------------------------------------------------------------------------
 * Fast, exact "%.12E".  The output files are millions of lines of four such numbers;
 * once the step loop runs on the GPU, fprintf's general-purpose conversion is what the
 * program spends its time in (SURVEY.md section 8f, rank 1).  v = m * 2^e exactly, so
 * v * 10^p = m * 5^p * 2^(e+p) is an integer shift away from a 128-bit product; rounding
 * half-to-even on that exact value gives the same 13 digits glibc prints.  Values outside
 * the range the 128-bit product covers fall back to snprintf.
 * tests/test_host_format.py compares it with printf on millions of values.
 * --------------------------------------------------------------------------------- */
typedef unsigned __int128 u128;

static u128 pow5_table[56];
static int pow5_ready = 0;

static void pow5_init(void)
{
  pow5_table[0] = 1;
  for (int i = 1; i < 56; i++) pow5_table[i] = pow5_table[i - 1] * 5;
  pow5_ready = 1;
}

int lbm_format_e12(char* out, double v)
{
  union { double d; uint64_t u; } x;
  x.d = v;
  const int neg = (int)(x.u >> 63);
  const uint64_t frac = x.u & ((1ULL << 52) - 1);
  const int be = (int)((x.u >> 52) & 0x7ff);
  if (be == 0x7ff) return sprintf(out, "%.12E", v);
  char* o = out;
  if (neg) *o++ = '-';
  if (be == 0 && frac == 0) {
    memcpy(o, "0.000000000000E+00", 18);
    o += 18;
    *o = '\0';
    return (int)(o - out);
  }
  if (!pow5_ready) pow5_init();
  uint64_t m = (be == 0) ? frac : (frac | (1ULL << 52));
  int e = (be == 0) ? -1074 : be - 1075;
  const int tz = __builtin_ctzll(m);
  m >>= tz;
  e += tz;
  const int bl = 64 - __builtin_clzll(m);
  int k = (int)floor((double)(e + bl - 1) * 0.30102999566398120);
  const uint64_t lo_lim = 1000000000000ULL, hi_lim = 10000000000000ULL;
  uint64_t n = 0;
  for (int tries = 0; ; tries++) {
    const int p = 12 - k;
    if (tries > 3 || p < 0 || p > 55) return sprintf(out, "%.12E", v);
    /* bits of m * 5^p: bl + ceil(p * log2(5)) */
    const int need = bl + (int)(p * 2.3219280948873623) + 1;
    if (need > 126) return sprintf(out, "%.12E", v);
    const u128 a = (u128)m * pow5_table[p];
    const int sh = e + p;
    u128 q;
    if (sh >= 0) {
      if (need + sh > 126) return sprintf(out, "%.12E", v);
      q = a << sh;
    } else {
      const int s = -sh;
      if (s >= 127) return sprintf(out, "%.12E", v);
      q = a >> s;
      const u128 rem = a & (((u128)1 << s) - 1);
      const u128 half = (u128)1 << (s - 1);
      if (rem > half || (rem == half && (q & 1))) q++;
    }
    if (q < lo_lim) { k--; continue; }
    if (q >= hi_lim) { k++; continue; }
    n = (uint64_t)q;
    break;
  }
  char digits[13];
  for (int i = 12; i >= 0; i--) { digits[i] = (char)('0' + n % 10); n /= 10; }
  *o++ = digits[0];
  *o++ = '.';
  memcpy(o, digits + 1, 12);
  o += 12;
  *o++ = 'E';
  int ex = k;
  if (ex < 0) { *o++ = '-'; ex = -ex; } else { *o++ = '+'; }
  if (ex >= 100) { *o++ = (char)('0' + ex / 100); ex %= 100; }
  *o++ = (char)('0' + ex / 10);
  *o++ = (char)('0' + ex % 10);
  *o = '\0';
  return (int)(o - out);
}

static char* put_int(char* o, long long v)
{
  char tmp[24];
  int n = 0;
  if (v < 0) { *o++ = '-'; v = -v; }
  do { tmp[n++] = (char)('0' + v % 10); v /= 10; } while (v);
  while (n) *o++ = tmp[--n];
  return o;
}

/* formats rows [r_begin, r_end) of a block into buf; returns the number of bytes */
static size_t format_rows(char* buf, int nx, long long row0, long long r_begin, long long r_end,
                          const double* u_x, const double* u_y, const double* u, const double* pressure,
                          const uint32_t* obstacle_bits)
{
  char* o = buf;
  for (long long r = r_begin; r < r_end; r++) {
    const long long jj = row0 + r;
    for (int ii = 0; ii < nx; ii++) {
      const size_t n = (size_t)r * (size_t)nx + (size_t)ii;
      /* "%d %d %.12E %.12E %.12E %.12E %d\n" (d2q9-bgk.c:2978).  Last column: the cell's
       * own obstacle flag.  The reference prints obstacles[ii*nx + jj], a transposed index
       * that differs from the golden files in check/ for non-symmetric masks; the golden
       * files hold the cell's own flag, which is what is written here (check.py ignores
       * the column). */
      o = put_int(o, ii); *o++ = ' ';
      o = put_int(o, jj); *o++ = ' ';
      o += lbm_format_e12(o, u_x[n]); *o++ = ' ';
      o += lbm_format_e12(o, u_y[n]); *o++ = ' ';
      o += lbm_format_e12(o, u[n]); *o++ = ' ';
      o += lbm_format_e12(o, pressure[n]); *o++ = ' ';
      *o++ = (char)('0' + lbm_obstacle_bit(obstacle_bits, nx, ii, (int)jj));
      *o++ = '\n';
    }
  }
  return (size_t)(o - buf);
}

/* The block is cut into pieces that are formatted in parallel (OpenMP, if the host was
 * built with it) and written in order: the text is identical for any thread count. */
void lbm_write_final_state_rows(void* fpv, int nx, long long row0, long long nrows,
                                const double* u_x, const double* u_y, const double* u,
                                const double* pressure, const uint32_t* obstacle_bits)
{
  FILE* fp = (FILE*)fpv;
  enum { LINE_MAX_BYTES = 128 };          /* 2 ints (<= 11 chars) + 4 x 19 chars + flag + separators */
  if (!pow5_ready) pow5_init();           /* before the threads start */
  long long pieces = nrows < 64 ? nrows : 64;
  if (pieces < 1) return;
  char** bufs = (char**)calloc((size_t)pieces, sizeof(char*));
  size_t* lens = (size_t*)calloc((size_t)pieces, sizeof(size_t));
  if (bufs == NULL || lens == NULL) die("cannot allocate memory for output rows", __LINE__, __FILE__);
  int failed = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(|:failed)
  for (long long p = 0; p < pieces; p++) {
    const long long rb = nrows * p / pieces, re = nrows * (p + 1) / pieces;
    bufs[p] = (char*)malloc((size_t)(re - rb) * (size_t)nx * LINE_MAX_BYTES + 1);
    if (bufs[p] == NULL) { failed |= 1; continue; }
    lens[p] = format_rows(bufs[p], nx, row0, rb, re, u_x, u_y, u, pressure, obstacle_bits);
  }
  if (failed) die("cannot allocate memory for output rows", __LINE__, __FILE__);
  for (long long p = 0; p < pieces; p++) {
    if (lens[p] && fwrite(bufs[p], 1, lens[p], fp) != lens[p]) die("could not write output file", __LINE__, __FILE__);
    free(bufs[p]);
  }
  free(bufs);
  free(lens);
}

void lbm_write_av_vels(const char* path, int n, const double* av_vels)
{
  FILE* fp = fopen(path, "w");
  if (fp == NULL) die("could not open file output file", __LINE__, __FILE__);
  static char big[1 << 20];
  setvbuf(fp, big, _IOFBF, sizeof big);
  char line[64];
  for (int ii = 0; ii < n; ii++) {
    /* "%d:\t%.12E\n" (d2q9-bgk.c:2993) */
    char* o = put_int(line, ii);
    *o++ = ':'; *o++ = '\t';
    o += lbm_format_e12(o, av_vels[ii]);
    *o++ = '\n';
    fwrite(line, 1, (size_t)(o - line), fp);
  }
  fclose(fp);
}

/* ---------------------------------------------------------------------------------
 * Checkpoint file (layout in lbm_io.h).  Written and read through lbm_gpu_save_rows /
 * lbm_gpu_load_rows a block of rows at a time: the whole lattice is never on the host.
 * --------------------------------------------------------------------------------- */
static const char ckpt_magic[8] = {'L', 'B', 'M', 'C', 'K', 'P', 'T', '\0'};

static size_t ckpt_record_bytes(uint32_t kind) { return kind == LBM_CKPT_F64 ? 72 : kind == LBM_CKPT_F16 ? 18 : 36; }
static size_t ckpt_av_bytes(uint32_t kind) { return kind == LBM_CKPT_F64 ? 8 : 4; }
static const char* ckpt_kind_name(uint32_t kind)
{
  return kind == LBM_CKPT_F32 ? "fp32" : kind == LBM_CKPT_F64 ? "fp64 (LBM_PRECISION=f64)"
       : kind == LBM_CKPT_F16 ? "binary16 (LBM_PRECISION=f16)" : "unknown";
}

static void put_le(unsigned char* p, uint64_t v, int n)
{
  for (int i = 0; i < n; i++) p[i] = (unsigned char)(v >> (8 * i));
}
static uint64_t get_le(const unsigned char* p, int n)
{
  uint64_t v = 0;
  for (int i = 0; i < n; i++) v |= (uint64_t)p[i] << (8 * i);
  return v;
}

/* the av_vels and lattice sections are copied as they are in memory */
static void ckpt_require_little_endian(void)
{
  const uint16_t one = 1;
  if (*(const unsigned char*)&one != 1) die("checkpoint files are little-endian and this host is not", __LINE__, __FILE__);
}

uint64_t lbm_obstacle_hash(const uint32_t* bits, int nx, int ny)
{
  const size_t n = (size_t)((nx + 31) / 32) * (size_t)ny;
  uint64_t h = 0xcbf29ce484222325ULL;
  for (size_t i = 0; i < n; i++) {
    h ^= bits[i];
    h *= 0x100000001b3ULL;
  }
  return h;
}

void lbm_ckpt_header_init(lbm_ckpt_header* h, uint32_t kind, int strict, const lbm_param* pf,
                          const lbm_param_f64* pd, uint64_t obstacle_hash)
{
  memset(h, 0, sizeof *h);
  h->version = 1;
  h->kind = kind;
  h->strict = strict ? 1u : 0u;
  h->nx = pf->nx; h->ny = pf->ny; h->reynolds_dim = pf->reynolds_dim;
  memcpy(&h->density_f32, &pf->density, 4); memcpy(&h->accel_f32, &pf->accel, 4); memcpy(&h->omega_f32, &pf->omega, 4);
  memcpy(&h->density_f64, &pd->density, 8); memcpy(&h->accel_f64, &pd->accel, 8); memcpy(&h->omega_f64, &pd->omega, 8);
  h->obstacle_hash = obstacle_hash;
}

static void ckpt_encode(const lbm_ckpt_header* h, unsigned char* b)
{
  memset(b, 0, LBM_CKPT_HEADER_BYTES);
  memcpy(b, ckpt_magic, 8);
  put_le(b + 8, h->version, 4); put_le(b + 12, h->kind, 4); put_le(b + 16, h->strict, 4);
  put_le(b + 20, (uint32_t)h->nx, 4); put_le(b + 24, (uint32_t)h->ny, 4); put_le(b + 28, (uint32_t)h->reynolds_dim, 4);
  put_le(b + 32, h->density_f32, 4); put_le(b + 36, h->accel_f32, 4); put_le(b + 40, h->omega_f32, 4);
  put_le(b + 48, h->density_f64, 8); put_le(b + 56, h->accel_f64, 8); put_le(b + 64, h->omega_f64, 8);
  put_le(b + 72, (uint64_t)h->steps_done, 8); put_le(b + 80, h->obstacle_hash, 8); put_le(b + 88, h->checksum, 8);
}

static void ckpt_decode(const unsigned char* b, lbm_ckpt_header* h)
{
  h->version = (uint32_t)get_le(b + 8, 4); h->kind = (uint32_t)get_le(b + 12, 4); h->strict = (uint32_t)get_le(b + 16, 4);
  h->nx = (int32_t)get_le(b + 20, 4); h->ny = (int32_t)get_le(b + 24, 4); h->reynolds_dim = (int32_t)get_le(b + 28, 4);
  h->density_f32 = (uint32_t)get_le(b + 32, 4); h->accel_f32 = (uint32_t)get_le(b + 36, 4); h->omega_f32 = (uint32_t)get_le(b + 40, 4);
  h->density_f64 = get_le(b + 48, 8); h->accel_f64 = get_le(b + 56, 8); h->omega_f64 = get_le(b + 64, 8);
  h->steps_done = (int64_t)get_le(b + 72, 8); h->obstacle_hash = get_le(b + 80, 8); h->checksum = get_le(b + 88, 8);
}

long long lbm_ckpt_block_rows(const lbm_ckpt_header* h)
{
  long long n = (long long)((64u << 20) / ((size_t)h->nx * ckpt_record_bytes(h->kind)));
  if (n < 1) n = 1;
  if (n > h->ny) n = h->ny;
  return n;
}

void lbm_write_checkpoint(const char* path, const lbm_ckpt_header* h, const void* av_vels,
                          lbm_ckpt_rows_fn save_rows, void* ctx, void* buf)
{
  char message[1024];
  ckpt_require_little_endian();
  char* tmp = (char*)malloc(strlen(path) + 5);
  if (tmp == NULL) die("cannot allocate memory for the checkpoint path", __LINE__, __FILE__);
  sprintf(tmp, "%s.tmp", path);
  FILE* fp = fopen(tmp, "wb");
  if (fp == NULL) {
    snprintf(message, sizeof message, "could not open checkpoint file for writing: %s", tmp);
    die(message, __LINE__, __FILE__);
  }
  unsigned char hb[LBM_CKPT_HEADER_BYTES];
  ckpt_encode(h, hb);
  int ok = fwrite(hb, 1, sizeof hb, fp) == sizeof hb;
  const size_t avb = ckpt_av_bytes(h->kind);
  if (ok && h->steps_done > 0) ok = fwrite(av_vels, avb, (size_t)h->steps_done, fp) == (size_t)h->steps_done;
  const size_t row_bytes = (size_t)h->nx * ckpt_record_bytes(h->kind);
  const long long block = lbm_ckpt_block_rows(h);
  for (long long r0 = 0; ok && r0 < h->ny; r0 += block) {
    const long long nr = (r0 + block <= h->ny) ? block : h->ny - r0;
    save_rows(ctx, r0, nr, buf);
    ok = fwrite(buf, row_bytes, (size_t)nr, fp) == (size_t)nr;
  }
  ok = ok && fflush(fp) == 0 && fsync(fileno(fp)) == 0;
  ok = (fclose(fp) == 0) && ok;
  if (!ok) {
    snprintf(message, sizeof message, "could not write checkpoint file: %s", tmp);
    die(message, __LINE__, __FILE__);
  }
  if (rename(tmp, path) != 0) {
    snprintf(message, sizeof message, "could not rename %s to %s", tmp, path);
    die(message, __LINE__, __FILE__);
  }
  free(tmp);
}

FILE* lbm_open_checkpoint(const char* path, const lbm_ckpt_header* want, int max_iters, lbm_ckpt_header* got)
{
  char message[1024];
  ckpt_require_little_endian();
  FILE* fp = fopen(path, "rb");
  if (fp == NULL) {
    snprintf(message, sizeof message, "could not open checkpoint file: %s", path);
    die(message, __LINE__, __FILE__);
  }
  unsigned char hb[LBM_CKPT_HEADER_BYTES];
  const size_t n = fread(hb, 1, sizeof hb, fp);
  if (n < 8 || memcmp(hb, ckpt_magic, 8) != 0) {
    snprintf(message, sizeof message, "checkpoint %s: not a checkpoint of this program (wrong magic)", path);
    die(message, __LINE__, __FILE__);
  }
  if (n < sizeof hb) {
    snprintf(message, sizeof message, "checkpoint %s: truncated header (%zu of %d bytes)", path, n, LBM_CKPT_HEADER_BYTES);
    die(message, __LINE__, __FILE__);
  }
  ckpt_decode(hb, got);
#define CKPT_MISMATCH(...)                                   \
  do {                                                       \
    int k_ = snprintf(message, sizeof message, "checkpoint %s: ", path);   \
    snprintf(message + k_, sizeof message - (size_t)k_, __VA_ARGS__);      \
    die(message, __LINE__, __FILE__);                        \
  } while (0)
  if (got->version != want->version)
    CKPT_MISMATCH("format version %u, this program reads version %u", got->version, want->version);
  if (got->kind != want->kind)
    CKPT_MISMATCH("holds a %s lattice, this run asks for %s", ckpt_kind_name(got->kind), ckpt_kind_name(want->kind));
  if (got->strict != want->strict)
    CKPT_MISMATCH("written with LBM_STRICT=%u, this run has LBM_STRICT=%u", got->strict, want->strict);
  if (got->nx != want->nx) CKPT_MISMATCH("nx is %d, the parameter file's is %d", got->nx, want->nx);
  if (got->ny != want->ny) CKPT_MISMATCH("ny is %d, the parameter file's is %d", got->ny, want->ny);
  if (got->reynolds_dim != want->reynolds_dim)
    CKPT_MISMATCH("reynolds_dim is %d, the parameter file's is %d", got->reynolds_dim, want->reynolds_dim);
  if (got->density_f32 != want->density_f32 || got->density_f64 != want->density_f64)
    CKPT_MISMATCH("density differs from the parameter file's");
  if (got->accel_f32 != want->accel_f32 || got->accel_f64 != want->accel_f64)
    CKPT_MISMATCH("accel differs from the parameter file's");
  if (got->omega_f32 != want->omega_f32 || got->omega_f64 != want->omega_f64)
    CKPT_MISMATCH("omega differs from the parameter file's");
  if (got->obstacle_hash != want->obstacle_hash)
    CKPT_MISMATCH("written with another obstacle file (the obstacle mask hash differs)");
  if (got->steps_done < 0 || got->steps_done > max_iters)
    CKPT_MISMATCH("is at step %lld, beyond maxIters = %d of the parameter file", (long long)got->steps_done, max_iters);
  const long long expect = LBM_CKPT_HEADER_BYTES + got->steps_done * (long long)ckpt_av_bytes(got->kind) +
                           (long long)got->ny * got->nx * (long long)ckpt_record_bytes(got->kind);
  if (fseeko(fp, 0, SEEK_END) != 0) CKPT_MISMATCH("cannot seek");
  const long long size = (long long)ftello(fp);
  if (size != expect)
    CKPT_MISMATCH("file has %lld bytes, its header implies %lld (truncated or corrupt)", size, expect);
#undef CKPT_MISMATCH
  if (fseeko(fp, LBM_CKPT_HEADER_BYTES, SEEK_SET) != 0) die("cannot seek in the checkpoint file", __LINE__, __FILE__);
  return fp;
}

void lbm_read_checkpoint(FILE* fp, const lbm_ckpt_header* h, void* av_vels, lbm_ckpt_rows_fn load_rows,
                         void* ctx, void* buf)
{
  const size_t avb = ckpt_av_bytes(h->kind);
  if (h->steps_done > 0 && fread(av_vels, avb, (size_t)h->steps_done, fp) != (size_t)h->steps_done)
    die("could not read the av_vels of the checkpoint file", __LINE__, __FILE__);
  const size_t row_bytes = (size_t)h->nx * ckpt_record_bytes(h->kind);
  const long long block = lbm_ckpt_block_rows(h);
  for (long long r0 = 0; r0 < h->ny; r0 += block) {
    const long long nr = (r0 + block <= h->ny) ? block : h->ny - r0;
    if (fread(buf, row_bytes, (size_t)nr, fp) != (size_t)nr) die("could not read the lattice of the checkpoint file", __LINE__, __FILE__);
    load_rows(ctx, r0, nr, buf);
  }
  fclose(fp);
}

/* ------------------------------------------------------------------ obstacle force time series */
long long lbm_parse_force_every(const char* text)
{
  char* end = NULL;
  errno = 0;
  const long long k = strtoll(text, &end, 10);
  if (end == text || *end != '\0' || errno != 0 || k < 1 || k > 2147483647LL)
    die("LBM_FORCE_EVERY must be a positive number of steps", __LINE__, __FILE__);
  return k;
}

int lbm_parse_force_boxes(const char* spec, int nx, int ny, int* boxes)
{
  char msg[512];
  int n = 0;
  const char* p = spec;
  for (;;) {
    const char* end = strchr(p, ';');
    const size_t len = end ? (size_t)(end - p) : strlen(p);
    char item[128];
    if (n == LBM_FORCE_MAX_BOXES) {
      snprintf(msg, sizeof msg, "LBM_FORCE_BOXES: more than %d boxes", LBM_FORCE_MAX_BOXES);
      die(msg, __LINE__, __FILE__);
    }
    long long v[4];
    int ok = len > 0 && len < sizeof item;
    if (ok) {
      memcpy(item, p, len);
      item[len] = '\0';
      const char* q = item;
      for (int i = 0; i < 4 && ok; i++) {
        char* e = NULL;
        errno = 0;
        while (*q == ' ') q++;
        v[i] = strtoll(q, &e, 10);
        ok = e != q && errno == 0;
        q = e;
        while (*q == ' ') q++;
        if (ok && i < 3) ok = *q++ == ',';
      }
      ok = ok && *q == '\0';
    }
    if (!ok) {
      snprintf(msg, sizeof msg, "LBM_FORCE_BOXES: box %d (\"%.*s\") is not four integers x0,y0,x1,y1", n,
               (int)(len < 100 ? len : 100), p);
      die(msg, __LINE__, __FILE__);
    }
    if (!(0 <= v[0] && v[0] <= v[2] && v[2] <= nx && 0 <= v[1] && v[1] <= v[3] && v[3] <= ny)) {
      snprintf(msg, sizeof msg, "LBM_FORCE_BOXES: box %d (%lld,%lld,%lld,%lld) is not within 0 <= x0 <= x1 <= nx = %d "
               "and 0 <= y0 <= y1 <= ny = %d", n, v[0], v[1], v[2], v[3], nx, ny);
      die(msg, __LINE__, __FILE__);
    }
    for (int i = 0; i < 4; i++) boxes[4 * n + i] = (int)v[i];
    n++;
    if (!end) break;
    p = end + 1;
  }
  return n;
}

void lbm_write_force_line(FILE* fp, long long step, int n_boxes, const double* force)
{
  char line[32 + LBM_FORCE_MAX_BOXES * 2 * 24];
  int o = snprintf(line, sizeof line, "%lld", step);
  for (int i = 0; i < 2 * n_boxes; i++) {
    line[o++] = '\t';
    o += lbm_format_e12(line + o, force[i]);
  }
  line[o++] = '\n';
  if (fwrite(line, 1, (size_t)o, fp) != (size_t)o) die("could not write forces.dat", __LINE__, __FILE__);
}
