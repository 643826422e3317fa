/* lbm_io.h -- file contract of the reference CLI, host side (plain C99).
 *
 * Input:  7-value param file (d2q9-bgk.c:2736-2762), "x y 1" obstacle file
 *         (d2q9-bgk.c:2844-2857).
 * Output: final_state.dat "%d %d %.12E %.12E %.12E %.12E %d\n" (d2q9-bgk.c:2978) and
 *         av_vels.dat "%d:\t%.12E\n" (d2q9-bgk.c:2993).
 * Errors: die() prints "Error at line %d of file %s:\n%s\n" to stderr and exits with
 *         EXIT_FAILURE (d2q9-bgk.c:3001-3007).
 */
#ifndef LBM_IO_H
#define LBM_IO_H

#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include "lbm_gpu.h"

void die(const char* message, const int line, const char* file);

/* reads the 7 values; fills both the float (%f) and the double (%lf) view */
void lbm_read_params(const char* paramfile, lbm_param* pf, lbm_param_f64* pd);

/* parses the obstacle list straight into the LBM_GPU_OBST_BITS layout
 * (((nx+31)/32) uint32 words per row); returns a malloc'ed array */
uint32_t* lbm_read_obstacle_bits(const char* obstaclefile, int nx, int ny);

static inline int lbm_obstacle_bit(const uint32_t* bits, int nx, int ii, int jj)
{
  return (int)((bits[(size_t)jj * (size_t)((nx + 31) / 32) + (size_t)(ii >> 5)] >> (ii & 31)) & 1u);
}

/* appends rows [row0,row0+nrows) of final_state.dat; fields are dense nx-wide rows */
void lbm_write_final_state_rows(void* fp, int nx, long long row0, long long nrows,
                                const double* u_x, const double* u_y, const double* u,
                                const double* pressure, const uint32_t* obstacle_bits);

void lbm_write_av_vels(const char* path, int n, const double* av_vels);

/* exact equivalent of sprintf(out, "%.12E", v); returns the number of characters */
int lbm_format_e12(char* out, double v);

/* ---------------------------------------------------------------------------------
 * Checkpoint file (LBM_CHECKPOINT / LBM_RESTART): one binary file, little-endian.
 *   header, LBM_CKPT_HEADER_BYTES bytes at fixed offsets:
 *      0  char[8]  magic "LBMCKPT\0"        8  u32 format version (1)
 *     12  u32 storage kind (LBM_CKPT_*)     16  u32 LBM_STRICT (0 or 1)
 *     20  i32 nx    24  i32 ny    28  i32 reynolds_dim
 *     32  u32 bits of the fp32 parse of density, 36 accel, 40 omega    44  u32 zero
 *     48  u64 bits of the fp64 parse of density, 56 accel, 64 omega
 *     72  i64 t, the timesteps done     80  u64 lbm_obstacle_hash of the obstacle bits
 *     88  u64 lbm_gpu_digest checksum of the lattice
 *   then t av_vels values as the run produced them (float; double for f64),
 *   then the ny x nx records of lbm_gpu_save_rows (row 0 first): 36, 72 or 18 bytes per cell.
 * --------------------------------------------------------------------------------- */
#define LBM_CKPT_HEADER_BYTES 96
enum { LBM_CKPT_F32 = 0, LBM_CKPT_F64 = 1, LBM_CKPT_F16 = 2 };

typedef struct {
  uint32_t version, kind, strict;
  int32_t nx, ny, reynolds_dim;
  uint32_t density_f32, accel_f32, omega_f32;
  uint64_t density_f64, accel_f64, omega_f64;
  int64_t steps_done;
  uint64_t obstacle_hash;
  uint64_t checksum;
} lbm_ckpt_header;

/* FNV-1a over the 32-bit words of the LBM_GPU_OBST_BITS mask (row-major) */
uint64_t lbm_obstacle_hash(const uint32_t* bits, int nx, int ny);

/* the header fields this run determines (steps_done and checksum are set when writing) */
void lbm_ckpt_header_init(lbm_ckpt_header* h, uint32_t kind, int strict, const lbm_param* pf,
                          const lbm_param_f64* pd, uint64_t obstacle_hash);

/* Moves rows [row0, row0 + nrows) of the lattice between the device and buf (the host program
 * passes lbm_gpu_save_rows / lbm_gpu_load_rows wrapped in its die() convention; this file makes
 * no library calls, so that the readers and writers build without the library). */
typedef void (*lbm_ckpt_rows_fn)(void* ctx, long long row0, long long nrows, void* buf);

/* rows per block of the lattice section: about 64 MiB of records, at least 1, at most ny */
long long lbm_ckpt_block_rows(const lbm_ckpt_header* h);

/* Writes h (steps_done and checksum set by the caller), the first h->steps_done av_vels values
 * and the lattice, a block of rows at a time through buf (lbm_ckpt_block_rows rows), to
 * <path>.tmp; then fflush, fsync and rename to <path>, so that an interrupted write leaves an
 * earlier checkpoint intact. */
void lbm_write_checkpoint(const char* path, const lbm_ckpt_header* h, const void* av_vels,
                          lbm_ckpt_rows_fn save_rows, void* ctx, void* buf);

/* Opens a checkpoint and checks it against `want` (every field but steps_done and checksum),
 * t <= max_iters and the exact size the header implies; die() names any mismatch.  Needs no
 * GPU.  Returns the file positioned at the av_vels section and the header in `got`. */
FILE* lbm_open_checkpoint(const char* path, const lbm_ckpt_header* want, int max_iters, lbm_ckpt_header* got);

/* Reads the t av_vels values (float, or double for LBM_CKPT_F64) into av_vels, then the lattice
 * a block of rows at a time through buf into load_rows; closes fp.  The caller compares the
 * loaded lattice's checksum with h->checksum. */
void lbm_read_checkpoint(FILE* fp, const lbm_ckpt_header* h, void* av_vels, lbm_ckpt_rows_fn load_rows,
                         void* ctx, void* buf);

/* ---------------------------------------------------------------------------------
 * Obstacle force time series (LBM_FORCE_EVERY / LBM_FORCE_BOXES): forces.dat has one line per
 * sample state t = k, 2k, ... <= maxIters: t, then fx and fy of each box ("%.12E"), tab-separated.
 * --------------------------------------------------------------------------------- */
#define LBM_FORCE_MAX_BOXES 256      /* what lbm_gpu_obstacle_force accepts */

/* LBM_FORCE_EVERY: a positive step count, else die() */
long long lbm_parse_force_every(const char* text);

/* LBM_FORCE_BOXES "x0,y0,x1,y1;...": half-open global cell ranges with 0 <= x0 <= x1 <= nx and
 * 0 <= y0 <= y1 <= ny, at most LBM_FORCE_MAX_BOXES of them, into boxes[4 * i ...]; returns their
 * number.  A malformed box or one outside the grid ends in die() with a message that names it. */
int lbm_parse_force_boxes(const char* spec, int nx, int ny, int* boxes /* 4 * LBM_FORCE_MAX_BOXES */);

/* one line of forces.dat: step, then force[0 .. 2 * n_boxes) */
void lbm_write_force_line(FILE* fp, long long step, int n_boxes, const double* force);

#endif
