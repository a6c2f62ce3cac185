/*
 * psulvsb_io.h -- C ABI of the host-side callers' helpers around the PSULVSB hot path
 * (libpsulvsb_b200.so).  The file readers are host code; the pre-filter and the reduced-set builder run on the
 * device (csrc/k7_prefilter.cu) and return PSULVSB_ERR_NO_DEVICE without one -- there is no CPU fallback.
 *
 * They replace, dependency-free, what the reference's experiment drivers do on the host on either
 * side of RobustRegistrationSolver::solve():
 *   - the normal-angle histogram pre-filter and the reduced-set builder, which sit INSIDE the
 *     reference's timed region: examples/teaser_cpp_ply/PSULVSB.cc:87-172 (histogram_outlier_removal)
 *     and :174-188 (mask_filter);
 *   - PLY vertex input: teaser/src/ply_io.cc:26-79 (PLYReader::read over tinyply; x, y, z as float32
 *     or float64, ascii / binary_little_endian / binary_big_endian);
 *   - the correspondence files of the real-data drivers: "x y z x y z" per line (@corr.txt,
 *     TEASER-plusplus/examples/teaser_cpp_ply/teaser_cpp_ply_main.cc:266-283), the count-header
 *     variant written by teaser_cpp_ply.cc:236-251, the 4x4 @GTmat.txt (:291-299) and gt.log (:236-246).
 * All matrices are column-major 3xN double (Eigen's layout).  Return PSULVSB_OK or an error code;
 * psulvsb_last_error() has the message.
 */
#ifndef PSULVSB_IO_H_
#define PSULVSB_IO_H_

#include "psulvsb.h"

#ifdef __cplusplus
extern "C" {
#endif

/* PSULVSB.cc:87-172.  normals: column-major 3xn (need not be unit length; NaN columns are skipped).
 * keep_mask[n] in/out: the caller passes zeros (PSULVSB.cc:310); bins further than 2 from the peak
 * get -1, bins higher than mean + 1 sigma get 1.  *remain_count = number of 1s written. */
int psulvsb_histogram_outlier_removal(const double* src_normals, const double* tgt_normals, int n, int* keep_mask,
                                      int* remain_count);
/* PSULVSB.cc:174-188.  src_reduce / tgt_reduce: capacity 3 x n doubles; reduce_map[n]: reduced column
 * of original i or -1 (dense form of the reference's std::map<int,int>); *C = number of kept columns. */
int psulvsb_mask_filter(const double* src, const double* tgt, const int* keep_mask, int n, double* src_reduce,
                        double* tgt_reduce, int* reduce_map, int* C);

/* Both of the above in one device call (one staging copy, one launch): what the reference driver times before
 * solve(), PSULVSB.cc:310-317.  keep_mask[n] in/out as for psulvsb_histogram_outlier_removal. */
int psulvsb_prefilter_reduce(const double* src_normals, const double* tgt_normals, const double* src, const double* tgt,
                             int n, int* keep_mask, double* src_reduce, double* tgt_reduce, int* reduce_map, int* C,
                             int* remain_count);

/* The same for B correspondence sets in ONE device launch (one CTA per set): arrays of B pointers, n[B] sizes in,
 * C[B] and (optional) remain_count[B] out.  What a batched driver runs before psulvsb_solve_batch. */
int psulvsb_prefilter_reduce_batch(int B, const double* const* src_normals, const double* const* tgt_normals,
                                   const double* const* src, const double* const* tgt, const int* n,
                                   int* const* keep_mask, double* const* src_reduce, double* const* tgt_reduce,
                                   int* const* reduce_map, int* C, int* remain_count);

/* PLY: number of vertices, then their x, y, z as float (teaser::PointXYZ is 3 x float). */
int psulvsb_ply_vertex_count(const char* path, long long* n);
int psulvsb_ply_read_xyz(const char* path, float* xyz, long long capacity, long long* n);
/* The same vertices with their colours, read in the same pass: the vertex properties red, green and blue, uchar / uint8
 * values divided by 255, float / double values as stored; rgb has xyz's layout (3 doubles per vertex).  A missing
 * channel or any other type is PSULVSB_ERR_INVALID with a message. */
int psulvsb_ply_read_xyz_rgb(const char* path, float* xyz, double* rgb, long long capacity, long long* n);

/* Correspondence text files.  A first line holding a single integer (the count-header variant) is
 * skipped; malformed lines are skipped like the reference's `if (iss >> ...)`. */
int psulvsb_corr_count(const char* path, long long* n);
int psulvsb_corr_read(const char* path, double* src, double* dst, long long capacity, long long* n);
/* 4x4 ground-truth transform, 4 numbers per row in the file -> column-major T[16]. */
int psulvsb_gtmat_read(const char* path, double* T);
/* gt.log: lines "i j value" -> pairs[2k], pairs[2k+1]. */
int psulvsb_gtlog_read(const char* path, int* pairs, long long capacity, long long* n);

#ifdef __cplusplus
}
#endif
#endif /* PSULVSB_IO_H_ */
