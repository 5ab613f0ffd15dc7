/* fs_directivity.h -- the directivity factor of a path (fs_set_directivity_patterns, fs_set_source_directivity), written once
 * for k_eval / k_eval_mis and the CPU reference (tests/oracle_ext/fso_directivity.c), which include this file as C.
 *
 * Bit-exactness: binary32 * + and explicit fmaf only, in a fixed order (the CUDA translation units are compiled with
 * --fmad=false, the reference with -ffp-contract=off).
 *   c = clamp(dot(d, f), -1, 1)          dot = fmaf(d.z, f.z, fmaf(d.y, f.y, d.x * f.x)), as fs_dot; a NaN dot gives -1
 *   x = (c + 1) * 16, i = min(floor(x), 31), t = x - i
 *   g = T[i] + t (T[i+1] - T[i])         one fmaf: a constant table gives exactly that constant */
#ifndef FS_DIRECTIVITY_H
#define FS_DIRECTIVITY_H

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define FS_DIR_HD __host__ __device__ __forceinline__
#else
#define FS_DIR_HD static inline
#endif

#define FS_DIR_SEGMENTS 32u            /* FS_DIR_POINTS - 1 */

/* cosine between a unit emission direction d and the unit forward axis f, clamped to [-1, 1] */
FS_DIR_HD float fs_dir_cos(float dx, float dy, float dz, float fx, float fy, float fz)
{
    const float c = fmaf(dz, fz, fmaf(dy, fy, dx * fx));
    return fminf(fmaxf(c, -1.0f), 1.0f);
}

/* table point i (0..31) below c and the fraction t in [0, 1] towards point i + 1 */
FS_DIR_HD uint32_t fs_dir_index(float c, float* t)
{
    const float x = (c + 1.0f) * 16.0f;
    float fi = floorf(x);
    if (fi > 31.0f) fi = 31.0f;
    *t = x - fi;
    return (uint32_t)fi;
}

/* energy gain between table points t0 = T[i] and t1 = T[i+1] */
FS_DIR_HD float fs_dir_lerp(float t0, float t1, float t) { return fmaf(t, t1 - t0, t0); }

#endif
