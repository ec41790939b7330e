/* Ray directions of the mesh occupancy query (`RaycastingScene.compute_occupancy` / `compute_signed_distance`):
 * plain C, included by csrc/bslam_mesh_raycast.cu (host side; the set is passed to the kernel by value) and by the
 * brute-force CPU reference tests/mesh_query_ref.c, so that both cast the same float32 directions.
 *
 * Direction i (0-based) is the R2 low-discrepancy point (Roberts 2018, the plastic number p: frac(0.5 + (i + 1) / p),
 * frac(0.5 + (i + 1) / p^2)) mapped area-preservingly onto the unit sphere, in float64, then cast to float32.  Every
 * prefix of the sequence is spread over the sphere, so the first nsamples directions are a fair set for any nsamples.
 * No direction lies on a coordinate axis or in a coordinate plane (every component has magnitude >= 0.024), so rays from
 * grid points do not run along the faces and edges of axis-aligned meshes. */
#ifndef BSLAM_MESH_DIRS_H
#define BSLAM_MESH_DIRS_H

#include <math.h>

#define BSLAM_MESH_MAX_SAMPLES 31

static inline void bslam_mesh_direction_set(int n, float *dirs /* [n][3] */) {
    const double p = 1.32471795724474602596, a1 = 1.0 / p, a2 = 1.0 / (p * p), two_pi = 6.283185307179586476925;
    for (int i = 0; i < n; ++i) {
        const double x = fmod(0.5 + a1 * (double)(i + 1), 1.0), y = fmod(0.5 + a2 * (double)(i + 1), 1.0);
        const double z = 1.0 - 2.0 * x, r = sqrt(fmax(0.0, 1.0 - z * z)), phi = two_pi * y;
        dirs[3 * i] = (float)(r * cos(phi));
        dirs[3 * i + 1] = (float)(r * sin(phi));
        dirs[3 * i + 2] = (float)z;
    }
}

#endif
