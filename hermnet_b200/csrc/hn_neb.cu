// Nudged elastic band forces of the device loop: improved tangent (Henkelman & Jonsson, JCP 113, 9978 (2000)) and
// climbing image (Henkelman, Uberuaga & Jonsson, JCP 113, 9901 (2000)), as ASE's NEB(method="improvedtangent").
// Band-major layout: band b holds its K interior images one after the other, image g = b K + k is the contiguous atom
// range [image_ptr[g], image_ptr[g+1]) of n_b atoms, so the same atom of the neighbouring images sits at i -/+ n_b; the
// endpoints of band b are rows band_ptr[b] + local of `initial` / `final`.  With D+ = R_{k+1} - R_k, D- = R_k - R_{k-1}
// and the tangent tau = a D+ + b D-, three launches after each evaluation:
//   reduce   per atom, then per image in a fixed order: S++, S--, S+-, F.D+, F.D- (float64)
//   step     per band: tangent weights (a, b) from the energies, the climbing image, coef = q (a, b)
//   project  per atom: F <- F + c+ D+ + c- D-  (float64 arithmetic, fp32 in place)
#include "hn_common.cuh"
#include "hn_reduce.cuh"

namespace {

struct NebSums {
    double pp, mm, pm, fp, fm;   // |D+|^2, |D-|^2, D+.D-, F.D+, F.D-
    __device__ __forceinline__ void merge(const NebSums &o) { pp += o.pp, mm += o.mm, pm += o.pm, fp += o.fp, fm += o.fm; }
    __device__ __forceinline__ NebSums shfl_xor(int o) const {
        return {__shfl_xor_sync(0xffffffffu, pp, o), __shfl_xor_sync(0xffffffffu, mm, o), __shfl_xor_sync(0xffffffffu, pm, o),
                __shfl_xor_sync(0xffffffffu, fp, o), __shfl_xor_sync(0xffffffffu, fm, o)};
    }
};

// Where the neighbours of the atoms of image g are: i - prev_step / i + next_step inside the band, or endpoint row
// i + end_off at the band's ends.
struct ImageNbrs {
    int n_b, end_off;
    bool first, last;
};

__device__ __forceinline__ ImageNbrs image_nbrs(int g, int K, const int *__restrict__ image_ptr, const int *__restrict__ band_ptr) {
    const int b = g / K, k = g - b * K, p = __ldg(image_ptr + g);
    return {__ldg(image_ptr + g + 1) - p, __ldg(band_ptr + b) - p, k == 0, k == K - 1};
}

// D+ and D- of atom i (float64 differences of fp32 positions)
__device__ __forceinline__ void deltas(const float *__restrict__ pos, const float *__restrict__ initial,
                                       const float *__restrict__ final_, const ImageNbrs &nb, int i, double dp[3], double dm[3]) {
    const float *x = pos + 3 * (size_t)i;
    const float *xm = nb.first ? initial + 3 * (size_t)(i + nb.end_off) : x - 3 * (size_t)nb.n_b;
    const float *xp = nb.last ? final_ + 3 * (size_t)(i + nb.end_off) : x + 3 * (size_t)nb.n_b;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const double xc = x[c];
        dp[c] = (double)__ldg(xp + c) - xc;
        dm[c] = xc - (double)__ldg(xm + c);
    }
}

__global__ void neb_reduce_pieces_kernel(const float *__restrict__ pos, const float *__restrict__ force,
                                         const float *__restrict__ initial, const float *__restrict__ final_,
                                         const int *__restrict__ image, const int *__restrict__ image_ptr,
                                         const int *__restrict__ band_ptr, int K, int n_atoms, int n_chunks,
                                         NebSums *__restrict__ part) {
    hn::reduce_pieces<NebSums>(image, image_ptr, n_atoms, n_chunks, part, [&](int g) {
        const ImageNbrs nb = image_nbrs(g, K, image_ptr, band_ptr);
        return [=](NebSums &acc, int i) {
            double dp[3], dm[3];
            deltas(pos, initial, final_, nb, i, dp, dm);
            const double f0 = __ldg(force + 3 * (size_t)i), f1 = __ldg(force + 3 * (size_t)i + 1), f2 = __ldg(force + 3 * (size_t)i + 2);
            acc.pp += dp[0] * dp[0] + dp[1] * dp[1] + dp[2] * dp[2];
            acc.mm += dm[0] * dm[0] + dm[1] * dm[1] + dm[2] * dm[2];
            acc.pm += dp[0] * dm[0] + dp[1] * dm[1] + dp[2] * dm[2];
            acc.fp += f0 * dp[0] + f1 * dp[1] + f2 * dp[2];
            acc.fm += f0 * dm[0] + f1 * dm[1] + f2 * dm[2];
        };
    });
}

__global__ void neb_reduce_final_kernel(const NebSums *__restrict__ part, const int *__restrict__ image_ptr, int n_img, int per,
                                        double *__restrict__ out) {
    int g;
    NebSums acc;
    if (!hn::reduce_slots(part, image_ptr, n_img, per, g, acc)) return;
    double *o = out + 5 * (size_t)g;
    o[0] = acc.pp, o[1] = acc.mm, o[2] = acc.pm, o[3] = acc.fp, o[4] = acc.fm;
}

// One thread per band: the first interior image of maximal energy, then (a, b) and q of each image.
__global__ void neb_step_kernel(const double *__restrict__ sums, const float *__restrict__ energy, const float *__restrict__ end_energy,
                                const double *__restrict__ spring, int climb, int n_bands, int K, double *__restrict__ coef,
                                int *__restrict__ imax) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n_bands) return;
    const float *E = energy + (size_t)b * K;
    int top = 0;
    for (int k = 1; k < K; ++k)
        if ((double)E[k] > (double)E[top]) top = k;
    imax[b] = top + 1;
    const double ks = spring[b];
    for (int k = 0; k < K; ++k) {
        const size_t g = (size_t)b * K + k;
        const double e = E[k], em = k == 0 ? (double)end_energy[2 * b] : (double)E[k - 1],
                     ep = k == K - 1 ? (double)end_energy[2 * b + 1] : (double)E[k + 1];
        double a, w;                                        // tau = a D+ + w D-
        if (ep > e && e > em) {
            a = 1.0, w = 0.0;
        } else if (ep < e && e < em) {
            a = 0.0, w = 1.0;
        } else {
            const double up = fabs(ep - e), dn = fabs(em - e), vmax = fmax(up, dn), vmin = fmin(up, dn);
            if (vmax == 0.0) a = 1.0, w = 1.0;              // three equal energies: the limit of the weights
            else if (ep > em) a = vmax, w = vmin;
            else a = vmin, w = vmax;
        }
        const double *s = sums + 5 * g;
        const double spp = s[0], smm = s[1], spm = s[2], fp = s[3], fm = s[4];
        const double T = a * a * spp + 2.0 * a * w * spm + w * w * smm, ft = a * fp + w * fm;
        double q = 0.0;
        if (T > 0.0) q = (climb && k == top) ? -2.0 * ft / T : -ft / T + ks * (sqrt(spp) - sqrt(smm)) / sqrt(T);
        coef[2 * g] = q * a, coef[2 * g + 1] = q * w;
    }
}

__global__ void neb_project_kernel(float *__restrict__ force, const float *__restrict__ pos, const float *__restrict__ initial,
                                   const float *__restrict__ final_, const int *__restrict__ image, const int *__restrict__ image_ptr,
                                   const int *__restrict__ band_ptr, int K, const double *__restrict__ coef, int n_atoms) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_atoms) return;
    const int g = __ldg(image + i);
    const ImageNbrs nb = image_nbrs(g, K, image_ptr, band_ptr);
    double dp[3], dm[3];
    deltas(pos, initial, final_, nb, i, dp, dm);
    const double cp = __ldg(coef + 2 * (size_t)g), cm = __ldg(coef + 2 * (size_t)g + 1);
    float *f = force + 3 * (size_t)i;
#pragma unroll
    for (int c = 0; c < 3; ++c) f[c] = (float)((double)f[c] + cp * dp[c] + cm * dm[c]);
}

}  // namespace

extern "C" int64_t hn_neb_reduce_workspace_bytes(int64_t n_atoms, int32_t n_img) {
    if (n_atoms <= 0 || n_img <= 0) return 0;
    return (hn::reduce_chunks(n_atoms) + n_img) * (int64_t)sizeof(NebSums);
}

static int neb_layout_checks(const char *where, int32_t n_bands, int32_t n_images, int64_t n_atoms) {
    HN_REQUIRE(n_atoms >= 0 && n_atoms < (1ll << 31), where, "n_atoms must be in [0, 2^31)");
    HN_REQUIRE(n_bands >= 0 && n_images >= 1, where, "n_bands must be >= 0 and n_images >= 1");
    HN_REQUIRE((int64_t)n_bands * n_images < (1ll << 31), where, "n_bands * n_images must be < 2^31");
    return 0;
}

extern "C" int hn_neb_reduce(const float *pos, const float *force, const float *initial, const float *final_, const int32_t *image,
                             const int32_t *image_ptr, const int32_t *band_ptr, int32_t n_bands, int32_t n_images, int64_t n_atoms,
                             double *sums, void *workspace, int64_t workspace_bytes, void *stream) {
    if (neb_layout_checks("hn_neb_reduce", n_bands, n_images, n_atoms)) return 1;
    const int n_img = n_bands * n_images;
    if (n_img == 0 || n_atoms == 0) return 0;
    HN_REQUIRE(pos && force && initial && final_ && image && image_ptr && band_ptr && sums, "hn_neb_reduce", "null pointer");
    HN_REQUIRE(workspace && workspace_bytes >= hn_neb_reduce_workspace_bytes(n_atoms, n_img), "hn_neb_reduce",
               "workspace smaller than hn_neb_reduce_workspace_bytes");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t chunks = hn::reduce_chunks(n_atoms);
    NebSums *part = (NebSums *)workspace;
    neb_reduce_pieces_kernel<<<(unsigned)((chunks * 32 + 255) / 256), 256, 0, s>>>(pos, force, initial, final_, image, image_ptr,
                                                                                    band_ptr, n_images, (int)n_atoms, (int)chunks, part);
    HN_CUDA(cudaGetLastError(), "hn_neb_reduce");
    const int per = hn::reduce_slot_threads(chunks, n_img);
    neb_reduce_final_kernel<<<(unsigned)(((int64_t)n_img * per + 255) / 256), 256, 0, s>>>(part, image_ptr, n_img, per, sums);
    return hn::check_launch("hn_neb_reduce");
}

extern "C" int hn_neb_step(const double *sums, const float *energy, const float *end_energy, const double *spring, int32_t climb,
                           int32_t n_bands, int32_t n_images, double *coef, int32_t *imax, void *stream) {
    if (neb_layout_checks("hn_neb_step", n_bands, n_images, 0)) return 1;
    if (n_bands == 0) return 0;
    HN_REQUIRE(sums && energy && end_energy && spring && coef && imax, "hn_neb_step", "null pointer");
    neb_step_kernel<<<(unsigned)((n_bands + 127) / 128), 128, 0, (cudaStream_t)stream>>>(sums, energy, end_energy, spring, climb != 0,
                                                                                        n_bands, n_images, coef, imax);
    return hn::check_launch("hn_neb_step");
}

extern "C" int hn_neb_project(float *force, const float *pos, const float *initial, const float *final_, const int32_t *image,
                              const int32_t *image_ptr, const int32_t *band_ptr, int32_t n_bands, int32_t n_images,
                              const double *coef, int64_t n_atoms, void *stream) {
    if (neb_layout_checks("hn_neb_project", n_bands, n_images, n_atoms)) return 1;
    if (n_atoms == 0 || n_bands == 0) return 0;
    HN_REQUIRE(force && pos && initial && final_ && image && image_ptr && band_ptr && coef, "hn_neb_project", "null pointer");
    neb_project_kernel<<<(unsigned)((n_atoms + 255) / 256), 256, 0, (cudaStream_t)stream>>>(force, pos, initial, final_, image,
                                                                                            image_ptr, band_ptr, n_images, coef,
                                                                                            (int)n_atoms);
    return hn::check_launch("hn_neb_project");
}
