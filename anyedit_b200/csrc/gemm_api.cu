// anysd_gemm_f16: argument validation and kernel selection for every dense contraction on the path.
#include "common.cuh"

#include <stdlib.h>
#include <string.h>

namespace anysd {
int launch_gemm_mma(const anysd_gemm_params* q, cudaStream_t st);
int launch_gemm_tc5(const anysd_gemm_params* q, cudaStream_t st);
bool tc5_supported(const anysd_gemm_params* q);
int launch_gemm_tc5p(const anysd_gemm_params* q, cudaStream_t st);
bool tc5p_supported(const anysd_gemm_params* q);
int tc5p_stats_slabs(const anysd_gemm_params* q);
size_t tc5p_splitk_bytes(const anysd_gemm_params* q);
int tc5p_schedule(const anysd_gemm_params* q, int* ctas, int* bn, int* splits, int* ext, int* ln);
}

using namespace anysd;

enum { GEMM_MMA = 0, GEMM_TC5 = 1, GEMM_TC5P = 2 };

static int gemm_validate(const anysd_gemm_params* p) {
    ANYSD_REQUIRE(p != nullptr, ANYSD_EINVAL, "gemm: null params");
    ANYSD_REQUIRE(p->A && p->W && p->out, ANYSD_EINVAL, "gemm: null A/W/out");
    ANYSD_REQUIRE(p->M > 0 && p->N > 0 && p->K > 0, ANYSD_EINVAL, "gemm: bad M=%d N=%d K=%d", p->M, p->N, p->K);
    ANYSD_REQUIRE(p->K % 8 == 0 && p->ldw % 8 == 0 && p->ldw >= p->K, ANYSD_EINVAL,
                  "gemm: K=%d and ldw=%d must be multiples of 8 with ldw >= K", p->K, p->ldw);
    ANYSD_REQUIRE(((uintptr_t)p->A % 16) == 0 && ((uintptr_t)p->W % 16) == 0, ANYSD_EINVAL,
                  "gemm: A and W must be 16-byte aligned");
    ANYSD_REQUIRE(p->act >= 0 && p->act <= 4, ANYSD_EINVAL, "gemm: bad act %d", p->act);
    ANYSD_REQUIRE(p->out_dtype == ANYSD_F16 || p->out_dtype == ANYSD_F32, ANYSD_EINVAL, "gemm: bad out dtype");
    const int n_out = (p->act == 2) ? p->N / 2 : p->N;
    ANYSD_REQUIRE(p->act != 2 || p->N % 2 == 0, ANYSD_EINVAL, "gemm: GEGLU needs an even N");
    ANYSD_REQUIRE(p->ldo >= n_out, ANYSD_EINVAL, "gemm: ldo=%d < %d output columns", p->ldo, n_out);
    ANYSD_REQUIRE(!p->residual || p->ldr >= n_out, ANYSD_EINVAL, "gemm: ldr too small");
    ANYSD_REQUIRE(!p->rowadd || (p->rows_per_batch > 0 && p->ld_rowadd >= p->N), ANYSD_EINVAL,
                  "gemm: rowadd needs rows_per_batch > 0 and ld_rowadd >= N");
    if (p->conv) {
        ANYSD_REQUIRE(p->conv == 1, ANYSD_EINVAL, "gemm: conv must be 0 or 1 (3x3, pad 1)");
        ANYSD_REQUIRE(p->Nimg > 0 && p->H > 0 && p->Wd > 0 && p->Cin > 0 && p->Cin % 8 == 0, ANYSD_EINVAL,
                      "conv3x3: bad image dims N=%d H=%d W=%d Cin=%d (Cin must be a multiple of 8)", p->Nimg, p->H,
                      p->Wd, p->Cin);
        ANYSD_REQUIRE(p->stride == 1 || p->stride == 2, ANYSD_EINVAL, "conv3x3: stride must be 1 or 2");
        ANYSD_REQUIRE(p->upsample == 0 || p->upsample == 1, ANYSD_EINVAL, "conv3x3: upsample must be 0 or 1");
        ANYSD_REQUIRE(p->K == 9 * p->Cin, ANYSD_EINVAL, "conv3x3: K=%d != 9*Cin=%d", p->K, 9 * p->Cin);
        ANYSD_REQUIRE(p->conv_pad == 0 || (p->conv_pad == 1 && p->stride == 2 && !p->upsample), ANYSD_EINVAL,
                      "conv3x3: conv_pad must be 0, or 1 with stride 2 (right/bottom padding of the first-stage Downsample)");
        const int Hl = p->H << p->upsample, Wl = p->Wd << p->upsample;
        const int Ho = p->conv_pad ? (Hl - 2) / 2 + 1 : (Hl - 1) / p->stride + 1;
        const int Wo = p->conv_pad ? (Wl - 2) / 2 + 1 : (Wl - 1) / p->stride + 1;
        ANYSD_REQUIRE((long long)p->Nimg * Ho * Wo == p->M, ANYSD_EINVAL, "conv3x3: M=%d != N*Ho*Wo=%lld", p->M,
                      (long long)p->Nimg * Ho * Wo);
    } else {
        ANYSD_REQUIRE(p->lda % 8 == 0 && p->lda >= p->K, ANYSD_EINVAL, "gemm: lda=%d must be a multiple of 8 and >= K",
                      p->lda);
    }
    return ANYSD_OK;
}

// Kernel selection, shared by the launch and anysd_gemm_schedule: GEMM_MMA / GEMM_TC5 / GEMM_TC5P, or an error code (< 0) when the
// params ask for something only the persistent kernel can do and it cannot take them.
static int gemm_kernel(const anysd_gemm_params* p) {
    // Kernel selection.  The persistent tcgen05/TMA kernel (gemm_tc5p.cu) takes every fp16-output contraction
    // whose layout constraints hold: all nn.Linear / 1x1 convs and every 3x3 conv with Cin % 64 == 0 (stride 1|2,
    // upsample through the workspace).  The one-tile-per-CTA tcgen05 kernel (gemm_tc5.cu) takes the fp32-output
    // ones (time-embedding path).  mma.sync covers what is left: the Cin = 8 input conv and the N = 4 output conv.
    // ANYSD_GEMM=mma|tc5|tc5p is a test/debug switch used to cross-check the kernels against each other.
    static const char* force = getenv("ANYSD_GEMM");
    const bool allow_p = !force || !strcmp(force, "tc5p");
    const bool allow_1 = !force || !strcmp(force, "tc5");
    if (allow_p && tc5p_supported(p)) return GEMM_TC5P;
    ANYSD_REQUIRE(p->row_stats == nullptr && p->ln_stats == nullptr, ANYSD_EUNSUPPORTED,
                  "gemm: LayerNorm fold / row statistics need the persistent tcgen05 path");
    ANYSD_REQUIRE(p->stats == nullptr, ANYSD_EUNSUPPORTED, "gemm: output statistics need the persistent tcgen05 path");
    ANYSD_REQUIRE(!(p->conv && p->conv_pad), ANYSD_EUNSUPPORTED,
                  "conv3x3 with right/bottom padding needs the persistent tcgen05 path (fp16 output, Cin %% 64 == 0)");
    if ((allow_1 || (force && !strcmp(force, "tc5p"))) && tc5_supported(p)) return GEMM_TC5;
    return GEMM_MMA;
}

extern "C" int anysd_gemm_f16(const anysd_gemm_params* p, anysd_stream_t stream) {
    const int rc = gemm_validate(p);
    if (rc != ANYSD_OK) return rc;
    switch (const int k = gemm_kernel(p)) {
        case GEMM_TC5P: return launch_gemm_tc5p(p, (cudaStream_t)stream);
        case GEMM_TC5: return launch_gemm_tc5(p, (cudaStream_t)stream);
        case GEMM_MMA: return launch_gemm_mma(p, (cudaStream_t)stream);
        default: return k;
    }
}

extern "C" int anysd_gemm_schedule(const anysd_gemm_params* p, int* kernel, int* ctas, int* bn, int* splits, int* ext, int* ln) {
    const int rc = gemm_validate(p);
    if (rc != ANYSD_OK) return rc;
    const int k = gemm_kernel(p);
    if (k < 0) return k;
    int c = 0, w = 0, s = 0, x = 0, l = 0;
    if (k == GEMM_TC5P) {
        const int rs = tc5p_schedule(p, &c, &w, &s, &x, &l);
        if (rs != ANYSD_OK) return rs;
    }
    if (kernel) *kernel = k;
    if (ctas) *ctas = c;
    if (bn) *bn = w;
    if (splits) *splits = s;
    if (ext) *ext = x;
    if (ln) *ln = l;
    return ANYSD_OK;
}

extern "C" int anysd_gemm_stats_slabs(const anysd_gemm_params* p) {
    if (p == nullptr || !p->A || !p->W || !p->out) return 0;
    static const char* force = getenv("ANYSD_GEMM");
    if (force && strcmp(force, "tc5p")) return 0;
    if (p->conv && (p->Cin <= 0 || p->K != 9 * p->Cin)) return 0;
    return tc5p_supported(p) ? tc5p_stats_slabs(p) : 0;
}

extern "C" size_t anysd_gemm_splitk_workspace_bytes(const anysd_gemm_params* p) {
    if (p == nullptr || !p->A || !p->W || !p->out) return 0;
    static const char* force = getenv("ANYSD_GEMM");
    if (force && strcmp(force, "tc5p")) return 0;
    if (p->conv && (p->Cin <= 0 || p->K != 9 * p->Cin)) return 0;
    return tc5p_supported(p) ? tc5p_splitk_bytes(p) : 0;
}
