// libfastvithd_b200.so -- C ABI (include/fastvithd_b200.h) over the sm_100a kernels.
//
// Host side of the library: architecture plan of `fastvithd()` (mci.py:1454-1478), packed-weight
// table, workspace carving, TMA descriptor cache, launch sequence.  No torch, no CPU compute path.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "../../include/fastvithd_b200.h"
#include "dwconv.cuh"
#include "gemm_tcgen05.cuh"
#include "mlp_fused.cuh"
#include "mlp_cluster.cuh"
#include "preprocess.cuh"
#include "stem_attn_se.cuh"
#include "mixer_tc.cuh"
#include "mixer_umma.cuh"
#include "mixer_tc2.cuh"
#include "mixer_tz.cuh"
#include "stem2.cuh"
#include "llm.cuh"
#include "convffn.cuh"
#include "attention_umma.cuh"

using namespace fvhd;

namespace {

const int kLayers[5] = {2, 12, 24, 4, 2};           // mci.py:1457
const int kDims[5] = {96, 192, 384, 768, 1536};     // mci.py:1458
const int kSeRd = 192;                               // int(3072 * 0.0625), mci.py:49
std::string g_create_error;

struct WeightSpec { std::string name; int dtype; int64_t numel; };

struct RunCtx {
    int img_dtype;              // selects the stem instantiation; every pointer goes through the device IoBlock
};
typedef std::function<cudaError_t(cudaStream_t, const RunCtx&)> Step;

struct UnitDesc {
    std::string name;
    int kind;                   // 0 stem, 1 repmixer, 2 down, 3 cpe, 4 attn, 5 conv_exp, 6 projector
    int stage, block;
    int cin, cout, hin, win, hout, wout;
    int64_t in_elems, out_elems;
    double flops, min_bytes;
    std::string prefix;         // packed weight prefix
};

struct Plan {                   // launch sequence for one batch size
    int batch = 0;
    std::vector<Step> steps;
    std::vector<std::pair<int, int>> unit_steps;   // [begin, end) per unit
    std::vector<bf16*> unit_in, unit_out;          // workspace buffers per unit
    struct Info { const char* kernel; int unit; double flops; double bytes; };
    std::vector<Info> info;                        // one per step (== one kernel launch)
    IoBlock* io = nullptr;                         // device IO block of this plan (in the workspace)
    std::map<int, cudaGraphExec_t> graphs;         // key: img_dtype | last_step << 2 | copy_tokens << 20
    void add(const Step& s, const char* kernel, int unit, double flops, double bytes) {
        steps.push_back(s);
        info.push_back({kernel, unit, flops, bytes});
    }
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Kernel-selection switches.  read_options() reads them from the environment once per handle, in fvhd_create: a switch set
// after a handle exists does not affect that handle.  Defaults are the measured choices; the other values keep the alternatives
// selectable for A/B measurements and as references for the tests.
//
//   switch               values (default first)    selects
//   FVHD_NO_GRAPH        unset | 1                 1: forwards launch their steps one by one instead of replaying a captured CUDA graph
//   FVHD_NO_PDL          unset | 1                 1: plain stream order for every launch (no programmatic dependent launch)
//   FVHD_NO_SPLITK       unset | 1                 1: small-M GEMMs run one CTA per output tile (no k-slices)
//   FVHD_GEMM_CS         1 | 2 | 4                 GEMM cluster-size cap.  1: at batch 1 the delivered-bytes rate is the limit and multicast only
//                                                  reduces L2 reads -- measured no gain (profiles/r01_f_summary.md)
//   FVHD_NO_FUSED_MLP    unset | 1                 1: every ConvFFN as two GEMMs (reference path of the bit-exactness test); implies the next
//   FVHD_NO_CLUSTER_MLP  unset | 1                 1: the stage-2 (C = 384) ConvFFN never on the 4-CTA-cluster kernel (mlp_cluster.cuh)
//   FVHD_CONVFFN         2 | 1                     RepMixer ConvFFN.  2: convffn.cuh, except stage 2 at small batches (cluster kernel);
//                                                  1: mlp_fused.cuh (C <= 192), cluster kernel or two GEMMs (C = 384)
//   FVHD_CONVFFN_CS      1 | 2                     2: convffn.cuh as 2-CTA clusters sharing the weight stream by TMA multicast.  Bit-identical, but
//                                                  measured NEUTRAL at batch 32 (C = 384: 303.5 vs 304.0 us, C = 192: 383.7 vs 386.4 us per launch):
//                                                  the kernel is bound by its MMA1 -> GELU -> MMA2 chain, not by operand ingest
//   FVHD_MIXER           unset | z | t | 2 | u | f RepMixer depthwise pair.  unset: Toeplitz products on tcgen05 (mixer_tz.cuh) where a launch has
//                                                  at least one 64 x 32 x 8 item per SM, mixer_tc.cuh below that; z: Toeplitz everywhere; t: 7x7 on
//                                                  mma.sync (mixer_tc.cuh, the round-1 / early round-2 default); 2: both convs on mma.sync, 16 ch per
//                                                  CTA (mixer_tc2.cuh); u: tcgen05 diagonal taps (mixer_umma.cuh: correct, but smem-A-read bound --
//                                                  602 vs 434 us/img at batch 32, profiles/r02_*); f: FMA pipes (dwconv.cuh).
//                                                  fvhd_mixer: 2 -> tc2, t -> tc, unset or z -> tz, any other value -> umma
//   FVHD_MIX_TILE        unset | a | 8 | 1 | 5     set: the FMA-pipe kernels of dwconv.cuh, ahead of FVHD_MIXER.  a: automatic tile (8 x 16 below two
//                                                  CTAs per SM); 8: 8 x 16 / 128 thr; 1: 16 x 16 / 256 thr; 5: 16 x 16 / 512 thr; other values: as t
//                                                  (as f under FVHD_MIXER=f)
//   FVHD_TZ_PAIR         2 | 1..8                  Toeplitz mixer sibling-cluster size (1: plain launch), halved until it divides the channel groups
//   FVHD_TZ_PDL          3 | 0..3                  Toeplitz mixer: bit 0 = launch with the PDL attribute, bit 1 = trigger the successor early
//   FVHD_TZ_SKIP         0 | 1..15                 Toeplitz mixer timing experiments: work the kernel skips (MixZParams::dbg)
//   FVHD_ATTN            a | u | m                 MHSA core.  a: tcgen05 / TMEM (attention_umma.cuh) from 512 tokens, mma.sync below; u / m force
//                                                  one.  fvhd_attention: u -> tcgen05, any other value -> mma.sync
//   FVHD_STEM            2 | 1                     2: stem2.cuh (persistent, packed-half GELUs, 16-B patch loads); 1: first-generation stem_kernel
//   FVHD_LLM_ATTN        unset | f                 LLM prefill attention.  unset: causal_attn_mma_kernel; f: FMA pipes (first version)
//   FVHD_DEBUG_PLAN      unset | any               set: every GEMM configuration is printed to stderr as a plan is built
struct Options {
    bool graph = true, pdl = true, splitk = true, fused_mlp = true, cluster_mlp = true, llm_attn_fma = false, debug_plan = false;
    int gemm_max_cs = 1, convffn_gen = 2, convffn_cs = 1, stem_gen = 2, tz_pair = 2, tz_pdl = 3, tz_skip = 0;
    char attn = 'a';
    char mixer = 0;             // 0: unset (automatic choice per launch); an empty value reads as 'z'
    char mix_tile = 0;          // 0: unset; an empty value reads as '?' (set, no tile letter)
};

Options read_options() {
    Options o;
    auto one = [](const char* name) { const char* e = getenv(name); return e && e[0] == '1'; };
    o.graph = !one("FVHD_NO_GRAPH");
    o.pdl = !one("FVHD_NO_PDL");
    o.splitk = !one("FVHD_NO_SPLITK");
    o.fused_mlp = !one("FVHD_NO_FUSED_MLP");
    o.cluster_mlp = o.fused_mlp && !one("FVHD_NO_CLUSTER_MLP");
    const char* e;
    if ((e = getenv("FVHD_GEMM_CS")) && (e[0] == '1' || e[0] == '2' || e[0] == '4')) o.gemm_max_cs = e[0] - '0';
    if ((e = getenv("FVHD_CONVFFN")) && (e[0] == '1' || e[0] == '2')) o.convffn_gen = e[0] - '0';
    if ((e = getenv("FVHD_CONVFFN_CS")) && (e[0] == '1' || e[0] == '2')) o.convffn_cs = e[0] - '0';
    if ((e = getenv("FVHD_MIXER"))) o.mixer = e[0] ? e[0] : 'z';
    if ((e = getenv("FVHD_MIX_TILE"))) o.mix_tile = e[0] ? e[0] : '?';
    if ((e = getenv("FVHD_TZ_PAIR")) && e[0] >= '0' && e[0] <= '8') o.tz_pair = e[0] > '0' ? e[0] - '0' : 1;
    if ((e = getenv("FVHD_TZ_PDL"))) o.tz_pdl = atoi(e);
    if ((e = getenv("FVHD_TZ_SKIP"))) o.tz_skip = atoi(e);
    if ((e = getenv("FVHD_ATTN")) && e[0]) o.attn = e[0];
    o.stem_gen = one("FVHD_STEM") ? 1 : 2;
    o.llm_attn_fma = (e = getenv("FVHD_LLM_ATTN")) && e[0] == 'f';
    o.debug_plan = getenv("FVHD_DEBUG_PLAN") != nullptr;
    return o;
}

}  // namespace

// LLM prefill engine attached to a handle (row f3): caller-owned weights, library-owned activations / KV cache, one plan per length.
struct LlmState {
    fvhd_llm_config c{};
    int nqkv = 0;                       // (heads + 2 kv_heads) * head_dim
    std::vector<const void*> w;         // 7 per layer + final norm + lm_head
    bf16 *x0 = nullptr, *x1 = nullptr, *x2 = nullptr, *xn = nullptr;      // x0: the caller's input (never written by a prefill)
    bf16 *qkv = nullptr, *att = nullptr, *gu = nullptr, *hm = nullptr, *logits = nullptr;
    bf16 *kc = nullptr, *vc = nullptr;  // [layers][max_seq][kv_heads * head_dim]
    float2* rope = nullptr;             // [max_seq][head_dim / 2]
    int* token = nullptr;
    std::map<int, Plan> plans;          // key: sequence length
};

struct fvhd_handle_s {
    LlmState* llm = nullptr;
    fvhd_config cfg;
    Options opt;
    std::string err;
    int R = 0, ntok = 0;
    std::vector<WeightSpec> specs;
    std::vector<UnitDesc> units;
    std::map<std::string, const void*> wptr;
    bool loaded = false;
    bool cuda_ready = false;
    void* ws = nullptr;
    size_t ws_bytes = 0;
    EncodeTiledFn encode = nullptr;
    int num_sms = 148;
    int cf_clusters[3] = {0, 0, 0};   // resident 2-CTA clusters of convffn_tcgen05_kernel<C, 2>, C = 96 / 192 / 384
    int tz_clusters[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // [cs]: resident cs-CTA clusters of repmixer_tz_kernel (cs = 2, 4, 8)
    int mlpc_clusters = 0;        // resident 4-CTA clusters of mlp_cluster_tcgen05_kernel (cudaOccupancyMaxActiveClusters)
    cudaStream_t cap_stream = nullptr;   // private stream used only to capture graphs (the legacy default stream cannot be captured)
    std::map<int, Plan> plans;
    int64_t act0 = 0;           // elements of the largest activation per image: (R/4)^2 * 96
    void *stage_in = nullptr, *stage_out = nullptr;   // fvhd_encode_images_host device staging
    // row f1 (preprocess): device coefficient tables cached per (in_size, out_size), horizontal-pass scratch, 1/255 LUT
    struct RsTable { int* bounds; int* kk; int ksize; };
    std::map<std::pair<int, int>, RsTable> rs_tables;
    uint8_t* rs_tmp = nullptr; size_t rs_tmp_bytes = 0;
    uint8_t* rs_src = nullptr; size_t rs_src_bytes = 0;
    float* rs_lut = nullptr;
    size_t stage_in_bytes = 0, stage_out_bytes = 0;
    float* splitk_ws = nullptr;     // split-K partial tiles (GEMM_SPLITK_WS_BYTES) + per-tile arrival counters, owned by the handle
    int* splitk_cnt = nullptr;
};

namespace {

int fail(fvhd_handle h, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define CUDA_TRY(h, expr)                                                                      \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess) return fail(h, FVHD_ERR_CUDA, "%s -> %s", #expr, cudaGetErrorString(e__)); \
    } while (0)

void add_spec(fvhd_handle h, const std::string& n, int dt, int64_t numel) { h->specs.push_back({n, dt, numel}); }

void add_convffn_specs(fvhd_handle h, const std::string& p, int c, bool f16_fc2 = false) {
    add_spec(h, p + "dw.w", FVHD_F32, 49LL * c);
    add_spec(h, p + "dw.b", FVHD_F32, c);
    add_spec(h, p + "fc1.w", FVHD_BF16, 4LL * c * c);
    add_spec(h, p + "fc1.b", FVHD_F32, 4LL * c);
    add_spec(h, p + "fc2.w", FVHD_BF16, 4LL * c * c);
    if (f16_fc2) add_spec(h, p + "fc2.wh", FVHD_F16, 4LL * c * c);      // f16 copy of fc2.w for the f16-hidden fused ConvFFN kernel (convffn.cuh)
    add_spec(h, p + "fc2.b", FVHD_F32, c);
}

// Architecture walk of FastViT.__init__ (mci.py:1353-1411) for `fastvithd`.
void build_arch(fvhd_handle h) {
    const int R = h->R;
    const int H = h->cfg.projector_hidden;
    int hw = R / 4;
    h->act0 = (int64_t)hw * hw * 96;
    {   // convolutional_stem (mci.py:553-603)
        UnitDesc u{};
        u.name = "stem"; u.kind = 0; u.cin = 3; u.cout = 96; u.hin = u.win = R; u.hout = u.wout = hw;
        u.in_elems = 3LL * R * R; u.out_elems = (int64_t)hw * hw * 96;
        const double macs = (double)(R / 2) * (R / 2) * 96 * 27 + (double)hw * hw * 96 * 9 + (double)hw * hw * 96 * 96;
        u.flops = 2 * macs;
        u.min_bytes = (u.in_elems + u.out_elems) * 2.0 + (27 * 96 + 9 * 96) * 4 + 96 * 96 * 2;
        u.prefix = "stem.";
        h->units.push_back(u);
        add_spec(h, "stem.w0", FVHD_F32, 27 * 96); add_spec(h, "stem.b0", FVHD_F32, 96);
        add_spec(h, "stem.w1", FVHD_F32, 9 * 96);  add_spec(h, "stem.b1", FVHD_F32, 96);
        add_spec(h, "stem.w2", FVHD_BF16, 96 * 96); add_spec(h, "stem.b2", FVHD_F32, 96);
    }
    int idx = 0;
    for (int i = 0; i < 5; ++i) {
        const int c = kDims[i];
        const int64_t px = (int64_t)hw * hw;
        if (i >= 3) {   // RepCPE (mci.py:971-980)
            UnitDesc u{};
            u.name = "network." + std::to_string(idx); u.kind = 3; u.stage = i;
            u.cin = u.cout = c; u.hin = u.win = u.hout = u.wout = hw;
            u.in_elems = u.out_elems = px * c;
            u.flops = 2.0 * px * c * 49; u.min_bytes = 4.0 * px * c + 50.0 * c * 4;
            u.prefix = u.name + ".";
            h->units.push_back(u);
            add_spec(h, u.prefix + "dw.w", FVHD_F32, 49LL * c); add_spec(h, u.prefix + "dw.b", FVHD_F32, c);
            ++idx;
        }
        for (int b = 0; b < kLayers[i]; ++b) {
            UnitDesc u{};
            u.name = "network." + std::to_string(idx) + "." + std::to_string(b);
            u.stage = i; u.block = b; u.cin = u.cout = c; u.hin = u.win = u.hout = u.wout = hw;
            u.in_elems = u.out_elems = px * c;
            u.prefix = u.name + ".";
            double macs = (double)px * c * 49 + 2.0 * px * c * 4 * c;
            double wbytes = 8.0 * c * c * 2 + (49.0 * c + 6 * c) * 4;
            if (i < 3) {    // RepMixerBlock (mci.py:1042-1113)
                u.kind = 1;
                macs += (double)px * c * 9;
                wbytes += 10.0 * c * 4;
                add_spec(h, u.prefix + "mix.w", FVHD_F32, 9LL * c); add_spec(h, u.prefix + "mix.b", FVHD_F32, c);
            } else {        // AttentionBlock (mci.py:1116-1192)
                u.kind = 4;
                macs += (double)px * c * 3 * c + (double)px * c * c + 2.0 * px * px * c;
                wbytes += 4.0 * c * c * 2 + 3.0 * c * 4;
                add_spec(h, u.prefix + "ln.w", FVHD_F32, c); add_spec(h, u.prefix + "ln.b", FVHD_F32, c);
                add_spec(h, u.prefix + "qkv.w", FVHD_BF16, 3LL * c * c);
                add_spec(h, u.prefix + "proj.w", FVHD_BF16, (int64_t)c * c); add_spec(h, u.prefix + "proj.b", FVHD_F32, c);
            }
            add_convffn_specs(h, u.prefix, c, i < 3);
            u.flops = 2 * macs; u.min_bytes = 4.0 * px * c + wbytes;
            h->units.push_back(u);
        }
        ++idx;
        if (i < 4) {    // PatchEmbed (mci.py:688-741)
            const int co = kDims[i + 1];
            UnitDesc u{};
            u.name = "network." + std::to_string(idx); u.kind = 2; u.stage = i;
            u.cin = c; u.cout = co; u.hin = u.win = hw; u.hout = u.wout = hw / 2;
            const int64_t opx = (int64_t)(hw / 2) * (hw / 2);
            u.in_elems = px * c; u.out_elems = opx * co;
            u.flops = 2.0 * (opx * co * 49.0 + (double)opx * co * co);
            u.min_bytes = 2.0 * (u.in_elems + u.out_elems) + (double)co * co * 2 + 51.0 * co * 4;
            u.prefix = u.name + ".";
            h->units.push_back(u);
            add_spec(h, u.prefix + "dw.w", FVHD_F32, 49LL * co); add_spec(h, u.prefix + "dw.b", FVHD_F32, co);
            add_spec(h, u.prefix + "pw.w", FVHD_BF16, (int64_t)co * co); add_spec(h, u.prefix + "pw.b", FVHD_F32, co);
            ++idx;
            hw /= 2;
        }
    }
    {   // conv_exp + SE (mci.py:1401-1411, 42-81) -> tokens [HW, 3072] (feature_select, mobileclip_encoder.py:60-68)
        UnitDesc u{};
        const int64_t px = (int64_t)hw * hw;
        u.name = "conv_exp"; u.kind = 5; u.cin = 1536; u.cout = 3072; u.hin = u.win = u.hout = u.wout = hw;
        u.in_elems = px * 1536; u.out_elems = px * 3072;
        u.flops = 2.0 * (px * 3072.0 * 9 + 2.0 * 3072 * kSeRd);
        u.min_bytes = 2.0 * (u.in_elems + u.out_elems) + 2.0 * 3072 * kSeRd * 2 + 3072.0 * 11 * 4;
        u.prefix = "conv_exp.";
        h->units.push_back(u);
        add_spec(h, "conv_exp.dw.w", FVHD_F32, 9 * 3072); add_spec(h, "conv_exp.dw.b", FVHD_F32, 3072);
        add_spec(h, "conv_exp.se.r.w", FVHD_BF16, (int64_t)kSeRd * 3072); add_spec(h, "conv_exp.se.r.b", FVHD_F32, kSeRd);
        add_spec(h, "conv_exp.se.e.w", FVHD_BF16, (int64_t)3072 * kSeRd); add_spec(h, "conv_exp.se.e.b", FVHD_F32, 3072);
    }
    if (H > 0) {    // mlp{N}x_gelu (multimodal_projector/builder.py:23-30)
        UnitDesc u{};
        const int64_t px = (int64_t)hw * hw;
        u.name = "projector"; u.kind = 6; u.cin = 3072; u.cout = H; u.hin = u.win = u.hout = u.wout = hw;
        u.in_elems = px * 3072; u.out_elems = px * H;
        double macs = (double)px * 3072 * H, wb = 3072.0 * H * 2 + H * 4.0;
        add_spec(h, "projector.0.w", FVHD_BF16, 3072LL * H); add_spec(h, "projector.0.b", FVHD_F32, H);
        if (h->cfg.projector_depth == 2) {
            macs += (double)px * H * H; wb += (double)H * H * 2 + H * 4.0;
            add_spec(h, "projector.2.w", FVHD_BF16, (int64_t)H * H); add_spec(h, "projector.2.b", FVHD_F32, H);
        }
        u.flops = 2 * macs; u.min_bytes = 2.0 * (u.in_elems + u.out_elems) + wb;
        u.prefix = "projector.";
        h->units.push_back(u);
    }
}

// ------------------------------------------------------------------ workspace carving
struct Buffers {
    bf16 *X0, *X1, *Y, *Z, *T1, *H4;
    float *pooled, *sr;
    IoBlock* io;
};
size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
size_t workspace_bytes(fvhd_handle h, int batch) {
    const size_t a = align_up((size_t)h->act0 * batch * 2, 1024);
    return 9 * a + align_up((size_t)batch * 3072 * 4, 1024) + align_up((size_t)batch * kSeRd * 4, 1024) + 1024 /*io block*/ + 1024;
}
Buffers carve(fvhd_handle h, int batch) {
    const size_t a = align_up((size_t)h->act0 * batch * 2, 1024);
    uint8_t* p = reinterpret_cast<uint8_t*>(align_up((size_t)h->ws, 1024));
    Buffers b;
    b.X0 = (bf16*)p; p += a;
    b.X1 = (bf16*)p; p += a;
    b.Y = (bf16*)p; p += a;
    b.Z = (bf16*)p; p += a;
    b.T1 = (bf16*)p; p += a;
    b.H4 = (bf16*)p; p += 4 * a;
    b.pooled = (float*)p; p += align_up((size_t)batch * 3072 * 4, 1024);
    b.sr = (float*)p; p += align_up((size_t)batch * kSeRd * 4, 1024);
    b.io = (IoBlock*)p;
    return b;
}

// ------------------------------------------------------------------ launches
// All kernels go through cudaLaunchKernelEx, with programmatic stream serialization (PDL) unless FVHD_NO_PDL: a kernel may begin
// its prologue while the previous one drains; the kernels themselves order their global accesses with pdl_wait().
const size_t kSplitKWsBytes = 32u << 20;
const int kSplitKTiles = 4096;
// Debug-only, process-wide state of fvhd_debug_gemm_trace (the hook takes no handle).
unsigned long long* g_gemm_trace = nullptr;   // device buffer, 16 stamps per CTA
int g_force_bn = 0;                            // force the N tile (0 = cost model)
int g_debug_gemm_cs = 0;                       // cluster-size cap ahead of the handle's FVHD_GEMM_CS (0 = not set)
template <typename... KArgs, typename... Args>
cudaError_t launch_kc(bool pdl, int cluster, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[2];
    int n = 0;
    if (pdl) {
        at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[n].val.programmaticStreamSerializationAllowed = 1;
        ++n;
    }
    if (cluster > 1) {
        at[n].id = cudaLaunchAttributeClusterDimension;
        at[n].val.clusterDim.x = (unsigned)cluster;
        at[n].val.clusterDim.y = 1;
        at[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = at;
    cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
template <typename... KArgs, typename... Args>
cudaError_t launch_k(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    return launch_kc(pdl, 1, kernel, grid, block, smem, st, args...);
}

// ------------------------------------------------------------------ CUDA lazy init
template <typename K> cudaError_t set_smem(K kernel, size_t bytes) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// How many cs-CTA clusters of `kernel` can be resident at once (clusters are placed per GPC); 0 when the query fails.
template <typename K> int resident_clusters(K kernel, int cs, int threads, size_t smem, int num_sms) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(num_sms / cs * cs));
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, kernel, &cfg) != cudaSuccess) { nc = 0; (void)cudaGetLastError(); }
    return nc;
}

int ensure_cuda(fvhd_handle h) {
    if (h->cuda_ready) return FVHD_OK;
    int dev = 0;
    CUDA_TRY(h, cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CUDA_TRY(h, cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10) return fail(h, FVHD_ERR_CUDA, "device is sm_%d%d; this library is sm_100a only", prop.major, prop.minor);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CUDA_TRY(h, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) return fail(h, FVHD_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    h->encode = reinterpret_cast<EncodeTiledFn>(fn);
    const int n = h->num_sms = prop.multiProcessorCount;
    CUDA_TRY(h, set_smem(gemm_bf16_tcgen05_kernel, 227 * 1024));
    CUDA_TRY(h, set_smem(mlp_fused_tcgen05_kernel, 227 * 1024));
    CUDA_TRY(h, set_smem(mlp_cluster_tcgen05_kernel, MLPC_SMEM));
    h->mlpc_clusters = resident_clusters(mlp_cluster_tcgen05_kernel, MLPC_CS, MLPC_THREADS, MLPC_SMEM, n);
    CUDA_TRY(h, set_smem(repmixer_dw_kernel<16, 16, 256>, MixCfgT<16, 16>::SMEM));
    CUDA_TRY(h, set_smem(repmixer_dw_kernel<8, 16, 128>, MixCfgT<8, 16>::SMEM));
    CUDA_TRY(h, set_smem(repmixer_dw_kernel<16, 16, 512, 6, 4, 2>, MixCfgT<16, 16>::SMEM));
    CUDA_TRY(h, set_smem(repmixer_tc_kernel, MixTc::SMEM));
    CUDA_TRY(h, set_smem(repmixer_umma_kernel, MixU::SMEM));
    CUDA_TRY(h, set_smem(repmixer_tc2_kernel, MixT2::SMEM));
    CUDA_TRY(h, set_smem(repmixer_tz_kernel, MixZ::SMEM));
    for (int cs = 2; cs <= 8; cs *= 2) h->tz_clusters[cs] = resident_clusters(repmixer_tz_kernel, cs, MixZ::THREADS, MixZ::SMEM, n);
    CUDA_TRY(h, set_smem(attention_umma_kernel, AttU::SMEM));
    CUDA_TRY(h, (set_smem(convffn_tcgen05_kernel<96, 1>, CfCfg<96>::SMEM)));
    CUDA_TRY(h, (set_smem(convffn_tcgen05_kernel<192, 1>, CfCfg<192>::SMEM)));
    CUDA_TRY(h, (set_smem(convffn_tcgen05_kernel<384, 1>, CfCfg<384>::SMEM)));
    CUDA_TRY(h, (set_smem(convffn_tcgen05_kernel<96, 2>, CfCfg<96>::SMEM)));
    CUDA_TRY(h, (set_smem(convffn_tcgen05_kernel<192, 2>, CfCfg<192>::SMEM)));
    CUDA_TRY(h, (set_smem(convffn_tcgen05_kernel<384, 2>, CfCfg<384>::SMEM)));
    h->cf_clusters[0] = resident_clusters(convffn_tcgen05_kernel<96, 2>, 2, CF_THREADS, CfCfg<96>::SMEM, n);
    h->cf_clusters[1] = resident_clusters(convffn_tcgen05_kernel<192, 2>, 2, CF_THREADS, CfCfg<192>::SMEM, n);
    h->cf_clusters[2] = resident_clusters(convffn_tcgen05_kernel<384, 2>, 2, CF_THREADS, CfCfg<384>::SMEM, n);
    CUDA_TRY(h, set_smem(dwconv_kernel<7, 1, 1, 0, 16, 16, 8>, DwCfg<7, 1, 1, 16, 16>::SMEM));
    CUDA_TRY(h, set_smem(dwconv_kernel<7, 1, 1, 0, 8, 16, 8>, DwCfg<7, 1, 1, 8, 16>::SMEM));
    CUDA_TRY(h, set_smem(dwconv_kernel<7, 2, 2, 1, 8, 8, 4>, DwCfg<7, 2, 2, 8, 8>::SMEM));
    CUDA_TRY(h, set_smem(dwconv_kernel<3, 1, 2, 0, 16, 16, 8>, DwCfg<3, 1, 2, 16, 16>::SMEM));
    CUDA_TRY(h, set_smem(stem_kernel<float>, STEM_SMEM));
    CUDA_TRY(h, set_smem(stem_kernel<__half>, STEM_SMEM));
    CUDA_TRY(h, set_smem(stem_kernel<bf16>, STEM_SMEM));
    CUDA_TRY(h, set_smem(stem2_kernel<float>, Stem2::SMEM));
    CUDA_TRY(h, set_smem(stem2_kernel<__half>, Stem2::SMEM));
    CUDA_TRY(h, set_smem(stem2_kernel<bf16>, Stem2::SMEM));
    CUDA_TRY(h, cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
    CUDA_TRY(h, cudaMalloc(&h->splitk_ws, kSplitKWsBytes));
    CUDA_TRY(h, cudaMalloc(&h->splitk_cnt, kSplitKTiles * sizeof(int)));
    CUDA_TRY(h, cudaMemset(h->splitk_cnt, 0, kSplitKTiles * sizeof(int)));
    h->cuda_ready = true;
    return FVHD_OK;
}

// bf16 row-major [rows, K] matrix with row pitch `ld` elements -> 2-D tensor map, box {64, box_rows}, 128-B swizzle.
int make_tmap(fvhd_handle h, CUtensorMap* m, const void* ptr, int64_t rows, int64_t K, int64_t ld, int box_rows, int box_cols = GEMM_BK,
              CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
    if (((uintptr_t)ptr & 15) || (ld * 2) % 16) return fail(h, FVHD_ERR_INVALID, "TMA operand must be 16-B aligned (ptr %p, ld %lld)", ptr, (long long)ld);
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = h->encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, FVHD_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%lld K=%lld ld=%lld box=%d", (int)r,
                                       (long long)rows, (long long)K, (long long)ld, box_rows);
    return FVHD_OK;
}

// NHWC bf16 activation [B, H, W, C] -> 4-D tensor map, box {32 channels, box_w, box_h, 1}, no swizzle, zero OOB fill.
int make_tmap_nhwc(fvhd_handle h, CUtensorMap* m, const void* ptr, int B, int H, int W, int C, int box_w, int box_h, int box_c = DW_CG) {
    if ((uintptr_t)ptr & 15) return fail(h, FVHD_ERR_INVALID, "TMA operand must be 16-B aligned (ptr %p)", ptr);
    if (box_w > 256 || box_h > 256) return fail(h, FVHD_ERR_INVALID, "TMA box %dx%d too large", box_w, box_h);
    cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
    cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = h->encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, FVHD_ERR_CUDA, "cuTensorMapEncodeTiled(4D) failed (%d) B=%d H=%d W=%d C=%d box=%dx%d", (int)r, B, H, W, C, box_w, box_h);
    return FVHD_OK;
}

// NHWC bf16 activation [B, H, W, C] viewed as {8 ch, W, H, C/8, B} -> 5-D tensor map, box {8, box_w, box_h, 2 chunks, 1}: lands in smem
// as [8-channel chunk][row][x][8 ch] -- the no-swizzle K-major core-matrix layout of mixer_umma.cuh.  Zero OOB fill.
int make_tmap_chunked(fvhd_handle h, CUtensorMap* m, const void* ptr, int B, int H, int W, int C, int box_w, int box_h) {
    if ((uintptr_t)ptr & 15) return fail(h, FVHD_ERR_INVALID, "TMA operand must be 16-B aligned (ptr %p)", ptr);
    cuuint64_t dims[5] = {8, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)(C / 8), (cuuint64_t)B};
    cuuint64_t strides[4] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, 16, (cuuint64_t)H * W * C * 2};
    cuuint32_t box[5] = {8, (cuuint32_t)box_w, (cuuint32_t)box_h, 2, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = h->encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(ptr), dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(h, FVHD_ERR_CUDA, "cuTensorMapEncodeTiled(5D) failed (%d) B=%d H=%d W=%d C=%d box=%dx%d", (int)r, B, H, W, C, box_w, box_h);
    return FVHD_OK;
}

// RepMixer depthwise pair on tcgen05 (mixer_umma.cuh): persistent CTAs, two per SM, each bound to one 16-channel group.
int make_mixer_umma_step(fvhd_handle h, Step* st, const bf16* x, bf16* y, bf16* z, const float* w3, const float* b3, const float* w7,
                         const float* b7, int batch, int H, int W, int C) {
    if (C % 16) return fail(h, FVHD_ERR_INVALID, "tcgen05 mixer needs C %% 16 == 0 (got %d)", C);
    MixUParams mp{};
    mp.y = y; mp.z = z; mp.w3 = w3; mp.b3 = b3; mp.w7 = w7; mp.b7 = b7;
    mp.B = batch; mp.H = H; mp.W = W; mp.C = C;
    mp.tiles_x = (W + MixU::TOW - 1) / MixU::TOW;
    mp.tiles_y = (H + MixU::TOH - 1) / MixU::TOH;
    mp.groups = C / MixU::CG;
    const int n_sp = batch * mp.tiles_x * mp.tiles_y;
    int per = (2 * h->num_sms) / mp.groups;             // two CTAs per SM
    if (per < 1) per = 1;
    if (per > n_sp) per = n_sp;
    mp.ctas_per_group = per;
    CUtensorMap tm;
    int rc = make_tmap_chunked(h, &tm, x, batch, H, W, C, MixU::P, MixU::XH);
    if (rc != FVHD_OK) return rc;
    const dim3 grid((unsigned)(per * mp.groups));
    const bool pdl = h->opt.pdl;
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_k(pdl, repmixer_umma_kernel, grid, dim3(MixU::THREADS), MixU::SMEM, s, tm, mp);
    };
    return FVHD_OK;
}

// RepMixer depthwise pair with the 7x7 on mma.sync (mixer_tc.cuh): persistent CTAs, ~two per SM in total, each bound to one
// 32-channel group and walking that group's (image, 16 x 16 tile) items.
int make_mixer_tc_step(fvhd_handle h, Step* st, const bf16* x, bf16* y, bf16* z, const float* w3, const float* b3, const float* w7,
                       const float* b7, int batch, int H, int W, int C) {
    if (C % DW_CG) return fail(h, FVHD_ERR_INVALID, "mma.sync mixer needs C %% 32 == 0 (got %d)", C);
    const int tx = (W + 15) / 16, ty = (H + 15) / 16;
    int per_group = (2 * h->num_sms) / (C / DW_CG);       // floor: a CTA beyond the resident slots would run its whole item loop as a second wave
    if (per_group < 1) per_group = 1;
    if (per_group > tx * ty * batch) per_group = tx * ty * batch;
    const dim3 grid(per_group, C / DW_CG, 1);
    CUtensorMap tm;
    int rc = make_tmap_nhwc(h, &tm, x, batch, H, W, C, MixTc::XP, MixTc::XH);
    if (rc != FVHD_OK) return rc;
    const bool pdl = h->opt.pdl;
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_k(pdl, repmixer_tc_kernel, grid, dim3(MixTc::NT), MixTc::SMEM, s, tm, y, z, w3, b3, w7, b7, H, W, C, tx, batch);
    };
    return FVHD_OK;
}

// RepMixer depthwise pair with both convs on mma.sync, 16 channels per CTA (mixer_tc2.cuh).
int make_mixer_tc2_step(fvhd_handle h, Step* st, const bf16* x, bf16* y, bf16* z, const float* w3, const float* b3, const float* w7,
                        const float* b7, int batch, int H, int W, int C) {
    if (C % MixT2::CG) return fail(h, FVHD_ERR_INVALID, "mma.sync mixer (16-channel groups) needs C %% 16 == 0 (got %d)", C);
    const int tx = (W + MixT2::TOW - 1) / MixT2::TOW, ty = (H + MixT2::TOH - 1) / MixT2::TOH;
    const dim3 grid(tx * ty, C / MixT2::CG, batch);
    CUtensorMap tm;
    int rc = make_tmap_nhwc(h, &tm, x, batch, H, W, C, MixT2::XP, MixT2::XH, MixT2::CG);
    if (rc != FVHD_OK) return rc;
    const bool pdl = h->opt.pdl;
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_k(pdl, repmixer_tc2_kernel, grid, dim3(MixT2::NT), MixT2::SMEM, s, tm, y, z, w3, b3, w7, b7, H, W, C, tx);
    };
    return FVHD_OK;
}

// RepMixer depthwise pair on the FMA pipes (dwconv.cuh), one CTA per (tile, 32-channel group, image); the tile per FVHD_MIX_TILE.
int make_mixer_dw_step(fvhd_handle h, Step* st, const bf16* x, bf16* y, bf16* z, const float* w3, const float* b3, const float* w7,
                       const float* b7, int batch, int H, int W, int C) {
    if (C % DW_CG) return fail(h, FVHD_ERR_INVALID, "FMA-pipe mixer needs C %% 32 == 0 (got %d)", C);
    const long ctas16 = (long)((W + 15) / 16) * ((H + 15) / 16) * (C / DW_CG) * batch;
    const char t = h->opt.mix_tile;
    const bool small = t == '8' || (t == 'a' && ctas16 < 2L * h->num_sms), wide = t == '5';
    const int TH = small ? 8 : 16;
    const int tx = (W + 15) / 16, ty = (H + TH - 1) / TH;
    const dim3 grid(tx * ty, C / DW_CG, batch);
    CUtensorMap tm;
    int rc = make_tmap_nhwc(h, &tm, x, batch, H, W, C, small ? MixCfgT<8, 16>::XP : MixCfgT<16, 16>::XP,
                            small ? MixCfgT<8, 16>::XH : MixCfgT<16, 16>::XH);
    if (rc != FVHD_OK) return rc;
    const bool pdl = h->opt.pdl;
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        if (wide) return launch_k(pdl, repmixer_dw_kernel<16, 16, 512, 6, 4, 2>, grid, dim3(512), MixCfgT<16, 16>::SMEM, s, tm, y, z, w3, b3, w7, b7, H, W, C, tx);
        if (small) return launch_k(pdl, repmixer_dw_kernel<8, 16, 128>, grid, dim3(128), MixCfgT<8, 16>::SMEM, s, tm, y, z, w3, b3, w7, b7, H, W, C, tx);
        return launch_k(pdl, repmixer_dw_kernel<16, 16, 256>, grid, dim3(256), MixCfgT<16, 16>::SMEM, s, tm, y, z, w3, b3, w7, b7, H, W, C, tx);
    };
    return FVHD_OK;
}

// RepMixer depthwise pair with the 7x7 as Toeplitz products on tcgen05 (mixer_tz.cuh): one persistent CTA per SM, each bound to one
// 8-channel group and walking that group's (image, 64 x 32 tile) items.
int make_mixer_tz_step(fvhd_handle h, Step* st, const bf16* x, bf16* y, bf16* z, const float* w3, const float* b3, const float* w7,
                       const float* b7, int batch, int H, int W, int C) {
    if (C % MixZ::CG) return fail(h, FVHD_ERR_INVALID, "Toeplitz tcgen05 mixer needs C %% 8 == 0 (got %d)", C);
    MixZParams mp{};
    mp.y = y; mp.z = z; mp.w3 = w3; mp.b3 = b3; mp.w7 = w7; mp.b7 = b7;
    mp.B = batch; mp.H = H; mp.W = W; mp.C = C;
    mp.tiles_x = (W + MixZ::ZC - 1) / MixZ::ZC;
    mp.tiles_y = (H + MixZ::ZR - 1) / MixZ::ZR;
    mp.groups = C / MixZ::CG;
    const int n_sp = batch * mp.tiles_x * mp.tiles_y;
    int cs = h->opt.tz_pair;                            // sibling clusters: must divide the number of channel groups
    while (cs > 1 && (mp.groups % cs || h->tz_clusters[cs] <= 0)) cs >>= 1;
    mp.pair_sync = cs > 1 ? cs : 0;
    int slots = cs > 1 ? h->tz_clusters[cs] * cs : h->num_sms;      // resident CTAs (one per SM; clusters are placed per GPC)
    if (slots > h->num_sms) slots = h->num_sms;
    int per = slots / mp.groups;
    if (per < 1) per = 1;
    if (per > n_sp) per = n_sp;
    mp.ctas_per_group = per;
    mp.dbg = h->opt.tz_skip;
    mp.pdl_trigger = (h->opt.tz_pdl & 2) ? 1 : 0;
    const bool pdl = h->opt.pdl && (h->opt.tz_pdl & 1);
    CUtensorMap tm;
    int rc = make_tmap_nhwc(h, &tm, x, batch, H, W, C, MixZ::XP, MixZ::XR, MixZ::CG);
    if (rc != FVHD_OK) return rc;
    CUtensorMap tmz;                                    // z store: one tile column (64 rows x 8 channels) per bulk copy
    if ((rc = make_tmap_nhwc(h, &tmz, z, batch, H, W, C, 1, MixZ::ZR, MixZ::CG)) != FVHD_OK) return rc;
    const dim3 grid((unsigned)(per * mp.groups));
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_kc(pdl, cs, repmixer_tz_kernel, grid, dim3(MixZ::THREADS), MixZ::SMEM, s, tm, tmz, mp);
    };
    return FVHD_OK;
}

// The RepMixer depthwise pair's kernels.  choose_mixer() is the plan's choice; fvhd_mixer maps FVHD_MIXER directly.
enum class Mixer { Tz, Tc, Tc2, Umma, Dw };

Mixer choose_mixer(fvhd_handle h, int batch, int H, int W, int C) {
    const char m = h->opt.mixer;
    if (h->opt.mix_tile) return (strchr("a815", h->opt.mix_tile) || m == 'f') ? Mixer::Dw : Mixer::Tc;
    if (m == '2' && C % MixT2::CG == 0) return Mixer::Tc2;
    if (m == 'u') return Mixer::Umma;
    if (m == 0 || m == 'z') {
        // Toeplitz tcgen05 mixer whenever there is at least one 64 x 32 x 8 item per SM; below that (stage 2 of a single
        // 1024-px image: 96 items) the finer-grained mma.sync kernel of mixer_tc.cuh has the shorter critical path
        // (16 vs 20 us per launch at batch 1).  An explicit FVHD_MIXER=z forces it everywhere.
        const long items = (long)batch * ((W + MixZ::ZC - 1) / MixZ::ZC) * ((H + MixZ::ZR - 1) / MixZ::ZR) * (C / MixZ::CG);
        if (m == 'z' || items >= h->num_sms || C % DW_CG != 0) return Mixer::Tz;
    }
    return m == 'f' ? Mixer::Dw : Mixer::Tc;
}

const struct { const char* kernel; decltype(&make_mixer_tz_step) make; } kMixers[] = {     // indexed by Mixer
    {"repmixer_tz_kernel", make_mixer_tz_step}, {"repmixer_tc_kernel", make_mixer_tc_step}, {"repmixer_tc2_kernel", make_mixer_tc2_step},
    {"repmixer_umma_kernel", make_mixer_umma_step}, {"repmixer_dw_kernel", make_mixer_dw_step}};

// GEMM configuration = (BN, cluster size CS, which operand the cluster shares).  Cost model per CTA tile (cycles):
//   load = num_kb * bytes_per_kblock / 36 B/clk   (gemm_trace: ~70 GB/s per SM while all SMs pull, ~10 TB/s chip-wide)
//   mma  = num_kb * 4 * (128 * BN / 256)          (tcgen05 M=128: 128*N/256 cycles per K=16 instruction)
//   epi  = 128 * BN * (GELU ? 10 : 6) / 256       (8 epilogue warps)
//   tile = max(load, mma, epi) + 400 ;  total = rounds * tile, rounds = ceil(cluster_tiles / resident_clusters)
struct GemmCfg { int bn, cs, share_b; long cost; int split; };
GemmCfg pick_gemm_cfg(int M, int N, int K, int act, int num_sms, int max_cs, bool allow_split) {
    const int tiles_m = (M + GEMM_BM - 1) / GEMM_BM;
    const int num_kb = (K + GEMM_BK - 1) / GEMM_BK;
    const int cands[5] = {256, 128, 96, 64, 32};
    GemmCfg best{128, 1, 0, -1, 1};
    for (int bn : cands) {
        if (bn == 96 && N % 96) continue;               // 96 only when it divides N (C = 96 / 192 / 384 layers)
        if (bn == 256 && N % 256) continue;
        if (bn > 32 && bn > ((N + 31) / 32) * 32) continue;
        const int tiles_n = (N + bn - 1) / bn;
        for (int cs = 1; cs <= max_cs; cs *= 2) {
            for (int share_b = 0; share_b < (cs == 1 ? 1 : 2); ++share_b) {
                if (cs > 1 && share_b && (bn / cs) % 8) continue;          // slice boxes stay whole swizzle atoms
                if (cs > 1 && share_b && tiles_m < cs) continue;
                if (cs > 1 && !share_b && tiles_n < cs) continue;
                const long ctiles = share_b ? (long)((tiles_m + cs - 1) / cs) * tiles_n : (long)tiles_m * ((tiles_n + cs - 1) / cs);
                const long resident = cs == 4 ? (num_sms / 4) - 1 : num_sms / cs;   // GPC granularity costs ~1 cluster of 4
                const long rounds = (ctiles + resident - 1) / resident;
                const long bytes_kb = cs == 1 ? 16384 + bn * 128 : (share_b ? 16384 + bn * 128 / cs : 16384 / cs + bn * 128);
                const long load = (long)num_kb * bytes_kb / 36;
                const long mma = (long)num_kb * 4 * (128 * bn / 256);
                const long epi = 128L * bn * (act ? 10 : 6) / 256;
                long tile = load > mma ? load : mma;
                if (epi > tile) tile = epi;
                const long cost = rounds * (tile + 400);
                if (best.cost < 0 || cost < best.cost) best = GemmCfg{bn, cs, share_b, cost, 1};
                // split-K variant (weight-streaming regime): S k-slices per tile, one work item per CTA, distributed reduction;
                // overhead = fp32 partial tile written + re-read (at the same ~36 B/clk) + the arrival wait (measured)
                if (allow_split && cs == 1 && 2 * ctiles <= num_sms && num_kb >= 8) {
                    int S = num_sms / (int)ctiles;
                    if (S > num_kb / 4) S = num_kb / 4;
                    while (S > 1 && (size_t)ctiles * S * GEMM_BM * bn * sizeof(float) > kSplitKWsBytes) --S;
                    if (S > 1) {
                        const int kbs = (num_kb + S - 1) / S;
                        S = (num_kb + kbs - 1) / kbs;
                        const long ld_s = (long)kbs * bytes_kb / 36, mma_s = (long)kbs * 4 * (128 * bn / 256);
                        // + 11 k cycles: publish -> all-slices-arrived -> re-read, measured with tools/gemm_trace.py llm (MMAs done -> epilogue
                        // done: 6.6 us for M 287 N 896 K 896 S 3, 9.5 us for K 4864 S 7; 1 us was assumed before)
                        const long cost_s = (ld_s > mma_s ? ld_s : mma_s) + 400 + 2 * (128L * bn * 4 / 36) + 11000;
                        if (cost_s < best.cost) best = GemmCfg{bn, 1, 0, cost_s, S};
                    }
                }
            }
        }
    }
    return best;
}

// Build one GEMM launch step.  D may be nullptr => taken from the IoBlock at run time.
int make_gemm_step(fvhd_handle h, Step* out, const IoBlock* io, int rows_per_image, const bf16* A, int lda, const bf16* W, const float* bias, const bf16* residual, int ldr,
                   bf16* D, int ldd, int M, int N, int K, int act) {
    if (N % 8 || K % 8) return fail(h, FVHD_ERR_INVALID, "GEMM N (%d) and K (%d) must be multiples of 8", N, K);
    const bool can_split = h->opt.splitk && D != nullptr && h->splitk_ws && N % 4 == 0 && ldd % 4 == 0 && (residual == nullptr || ldr % 4 == 0);
    GemmCfg c = pick_gemm_cfg(M, N, K, act, h->num_sms, g_debug_gemm_cs ? g_debug_gemm_cs : h->opt.gemm_max_cs, can_split);
    if (g_force_bn) { c.bn = g_force_bn; c.cs = 1; c.share_b = 0; c.split = 1; }
    GemmParams p{};
    p.M = M; p.N = N; p.K = K;
    p.BN = c.bn; p.cs = c.cs; p.share_b = c.share_b;
    const int num_kb = (K + GEMM_BK - 1) / GEMM_BK;
    p.stages = gemm_pick_stages(p.BN, num_kb);
    p.tiles_m = (M + GEMM_BM - 1) / GEMM_BM;
    p.tiles_n = (N + p.BN - 1) / p.BN;
    p.ctiles = p.share_b ? ((p.tiles_m + p.cs - 1) / p.cs) * p.tiles_n : p.tiles_m * ((p.tiles_n + p.cs - 1) / p.cs);
    p.split_k = 1; p.kb_per_split = num_kb; p.ws = nullptr; p.counters = nullptr;
    if (c.split > 1 && p.ctiles <= kSplitKDoneOfs) {
        const int kbs = (num_kb + c.split - 1) / c.split;
        p.split_k = (num_kb + kbs - 1) / kbs; p.kb_per_split = kbs; p.ws = h->splitk_ws; p.counters = h->splitk_cnt;
        p.ctiles *= p.split_k;                      // work items = (tile, k-slice), one per CTA
    }
    p.trace = g_gemm_trace;
    p.D = D; p.io = io; p.rows_per_image = rows_per_image > 0 ? rows_per_image : 1; p.ldd = ldd; p.bias = bias; p.residual = residual; p.ldr = ldr; p.act = act;
    CUtensorMap ta, tb, td;
    int rc;
    const int a_box = (p.cs > 1 && !p.share_b) ? GEMM_BM / p.cs : GEMM_BM;     // shared operand: each CTA loads a 1/CS slice
    const int b_box = (p.cs > 1 && p.share_b) ? p.BN / p.cs : p.BN;
    if ((rc = make_tmap(h, &ta, A, M, K, lda, a_box)) != FVHD_OK) return rc;
    if ((rc = make_tmap(h, &tb, W, N, K, K, b_box)) != FVHD_OK) return rc;
    // D leaves through TMA stores (box 64 cols x 32 rows, 128-B swizzle) when it is library memory known at plan time
    p.tma_store = (D != nullptr && p.BN >= 64) ? 1 : 0;
    if (p.tma_store) {
        if ((rc = make_tmap(h, &td, D, M, N, ldd, 32, 64)) != FVHD_OK) return rc;
    } else {
        td = ta;
    }
    const size_t smem = gemm_smem_bytes(p.BN, p.stages);
    const int resident = p.cs > 1 ? resident_clusters(gemm_bf16_tcgen05_kernel, p.cs, GEMM_THREADS, smem, h->num_sms) : h->num_sms;
    if (resident < 1) return fail(h, FVHD_ERR_CUDA, "no resident %d-CTA cluster of the GEMM kernel (%zu B of shared memory)", p.cs, smem);
    const int nclusters = p.ctiles < resident ? p.ctiles : resident;
    const dim3 grid((unsigned)(nclusters * p.cs));
    if (h->opt.debug_plan)
        fprintf(stderr, "[fvhd] gemm M=%d N=%d K=%d BN=%d stages=%d tiles=%dx%d split_k=%d kb/slice=%d items=%d grid=%u tma_store=%d act=%d\n", M, N, K, p.BN, p.stages,
                p.tiles_m, p.tiles_n, p.split_k, p.kb_per_split, p.ctiles, grid.x, p.tma_store, act);
    const int cs = p.cs;
    const bool pdl = h->opt.pdl;
    *out = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_kc(pdl, cs, gemm_bf16_tcgen05_kernel, grid, dim3(GEMM_THREADS), smem, s, ta, tb, td, p);
    };
    return FVHD_OK;
}

template <int KS, int S, int MULT, int ACT, int TOH, int TOW, int SW>
int make_dw_step(fvhd_handle h, Step* out_step, const bf16* in, bf16* out, const float* w, const float* b, int batch, int H, int W, int C) {
    using Cfg = DwCfg<KS, S, MULT, TOH, TOW>;
    const int Ho = (H + 2 * (KS / 2) - KS) / S + 1, Wo = (W + 2 * (KS / 2) - KS) / S + 1;
    const int tx = (Wo + TOW - 1) / TOW, ty = (Ho + TOH - 1) / TOH;
    const dim3 grid(tx * ty, C / DW_CG, batch);
    const size_t smem = Cfg::SMEM;
    CUtensorMap tm;
    int rc = make_tmap_nhwc(h, &tm, in, batch, H, W, C, Cfg::IWP, Cfg::IH);
    if (rc != FVHD_OK) return rc;
    const bool pdl = h->opt.pdl;
    *out_step = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_k(pdl, dwconv_kernel<KS, S, MULT, ACT, TOH, TOW, SW>, grid, dim3(DW_THREADS), smem, s, tm, out, w, b, H, W, C, Ho, Wo, tx);
    };
    return FVHD_OK;
}

// RepCPE / attention-block dw7x7 (stride 1): 16 x 16 tiles, or 8 x 16 tiles while 16 x 16 would leave SMs without a CTA (batch 1:
// stage 3 has 96 such CTAs, stage 4 has 48) -- the launch is pure latency there and half the rows per CTA halve it.
int make_dw7_step(fvhd_handle h, Step* out_step, const bf16* in, bf16* out, const float* w, const float* b, int batch, int H, int W, int C) {
    const long ctas16 = (long)((W + 15) / 16) * ((H + 15) / 16) * (C / DW_CG) * batch;
    if (ctas16 < h->num_sms && H > 8) return make_dw_step<7, 1, 1, 0, 8, 16, 8>(h, out_step, in, out, w, b, batch, H, W, C);
    return make_dw_step<7, 1, 1, 0, 16, 16, 8>(h, out_step, in, out, w, b, batch, H, W, C);
}

const float* WF(fvhd_handle h, const std::string& n) { return reinterpret_cast<const float*>(h->wptr.at(n)); }
const bf16* WB(fvhd_handle h, const std::string& n) { return reinterpret_cast<const bf16*>(h->wptr.at(n)); }

const char* kGemm = "gemm_bf16_tcgen05_kernel";
double gemm_flops(double M, double N, double K) { return 2.0 * M * N * K; }
double gemm_bytes(double M, double N, double K, bool res) { return 2.0 * (M * K + N * K + M * N * (res ? 2 : 1)) + 4.0 * N; }

int add_gemm(fvhd_handle h, Plan& pl, int unit, const bf16* A, int lda, const bf16* W, const float* bias, const bf16* residual, int ldr,
             bf16* D, int ldd, int M, int N, int K, int act) {
    Step g;
    int rc = make_gemm_step(h, &g, pl.io, h->ntok, A, lda, W, bias, residual, ldr, D, ldd, M, N, K, act);
    if (rc != FVHD_OK) return rc;
    pl.add(g, kGemm, unit, gemm_flops(M, N, K), gemm_bytes(M, N, K, residual != nullptr));
    return FVHD_OK;
}

int add_convffn_steps(fvhd_handle h, Plan& pl, int unit, const std::string& p, const Buffers& bf, const bf16* z, const bf16* resid, bf16* out, int M, int c) {
    int rc;
    if ((rc = add_gemm(h, pl, unit, z, c, WB(h, p + "fc1.w"), WF(h, p + "fc1.b"), nullptr, 0, bf.H4, 4 * c, M, 4 * c, c, 1)) != FVHD_OK) return rc;
    return add_gemm(h, pl, unit, bf.H4, 4 * c, WB(h, p + "fc2.w"), WF(h, p + "fc2.b"), resid, c, out, c, M, c, 4 * c, 0);
}

// ConvFFN of a RepMixer block as ONE kernel (C in {96, 192}): hidden stays in TMEM / smem (mlp_fused.cuh).
int make_fused_mlp_step(fvhd_handle h, Step* st, const bf16* z, const bf16* w1, const float* b1, const bf16* w2, const float* b2,
                        const bf16* resid, bf16* out, int M, int c) {
    MlpParams mp{};
    mp.M = M; mp.C = c; mp.tiles_m = (M + GEMM_BM - 1) / GEMM_BM;
    mp.b1 = b1; mp.b2 = b2; mp.resid = resid; mp.D = out;
    CUtensorMap tz, tw1, tw2, td;
    int rc;
    if ((rc = make_tmap(h, &tz, z, M, c, c, GEMM_BM)) != FVHD_OK) return rc;
    if ((rc = make_tmap(h, &tw1, w1, 4 * c, c, c, MLP_NH)) != FVHD_OK) return rc;
    if ((rc = make_tmap(h, &tw2, w2, c, 4 * c, 4 * c, c)) != FVHD_OK) return rc;
    if ((rc = make_tmap(h, &td, out, M, c, c, 32, 64)) != FVHD_OK) return rc;
    const dim3 grid((unsigned)(mp.tiles_m < h->num_sms ? mp.tiles_m : h->num_sms));
    const size_t smem = mlp_smem_bytes(c);
    const bool pdl = h->opt.pdl;
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_k(pdl, mlp_fused_tcgen05_kernel, grid, dim3(MLP_THREADS), smem, s, tz, tw1, tw2, td, mp);
    };
    return FVHD_OK;
}

// MHSA core on tcgen05 (attention_umma.cuh): one CTA per (256 queries, head, image).
int make_attention_umma_step(fvhd_handle h, Step* st, const bf16* qkv, bf16* out, int batch, int N, int c, float scale_log2e) {
    AttUParams ap{};
    ap.out = out; ap.N = N; ap.C = c; ap.qpairs = (N + 2 * AttU::QT - 1) / (2 * AttU::QT); ap.scale_log2e = scale_log2e;
    CUtensorMap tm;
    int rc = make_tmap(h, &tm, qkv, (int64_t)batch * N, 3LL * c, 3LL * c, AttU::KT, AttU::HD, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc != FVHD_OK) return rc;
    const dim3 grid((unsigned)ap.qpairs, (unsigned)(c / AttU::HD), (unsigned)batch);
    const bool pdl = h->opt.pdl;
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_k(pdl, attention_umma_kernel, grid, dim3(AttU::THREADS), AttU::SMEM, s, tm, ap);
    };
    return FVHD_OK;
}

// MHSA core on mma.sync (stem_attn_se.cuh): one CTA per (64 queries, head, image).
int make_attention_mma_step(fvhd_handle h, Step* st, const bf16* qkv, bf16* out, int batch, int N, int c, float scale_log2e) {
    const dim3 grid((N + 63) / 64, c / 32, batch);
    const bool pdl = h->opt.pdl;
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_k(pdl, attention_kernel, grid, dim3(128), 0, s, qkv, out, N, c, scale_log2e);
    };
    return FVHD_OK;
}

enum class Attn { Mma, Umma };

// Automatic choice: the tcgen05 / TMEM kernel from 512 tokens (one CTA = 256 queries x 1 head: at N = 256 there are too few
// CTAs and the mma.sync kernel's finer grid wins -- measured 12.3 vs 10.5 us at batch 1, 86 vs 84 us at batch 32).
Attn choose_attention(fvhd_handle h, int N) {
    return (h->opt.attn == 'u' || (h->opt.attn == 'a' && N >= 512)) ? Attn::Umma : Attn::Mma;
}

// Second-generation fused ConvFFN (convffn.cuh): one CTA per 128-pixel tile, 16 epilogue warps, packed-half GELU, C in {96, 192, 384}.
template <int C>
int make_convffn2_step_t(fvhd_handle h, Step* st, const bf16* z, const bf16* w1, const float* b1, const void* w2, int w2_f16, const float* b2,
                         const bf16* resid, bf16* out, int M) {
    MlpParams mp{};
    mp.M = M; mp.C = C; mp.tiles_m = (M + GEMM_BM - 1) / GEMM_BM;
    mp.w2_f16 = w2_f16;
    mp.b1 = b1; mp.b2 = b2; mp.resid = resid; mp.D = out;
    CUtensorMap tz, tw1, tw2;
    int rc;
    if ((rc = make_tmap(h, &tz, z, M, C, C, GEMM_BM)) != FVHD_OK) return rc;
    if ((rc = make_tmap(h, &tw1, w1, 4 * C, C, C, MLP_NH)) != FVHD_OK) return rc;
    if ((rc = make_tmap(h, &tw2, w2, C, 4 * C, 4 * C, CfCfg<C>::N2)) != FVHD_OK) return rc;
    const size_t smem = CfCfg<C>::SMEM;
    const bool pdl = h->opt.pdl;
    const int ci = C == 96 ? 0 : C == 192 ? 1 : 2;
    if (h->opt.convffn_cs == 2 && h->cf_clusters[ci] > 0) {     // 2-CTA clusters sharing the weight stream (halves each SM's weight ingest)
        const int want = (mp.tiles_m + 1) / 2;
        const dim3 grid2((unsigned)(2 * (want < h->cf_clusters[ci] ? want : h->cf_clusters[ci])));
        *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
            return launch_kc(pdl, 2, convffn_tcgen05_kernel<C, 2>, grid2, dim3(CF_THREADS), smem, s, tz, tw1, tw2, mp);
        };
        return FVHD_OK;
    }
    const dim3 grid((unsigned)(mp.tiles_m < h->num_sms ? mp.tiles_m : h->num_sms));
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_k(pdl, convffn_tcgen05_kernel<C, 1>, grid, dim3(CF_THREADS), smem, s, tz, tw1, tw2, mp);
    };
    return FVHD_OK;
}
int make_convffn2_step(fvhd_handle h, Step* st, const bf16* z, const bf16* w1, const float* b1, const void* w2, int w2_f16, const float* b2,
                       const bf16* resid, bf16* out, int M, int c) {
    if (c == 96) return make_convffn2_step_t<96>(h, st, z, w1, b1, w2, w2_f16, b2, resid, out, M);
    if (c == 192) return make_convffn2_step_t<192>(h, st, z, w1, b1, w2, w2_f16, b2, resid, out, M);
    if (c == 384) return make_convffn2_step_t<384>(h, st, z, w1, b1, w2, w2_f16, b2, resid, out, M);
    return fail(h, FVHD_ERR_INVALID, "convffn_tcgen05_kernel exists for C in {96, 192, 384}, got %d", c);
}

// Stage-2 ConvFFN (C = 384): one 4-CTA cluster per 128-pixel tile, hidden split across the cluster, DSMEM reduction.
int make_cluster_mlp_step(fvhd_handle h, Step* st, const bf16* z, const bf16* w1, const float* b1, const bf16* w2, const float* b2,
                          const bf16* resid, bf16* out, int M, unsigned long long* trace) {
    const int c = MLPC_C;
    if (h->mlpc_clusters <= 0) return fail(h, FVHD_ERR_CUDA, "no resident 4-CTA cluster for the stage-2 ConvFFN kernel");
    MlpParams mp{};
    mp.M = M; mp.C = c; mp.tiles_m = (M + GEMM_BM - 1) / GEMM_BM;
    mp.b1 = b1; mp.b2 = b2; mp.resid = resid; mp.D = out; mp.trace = trace;
    CUtensorMap tz, tw1, tw2;
    int rc;
    if ((rc = make_tmap(h, &tz, z, M, c, c, GEMM_BM)) != FVHD_OK) return rc;
    if ((rc = make_tmap(h, &tw1, w1, 4 * c, c, c, MLP_NH)) != FVHD_OK) return rc;
    if ((rc = make_tmap(h, &tw2, w2, c, 4 * c, 4 * c, MLPC_NHALF)) != FVHD_OK) return rc;
    const int clusters = mp.tiles_m < h->mlpc_clusters ? mp.tiles_m : h->mlpc_clusters;
    const dim3 grid((unsigned)(clusters * MLPC_CS));
    const bool pdl = h->opt.pdl;
    *st = [=](cudaStream_t s, const RunCtx&) -> cudaError_t {
        return launch_kc(pdl, MLPC_CS, mlp_cluster_tcgen05_kernel, grid, dim3(MLPC_THREADS), MLPC_SMEM, s, tz, tw1, tw2, mp);
    };
    return FVHD_OK;
}

// The ConvFFN of a RepMixer block over M pixels of C channels.
enum class ConvFfn { Gen2, Fused, Cluster, TwoGemms };

ConvFfn choose_convffn(fvhd_handle h, int M, int c) {
    const Options& o = h->opt;
    // the 4-CTA cluster kernel at small batches only: beyond two tiles per resident cluster the two plain GEMMs fill the machine better
    // (measured: batch 1 0.71 vs 0.91 ms for the 24 blocks, batch 4 2.23 vs 2.15 ms, batch 8 4.28 vs 3.67 ms)
    const bool few_tiles = c == MLPC_C && o.cluster_mlp && h->mlpc_clusters > 0 && (M + GEMM_BM - 1) / GEMM_BM <= 2 * h->mlpc_clusters;
    // second-generation single-CTA kernel: every C, any batch (stage 2 at batch <= 2 keeps the 4-CTA cluster kernel: 32 tiles per
    // image cannot fill 148 SMs one tile per CTA)
    if (o.fused_mlp && o.convffn_gen == 2 && !few_tiles) return ConvFfn::Gen2;
    if (o.fused_mlp && c <= 192) return ConvFfn::Fused;
    return few_tiles ? ConvFfn::Cluster : ConvFfn::TwoGemms;
}

enum class Stem { Gen1, Gen2 };

Stem choose_stem(fvhd_handle h) { return h->opt.stem_gen == 1 ? Stem::Gen1 : Stem::Gen2; }

int build_plan(fvhd_handle h, int batch, Plan& pl) {
    pl = Plan();
    pl.batch = batch;
    const Buffers bf = carve(h, batch);
    pl.io = bf.io;
    const IoBlock* io = bf.io;
    bf16* cur = bf.X0;
    bf16* nxt = bf.X1;
    int rc;
    const bool pdl = h->opt.pdl;
    const size_t nunits = h->units.size();
    for (size_t ui = 0; ui < nunits; ++ui) {
        const UnitDesc& u = h->units[ui];
        const int U = (int)ui;
        const int begin = (int)pl.steps.size();
        const std::string& p = u.prefix;
        const int c = u.cin, H = u.hin, W = u.win;
        const int M = batch * u.hout * u.wout;
        const double Md = (double)M;
        const bool last = ui + 1 == nunits;
        bf16* in = cur;
        bf16* out = nxt;
        switch (u.kind) {
        case 0: {   // stem: fused conv0+dw1 -> T1, then 1x1+GELU GEMM
            const float *w0 = WF(h, "stem.w0"), *b0 = WF(h, "stem.b0"), *w1 = WF(h, "stem.w1"), *b1 = WF(h, "stem.b1");
            const int R = h->R, tiles = (R / 4 + STEM_TO - 1) / STEM_TO;
            const dim3 grid(tiles * tiles, 1, batch);
            bf16* t0 = bf.T1;
            const double stem_flops = 2.0 * batch * ((double)(R / 2) * (R / 2) * 96 * 27 + (double)(R / 4) * (R / 4) * 96 * 9);
            const double stem_bytes = (double)batch * (3.0 * R * R * 2 + (double)(R / 4) * (R / 4) * 96 * 2);
            if (choose_stem(h) == Stem::Gen2) {
                const int n_tiles = tiles * tiles * batch;
                const dim3 grid2((unsigned)std::min(n_tiles, 3 * h->num_sms));
                pl.add([=](cudaStream_t s, const RunCtx& ctx) -> cudaError_t {
                    if (ctx.img_dtype == FVHD_F32) return launch_k(pdl, stem2_kernel<float>, grid2, dim3(Stem2::THREADS), Stem2::SMEM, s, io, t0, w0, b0, w1, b1, R, tiles, n_tiles);
                    if (ctx.img_dtype == FVHD_F16) return launch_k(pdl, stem2_kernel<__half>, grid2, dim3(Stem2::THREADS), Stem2::SMEM, s, io, t0, w0, b0, w1, b1, R, tiles, n_tiles);
                    return launch_k(pdl, stem2_kernel<bf16>, grid2, dim3(Stem2::THREADS), Stem2::SMEM, s, io, t0, w0, b0, w1, b1, R, tiles, n_tiles);
                }, "stem2_kernel", U, stem_flops, stem_bytes);
            } else {
            pl.add([=](cudaStream_t s, const RunCtx& ctx) -> cudaError_t {
                if (ctx.img_dtype == FVHD_F32) return launch_k(pdl, stem_kernel<float>, grid, dim3(STEM_THREADS), STEM_SMEM, s, io, t0, w0, b0, w1, b1, R, tiles);
                if (ctx.img_dtype == FVHD_F16) return launch_k(pdl, stem_kernel<__half>, grid, dim3(STEM_THREADS), STEM_SMEM, s, io, t0, w0, b0, w1, b1, R, tiles);
                return launch_k(pdl, stem_kernel<bf16>, grid, dim3(STEM_THREADS), STEM_SMEM, s, io, t0, w0, b0, w1, b1, R, tiles);
            }, "stem_kernel", U, stem_flops, stem_bytes);
            }
            if ((rc = add_gemm(h, pl, U, t0, 96, WB(h, "stem.w2"), WF(h, "stem.b2"), nullptr, 0, out, 96, M, 96, 96, 1)) != FVHD_OK) return rc;
            in = nullptr;
            break;
        }
        case 1: {   // RepMixerBlock: fused dw3x3 -> y, dw7x7(+BN) -> z ; fc1+GELU ; fc2 (+layer scale folded) + y
            const float *w3 = WF(h, p + "mix.w"), *b3 = WF(h, p + "mix.b"), *w7 = WF(h, p + "dw.w"), *b7 = WF(h, p + "dw.b");
            bf16 *y = bf.Y, *z = bf.Z;
            const auto& mk = kMixers[(int)choose_mixer(h, batch, H, W, c)];
            Step ms;
            if ((rc = mk.make(h, &ms, in, y, z, w3, b3, w7, b7, batch, H, W, c)) != FVHD_OK) return rc;
            pl.add(ms, mk.kernel, U, 2.0 * Md * c * 58, 3.0 * Md * c * 2);
            const bf16 *w1 = WB(h, p + "fc1.w"), *w2 = WB(h, p + "fc2.w");
            const float *b1 = WF(h, p + "fc1.b"), *b2 = WF(h, p + "fc2.b");
            Step fs;
            const char* fk = nullptr;       // the fused kernels' name; two GEMMs add their own steps
            switch (choose_convffn(h, M, c)) {
            case ConvFfn::Gen2: rc = make_convffn2_step(h, &fs, z, w1, b1, h->wptr.at(p + "fc2.wh"), 1, b2, y, out, M, c); fk = "convffn_tcgen05_kernel"; break;
            case ConvFfn::Fused: rc = make_fused_mlp_step(h, &fs, z, w1, b1, w2, b2, y, out, M, c); fk = "mlp_fused_tcgen05_kernel"; break;
            case ConvFfn::Cluster: rc = make_cluster_mlp_step(h, &fs, z, w1, b1, w2, b2, y, out, M, nullptr); fk = "mlp_cluster_tcgen05_kernel"; break;
            case ConvFfn::TwoGemms: rc = add_convffn_steps(h, pl, U, p, bf, z, y, out, M, c); break;
            }
            if (rc != FVHD_OK) return rc;
            if (fk) pl.add(fs, fk, U, 2.0 * gemm_flops(M, 4 * c, c), 2.0 * (3.0 * M * c + 8.0 * c * c) + 20.0 * c);
            break;
        }
        case 2: {   // PatchEmbed: dw7x7 s2 (x2 channels) + GELU ; 1x1 + GELU
            { Step ds; if ((rc = make_dw_step<7, 2, 2, 1, 8, 8, 4>(h, &ds, in, bf.T1, WF(h, p + "dw.w"), WF(h, p + "dw.b"), batch, H, W, c)) != FVHD_OK) return rc; pl.add(ds, "dwconv_kernel<7,2,2>", U, 2.0 * Md * u.cout * 49, 2.0 * ((double)batch * u.in_elems + Md * u.cout)); }
            if ((rc = add_gemm(h, pl, U, bf.T1, u.cout, WB(h, p + "pw.w"), WF(h, p + "pw.b"), nullptr, 0, out, u.cout, M, u.cout, u.cout, 1)) != FVHD_OK) return rc;
            break;
        }
        case 3:     // RepCPE: dw7x7 + bias (identity folded into the centre tap)
            { Step ds; if ((rc = make_dw7_step(h, &ds, in, out, WF(h, p + "dw.w"), WF(h, p + "dw.b"), batch, H, W, c)) != FVHD_OK) return rc; pl.add(ds, "dwconv_kernel<7,1,1>", U, 2.0 * Md * c * 49, 4.0 * Md * c); }
            break;
        case 4: {   // AttentionBlock
            const int N = H * W;
            const float *lw = WF(h, p + "ln.w"), *lb = WF(h, p + "ln.b");
            bf16 *t1 = bf.T1, *qkv = bf.H4, *x1 = bf.Y;
            const int lngrid = (M + 7) / 8;
            if (c != 768 && c != 1536) return fail(h, FVHD_ERR_INVALID, "LayerNorm kernel expects C in {768,1536}, got %d", c);
            pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t {
                if (c == 768) return launch_k(pdl, layernorm_channel_kernel<3>, dim3(lngrid), dim3(256), 0, s, in, t1, lw, lb, M, 1e-5f);
                return launch_k(pdl, layernorm_channel_kernel<6>, dim3(lngrid), dim3(256), 0, s, in, t1, lw, lb, M, 1e-5f);
            }, "layernorm_channel_kernel", U, 0.0, 4.0 * Md * c);
            if ((rc = add_gemm(h, pl, U, t1, c, WB(h, p + "qkv.w"), nullptr, nullptr, 0, qkv, 3 * c, M, 3 * c, c, 0)) != FVHD_OK) return rc;
            const float sl2 = 0.17677669529663687f * 1.4426950408889634f;   // 32^-0.5 * log2(e)
            const bool umma = choose_attention(h, N) == Attn::Umma;
            Step as;
            if ((rc = (umma ? make_attention_umma_step : make_attention_mma_step)(h, &as, qkv, t1, batch, N, c, sl2)) != FVHD_OK) return rc;
            pl.add(as, umma ? "attention_umma_kernel" : "attention_kernel", U, 4.0 * batch * (double)N * N * c, 8.0 * Md * c);
            if ((rc = add_gemm(h, pl, U, t1, c, WB(h, p + "proj.w"), WF(h, p + "proj.b"), in, c, x1, c, M, c, c, 0)) != FVHD_OK) return rc;
            { Step ds; if ((rc = make_dw7_step(h, &ds, x1, bf.Z, WF(h, p + "dw.w"), WF(h, p + "dw.b"), batch, H, W, c)) != FVHD_OK) return rc; pl.add(ds, "dwconv_kernel<7,1,1>", U, 2.0 * Md * c * 49, 4.0 * Md * c); }
            if ((rc = add_convffn_steps(h, pl, U, p, bf, bf.Z, x1, out, M, c)) != FVHD_OK) return rc;
            break;
        }
        case 5: {   // conv_exp: dw3x3 (x2 channels) -> SE -> GELU -> tokens
            const int HW = H * W;
            bf16* cexp = bf.T1;
            { Step ds; if ((rc = make_dw_step<3, 1, 2, 0, 16, 16, 8>(h, &ds, in, cexp, WF(h, p + "dw.w"), WF(h, p + "dw.b"), batch, H, W, c)) != FVHD_OK) return rc; pl.add(ds, "dwconv_kernel<3,1,2>", U, 2.0 * Md * 3072 * 9, 2.0 * Md * (1536 + 3072)); }
            float *pooled = bf.pooled, *sr = bf.sr;
            const bf16 *wr = WB(h, p + "se.r.w"), *we = WB(h, p + "se.e.w");
            const float *br = WF(h, p + "se.r.b"), *be = WF(h, p + "se.e.b");
            bf16* dst = last ? nullptr : out;
            pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t {
                return launch_k(pdl, se_pool_kernel, dim3(3072 / 64, batch), dim3(256), 0, s, cexp, pooled, HW, 3072);
            }, "se_pool_kernel", U, 0.0, 2.0 * Md * 3072);
            pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t {
                return launch_k(pdl, se_reduce_kernel, dim3(kSeRd / 8, batch), dim3(256), 0, s, pooled, wr, br, sr, 3072, kSeRd);
            }, "se_reduce_kernel", U, 2.0 * batch * 3072 * kSeRd, 2.0 * 3072 * kSeRd);
            pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t {
                return launch_k(pdl, se_expand_scale_gelu_kernel, dim3(3072 / 64, batch), dim3(256), 0, s, cexp, sr, we, be, dst, io, HW, 3072, kSeRd);
            }, "se_expand_scale_gelu_kernel", U, 2.0 * batch * 3072 * kSeRd, 4.0 * Md * 3072 + 2.0 * 3072 * kSeRd);
            break;
        }
        case 6: {   // projector
            const int Hd = u.cout;
            if (h->cfg.projector_depth == 2) {
                if ((rc = add_gemm(h, pl, U, in, 3072, WB(h, "projector.0.w"), WF(h, "projector.0.b"), nullptr, 0, bf.T1, Hd, M, Hd, 3072, 1)) != FVHD_OK) return rc;
                if ((rc = add_gemm(h, pl, U, bf.T1, Hd, WB(h, "projector.2.w"), WF(h, "projector.2.b"), nullptr, 0, nullptr, Hd, M, Hd, Hd, 0)) != FVHD_OK) return rc;
            } else {
                if ((rc = add_gemm(h, pl, U, in, 3072, WB(h, "projector.0.w"), WF(h, "projector.0.b"), nullptr, 0, nullptr, Hd, M, Hd, 3072, 0)) != FVHD_OK) return rc;
            }
            break;
        }
        default:
            return fail(h, FVHD_ERR_INVALID, "unknown unit kind %d", u.kind);
        }
        pl.unit_steps.push_back({begin, (int)pl.steps.size()});
        pl.unit_in.push_back(in);
        pl.unit_out.push_back(out);
        cur = out;
        nxt = (out == bf.X0) ? bf.X1 : bf.X0;
    }
    return FVHD_OK;
}

int get_plan(fvhd_handle h, int batch, Plan** out) {
    auto it = h->plans.find(batch);
    if (it == h->plans.end()) {
        Plan pl;
        int rc = build_plan(h, batch, pl);
        if (rc != FVHD_OK) return rc;
        it = h->plans.emplace(batch, std::move(pl)).first;
    }
    *out = &it->second;
    return FVHD_OK;
}

int check_ready(fvhd_handle h, int batch) {
    if (!h) return FVHD_ERR_INVALID;
    if (!h->loaded) return fail(h, FVHD_ERR_STATE, "fvhd_load_weights has not been called");
    if (batch < 1) return fail(h, FVHD_ERR_INVALID, "batch must be >= 1 (got %d)", batch);
    const int bc = batch < h->cfg.max_batch ? batch : h->cfg.max_batch;
    if (!h->ws || h->ws_bytes < workspace_bytes(h, bc))
        return fail(h, FVHD_ERR_WORKSPACE, "workspace %zu B < required %zu B for %d images per pass", h->ws_bytes, workspace_bytes(h, bc), bc);
    return ensure_cuda(h);
}

size_t dtype_size(int dt) { return dt == FVHD_F32 ? 4 : 2; }

// One stand-alone step on `stream` (the single-kernel entries).
int launch_step(fvhd_handle h, const Step& s, void* stream, const char* what) {
    cudaError_t e = s(reinterpret_cast<cudaStream_t>(stream), RunCtx{});
    if (e != cudaSuccess) return fail(h, FVHD_ERR_CUDA, "%s launch failed: %s", what, cudaGetErrorString(e));
    return FVHD_OK;
}

// Run steps [s0, s1) of a plan (direct launches).
int run_steps(fvhd_handle h, Plan& pl, int s0, int s1, cudaStream_t st, const RunCtx& ctx) {
    for (int i = s0; i < s1; ++i) {
        cudaError_t e = pl.steps[i](st, ctx);
        if (e != cudaSuccess) return fail(h, FVHD_ERR_CUDA, "launch of step %d (%s) failed: %s", i, pl.info[i].kernel, cudaGetErrorString(e));
    }
    return FVHD_OK;
}

int set_io(fvhd_handle h, Plan& pl, cudaStream_t st, const void* images, void* final_out, void* tokens_out, long long final_image_stride,
           const PeerList* peers = nullptr, const ScatterList* scatter = nullptr) {
    PeerList pl_peers{};
    if (peers) pl_peers = *peers;
    ScatterList sc{};
    if (scatter) sc = *scatter;
    cudaError_t e = launch_k(h->opt.pdl, set_io_kernel, dim3(1), dim3(FVHD_MAX_SCATTER), 0, st, pl.io, images, final_out, tokens_out, final_image_stride, pl_peers, sc);
    if (e != cudaSuccess) return fail(h, FVHD_ERR_CUDA, "set_io_kernel launch failed: %s", cudaGetErrorString(e));
    return FVHD_OK;
}

int launch_copy_tokens(fvhd_handle h, Plan& pl, cudaStream_t st, const bf16* src, size_t bytes) {
    const size_t n16 = bytes / 16;
    int blocks = (int)((n16 + 255) / 256);
    if (blocks > 1184) blocks = 1184;
    cudaError_t e = launch_k(h->opt.pdl, copy_tokens_kernel, dim3(blocks), dim3(256), 0, st, reinterpret_cast<const uint4*>(src), pl.io, n16);
    if (e != cudaSuccess) return fail(h, FVHD_ERR_CUDA, "copy_tokens_kernel launch failed: %s", cudaGetErrorString(e));
    return FVHD_OK;
}

// Steps [0, last_step) (+ token copy-out) as ONE graph launch; captured once per (dtype, last_step, copy) and replayed.
// Falls back to direct launches when graphs are disabled (FVHD_NO_GRAPH=1) or the caller is itself capturing `st`.
int run_forward(fvhd_handle h, Plan& pl, cudaStream_t st, const RunCtx& ctx, int last_step, const bf16* tok_src, size_t tok_bytes) {
    int rc;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cs);
    if (!h->opt.graph || cs != cudaStreamCaptureStatusNone) {
        if ((rc = run_steps(h, pl, 0, last_step, st, ctx)) != FVHD_OK) return rc;
        if (tok_src) return launch_copy_tokens(h, pl, st, tok_src, tok_bytes);
        return FVHD_OK;
    }
    const int key = ctx.img_dtype | (last_step << 2) | ((tok_src ? 1 : 0) << 20);
    auto it = pl.graphs.find(key);
    if (it == pl.graphs.end()) {
        cudaGraph_t graph = nullptr;
        cudaStream_t cap = h->cap_stream;
        CUDA_TRY(h, cudaStreamBeginCapture(cap, cudaStreamCaptureModeThreadLocal));
        rc = run_steps(h, pl, 0, last_step, cap, ctx);
        if (rc == FVHD_OK && tok_src) rc = launch_copy_tokens(h, pl, cap, tok_src, tok_bytes);
        cudaError_t e = cudaStreamEndCapture(cap, &graph);
        if (rc != FVHD_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e != cudaSuccess) return fail(h, FVHD_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(e));
        cudaGraphExec_t exec = nullptr;
        e = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) return fail(h, FVHD_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e));
        it = pl.graphs.emplace(key, exec).first;
    }
    CUDA_TRY(h, cudaGraphLaunch(it->second, st));
    return FVHD_OK;
}

// ------------------------------------------------------------------ LLM prefill (row f3)
void llm_free(LlmState* L) {
    for (auto& kv : L->plans)
        for (auto& g : kv.second.graphs) cudaGraphExecDestroy(g.second);
    L->plans.clear();
    void* bufs[] = {L->x0, L->x1, L->x2, L->xn, L->qkv, L->att, L->gu, L->hm, L->logits, L->kc, L->vc, L->rope, L->token};
    for (void* b : bufs) if (b) cudaFree(b);
}

// Launch sequence of one L-token prefill: per layer RMSNorm, qkv GEMM (+bias), RoPE + KV cache + causal GQA attention (one kernel), o GEMM (+residual),
// RMSNorm, gate/up GEMM, SwiGLU, down GEMM (+residual); then final RMSNorm on the last row, lm_head GEMM (M = 1), argmax.
int build_llm_plan(fvhd_handle h, LlmState* S, int L, Plan& pl) {
    const fvhd_llm_config& c = S->c;
    const int H = c.hidden, D = c.head_dim, I = c.intermediate, NQ = S->nqkv, HD = c.heads * D;
    pl = Plan();
    pl.batch = L;
    int rc;
    bf16 *xc = S->x0, *xx = S->x1;           // layer input (x0 = the caller's sequence, then x2) / post-attention stream
    const int ln_grid = (L + 7) / 8;
    const float sl2 = 1.4426950408889634f / sqrtf((float)D);
    const float2* rope = S->rope;
    const bool pdl = h->opt.pdl;
    auto add_gemm_l = [&](const bf16* A, int lda, const void* W, const void* bias, const bf16* resid, bf16* Dp, int M, int N, int K) -> int {
        Step g;
        int r = make_gemm_step(h, &g, nullptr, 1, A, lda, (const bf16*)W, (const float*)bias, resid, N, Dp, N, M, N, K, 0);
        if (r != FVHD_OK) return r;
        pl.add(g, kGemm, 0, gemm_flops(M, N, K), 2.0 * ((double)M * K + (double)N * K + (double)M * N));
        return FVHD_OK;
    };
    for (int l = 0; l < c.layers; ++l) {
        const void* const* w = S->w.data() + (size_t)l * 7;
        const float *ln1 = (const float*)w[0], *ln2 = (const float*)w[4];
        bf16 *xn = S->xn, *qkv = S->qkv, *att = S->att, *gu = S->gu, *hm = S->hm;
        bf16* kc = S->kc + (size_t)l * c.max_seq * c.kv_heads * D;
        bf16* vc = S->vc + (size_t)l * c.max_seq * c.kv_heads * D;
        const bf16* xin = xc;
        const float eps = c.rms_eps;
        pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t { return launch_k(pdl, rmsnorm_kernel, dim3(ln_grid), dim3(256), 0, s, xin, xn, ln1, L, H, eps); },
               "rmsnorm_kernel", 0, 0.0, 4.0 * L * H);
        if ((rc = add_gemm_l(xn, H, w[1], w[2], nullptr, qkv, L, NQ, H)) != FVHD_OK) return rc;
        const int heads = c.heads, kvh = c.kv_heads;
        if (h->opt.llm_attn_fma) {      // FVHD_LLM_ATTN=f: the FMA-pipe kernel (first version; kept for A/B)
            const dim3 agrid((L + LLM_ATTN_QB - 1) / LLM_ATTN_QB, heads);
            pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t {
                       if (D == 64) return launch_k(pdl, causal_attn_kernel<64>, agrid, dim3(LLM_ATTN_THREADS), LlmAttnSmem<64>::BYTES, s, (const bf16*)qkv, att, rope, kc, vc, L, heads, kvh, sl2);
                       return launch_k(pdl, causal_attn_kernel<128>, agrid, dim3(LLM_ATTN_THREADS), LlmAttnSmem<128>::BYTES, s, (const bf16*)qkv, att, rope, kc, vc, L, heads, kvh, sl2);
                   }, "causal_attn_kernel", 0, 2.0 * (double)L * L * HD, 2.0 * L * (NQ + HD));
        } else {
            const dim3 agrid((L + LLM_MMA_QB - 1) / LLM_MMA_QB, heads);
            pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t {
                       if (D == 64) return launch_k(pdl, causal_attn_mma_kernel<64>, agrid, dim3(LLM_MMA_THREADS), LlmAttnMmaSmem<64>::BYTES, s, (const bf16*)qkv, att, rope, kc, vc, L, heads, kvh, sl2);
                       return launch_k(pdl, causal_attn_mma_kernel<128>, agrid, dim3(LLM_MMA_THREADS), LlmAttnMmaSmem<128>::BYTES, s, (const bf16*)qkv, att, rope, kc, vc, L, heads, kvh, sl2);
                   }, "causal_attn_mma_kernel", 0, 2.0 * (double)L * L * HD, 2.0 * L * (NQ + HD));
        }
        if ((rc = add_gemm_l(att, HD, w[3], nullptr, xc, xx, L, H, HD)) != FVHD_OK) return rc;
        const bf16* x2 = xx;
        pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t { return launch_k(pdl, rmsnorm_kernel, dim3(ln_grid), dim3(256), 0, s, x2, xn, ln2, L, H, eps); },
               "rmsnorm_kernel", 0, 0.0, 4.0 * L * H);
        if ((rc = add_gemm_l(xn, H, w[5], nullptr, nullptr, gu, L, 2 * I, H)) != FVHD_OK) return rc;
        const int sgrid = (int)std::min<long>(((long)L * (I / 8) + 255) / 256, 1184);
        pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t { return launch_k(pdl, silu_mul_kernel, dim3(sgrid), dim3(256), 0, s, (const bf16*)gu, hm, L, I); },
               "silu_mul_kernel", 0, 0.0, 6.0 * L * I);
        if ((rc = add_gemm_l(hm, I, w[6], nullptr, xx, S->x2, L, H, I)) != FVHD_OK) return rc;
        xc = S->x2;                              // the input buffer x0 is only ever read: a prefill can be replayed
    }
    const float* fn = (const float*)S->w[(size_t)c.layers * 7];
    const void* lm = S->w[(size_t)c.layers * 7 + 1];
    const bf16* last = xc + (size_t)(L - 1) * H;
    bf16 *xn = S->xn, *logits = S->logits;
    int* tok = S->token;
    const float eps = c.rms_eps;
    const int V = c.vocab;
    pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t { return launch_k(pdl, rmsnorm_kernel, dim3(1), dim3(256), 0, s, last, xn, fn, 1, H, eps); },
           "rmsnorm_kernel", 0, 0.0, 4.0 * H);
    if ((rc = add_gemm_l(xn, H, lm, nullptr, nullptr, logits, 1, V, H)) != FVHD_OK) return rc;
    pl.add([=](cudaStream_t s, const RunCtx&) -> cudaError_t { return launch_k(pdl, argmax_kernel, dim3(1), dim3(1024), 0, s, (const bf16*)logits, V, tok); },
           "argmax_kernel", 0, 0.0, 2.0 * V);
    return FVHD_OK;
}

void destroy_plans(fvhd_handle h) {
    for (auto& kv : h->plans)
        for (auto& g : kv.second.graphs) cudaGraphExecDestroy(g.second);
    h->plans.clear();
}

}  // namespace

extern "C" {

int fvhd_api_version(void) { return FVHD_API_VERSION; }

const char* fvhd_last_error(fvhd_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int fvhd_create(const fvhd_config* cfg, fvhd_handle* out) {
    if (!cfg || !out) return fail(nullptr, FVHD_ERR_INVALID, "null argument");
    if (cfg->image_size < 64 || cfg->image_size % 64) return fail(nullptr, FVHD_ERR_INVALID, "image_size must be a positive multiple of 64 (got %d)", cfg->image_size);
    if (cfg->projector_hidden < 0 || cfg->projector_hidden % 8) return fail(nullptr, FVHD_ERR_INVALID, "projector_hidden must be a multiple of 8 (got %d)", cfg->projector_hidden);
    if (cfg->projector_hidden > 0 && cfg->projector_depth != 1 && cfg->projector_depth != 2)
        return fail(nullptr, FVHD_ERR_INVALID, "projector_depth must be 1 or 2 (mlp{N}x_gelu), got %d", cfg->projector_depth);
    if (cfg->max_batch < 1) return fail(nullptr, FVHD_ERR_INVALID, "max_batch must be >= 1");
    fvhd_handle h = new fvhd_handle_s();
    h->cfg = *cfg;
    h->opt = read_options();
    h->R = cfg->image_size;
    h->ntok = (cfg->image_size / FVHD_PATCH) * (cfg->image_size / FVHD_PATCH);
    build_arch(h);
    *out = h;
    return FVHD_OK;
}

int fvhd_destroy(fvhd_handle h) {
    if (h) {
        destroy_plans(h);
        if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
        if (h->splitk_ws) cudaFree(h->splitk_ws);
        if (h->splitk_cnt) cudaFree(h->splitk_cnt);
        if (h->stage_in) cudaFree(h->stage_in);
        if (h->stage_out) cudaFree(h->stage_out);
        for (auto& kv : h->rs_tables) { cudaFree(kv.second.bounds); cudaFree(kv.second.kk); }
        if (h->rs_tmp) cudaFree(h->rs_tmp);
        if (h->rs_src) cudaFree(h->rs_src);
        if (h->rs_lut) cudaFree(h->rs_lut);
        if (h->llm) { llm_free(h->llm); delete h->llm; }
    }
    delete h;
    return FVHD_OK;
}

int fvhd_num_weights(fvhd_handle h) { return h ? (int)h->specs.size() : FVHD_ERR_INVALID; }

int fvhd_weight_spec(fvhd_handle h, int i, const char** name, int* dtype, int64_t* numel) {
    if (!h || i < 0 || i >= (int)h->specs.size()) return FVHD_ERR_INVALID;
    if (name) *name = h->specs[i].name.c_str();
    if (dtype) *dtype = h->specs[i].dtype;
    if (numel) *numel = h->specs[i].numel;
    return FVHD_OK;
}

int fvhd_load_weights(fvhd_handle h, const fvhd_tensor* table, int n) {
    if (!h || !table) return FVHD_ERR_INVALID;
    std::map<std::string, const fvhd_tensor*> got;
    for (int i = 0; i < n; ++i) {
        if (!table[i].name) return fail(h, FVHD_ERR_WEIGHTS, "weight table entry %d has no name", i);
        got[table[i].name] = &table[i];
    }
    std::map<std::string, const void*> wp;
    for (const WeightSpec& s : h->specs) {
        auto it = got.find(s.name);
        if (it == got.end()) return fail(h, FVHD_ERR_WEIGHTS, "missing weight tensor '%s'", s.name.c_str());
        const fvhd_tensor* t = it->second;
        if (t->dtype != s.dtype || t->numel != s.numel)
            return fail(h, FVHD_ERR_WEIGHTS, "weight '%s': expected dtype %d numel %lld, got dtype %d numel %lld", s.name.c_str(), s.dtype,
                        (long long)s.numel, t->dtype, (long long)t->numel);
        if (!t->data || ((uintptr_t)t->data & 15)) return fail(h, FVHD_ERR_WEIGHTS, "weight '%s': device pointer must be non-null and 16-B aligned", s.name.c_str());
        wp[s.name] = t->data;
    }
    h->wptr.swap(wp);
    destroy_plans(h);
    h->loaded = true;
    return FVHD_OK;
}

size_t fvhd_workspace_bytes(fvhd_handle h, int batch) {
    if (!h || batch < 1) return 0;
    const int bc = batch < h->cfg.max_batch ? batch : h->cfg.max_batch;
    return workspace_bytes(h, bc);
}

int fvhd_set_workspace(fvhd_handle h, void* dptr, size_t bytes) {
    if (!h) return FVHD_ERR_INVALID;
    h->ws = dptr;
    h->ws_bytes = bytes;
    destroy_plans(h);
    return FVHD_OK;
}

int fvhd_num_tokens(fvhd_handle h) { return h ? h->ntok : FVHD_ERR_INVALID; }
int fvhd_out_dim(fvhd_handle h) { return h ? (h->cfg.projector_hidden > 0 ? h->cfg.projector_hidden : FVHD_EMBED_DIM) : FVHD_ERR_INVALID; }
int fvhd_num_units(fvhd_handle h) { return h ? (int)h->units.size() : FVHD_ERR_INVALID; }

int fvhd_unit_info(fvhd_handle h, int u, const char** name, int64_t* in_elems, int64_t* out_elems, int* out_h, int* out_w, int* out_c,
                   double* flops, double* min_bytes) {
    if (!h || u < 0 || u >= (int)h->units.size()) return FVHD_ERR_INVALID;
    const UnitDesc& d = h->units[u];
    if (name) *name = d.name.c_str();
    if (in_elems) *in_elems = d.in_elems;
    if (out_elems) *out_elems = d.out_elems;
    if (out_h) *out_h = d.hout;
    if (out_w) *out_w = d.wout;
    if (out_c) *out_c = d.cout;
    if (flops) *flops = d.flops;
    if (min_bytes) *min_bytes = d.min_bytes;
    return FVHD_OK;
}

int fvhd_launches_per_forward(fvhd_handle h, int batch) {
    if (!h || batch < 1) return FVHD_ERR_INVALID;
    // kernels of one pass over `bc` images (the plan build_plan makes for that batch size), + set_io_kernel
    auto pass_launches = [&](int bc) {
        int steps = 0;
        for (const UnitDesc& u : h->units) {
            switch (u.kind) {
            case 0: steps += 2; break;
            case 1: steps += choose_convffn(h, bc * u.hout * u.wout, u.cin) == ConvFfn::TwoGemms ? 3 : 2; break;   // mixer + ConvFFN
            case 2: steps += 2; break;
            case 3: steps += 1; break;
            case 4: steps += 7; break;
            case 5: steps += 4; break;   // dw + pool + reduce + expand
            case 6: steps += h->cfg.projector_depth; break;
            }
        }
        return steps + 1;
    };
    // fvhd_forward walks the batch in passes of max_batch images, the last one possibly smaller
    const int full = batch / h->cfg.max_batch, rem = batch % h->cfg.max_batch;
    return full * pass_launches(h->cfg.max_batch) + (rem ? pass_launches(rem) : 0);
}

}  // extern "C"

namespace {
int forward_impl(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch, void* tokens, void* projected,
                 long long out_image_stride, void* const* peer_out, int n_peers, void* const* scatter = nullptr);
}

extern "C" {

int fvhd_forward(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch, void* tokens, void* projected) {
    return forward_impl(h, stream, images, img_dtype, batch, tokens, projected, 0, nullptr, 0);
}

int fvhd_forward_strided(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch, void* tokens, void* projected,
                         long long out_image_stride) {
    return forward_impl(h, stream, images, img_dtype, batch, tokens, projected, out_image_stride, nullptr, 0);
}

int fvhd_forward_gather(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch, void* local_out,
                        void* const* peer_out, int n_peers) {
    if (!h) return FVHD_ERR_INVALID;
    if (h->cfg.projector_hidden <= 0) return fail(h, FVHD_ERR_INVALID, "fvhd_forward_gather needs a plan with a projector (the gathered tensor is the projected tokens)");
    if (n_peers < 0 || n_peers > FVHD_MAX_PEERS) return fail(h, FVHD_ERR_INVALID, "n_peers %d outside [0, %d]", n_peers, FVHD_MAX_PEERS);
    if (n_peers > 0 && !peer_out) return fail(h, FVHD_ERR_INVALID, "peer_out is null");
    for (int i = 0; i < n_peers; ++i)
        if (!peer_out[i] || ((uintptr_t)peer_out[i] & 15)) return fail(h, FVHD_ERR_INVALID, "peer_out[%d] must be a non-null, 16-B aligned device pointer", i);
    if (!local_out) return fail(h, FVHD_ERR_INVALID, "local_out is null");
    return forward_impl(h, stream, images, img_dtype, batch, nullptr, local_out, 0, peer_out, n_peers);
}

int fvhd_forward_scatter(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch, void* const* dst_per_image) {
    if (!h) return FVHD_ERR_INVALID;
    if (h->cfg.projector_hidden <= 0) return fail(h, FVHD_ERR_INVALID, "fvhd_forward_scatter needs a plan with a projector");
    if (!dst_per_image) return fail(h, FVHD_ERR_INVALID, "dst_per_image is null");
    if (h->cfg.max_batch > FVHD_MAX_SCATTER) return fail(h, FVHD_ERR_INVALID, "fvhd_forward_scatter supports max_batch <= %d", FVHD_MAX_SCATTER);
    for (int i = 0; i < batch; ++i)
        if (!dst_per_image[i] || ((uintptr_t)dst_per_image[i] & 15)) return fail(h, FVHD_ERR_INVALID, "dst_per_image[%d] must be a non-null, 16-B aligned device pointer", i);
    return forward_impl(h, stream, images, img_dtype, batch, nullptr, dst_per_image[0], 0, nullptr, 0, dst_per_image);
}

}  // extern "C"

namespace {
int forward_impl(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch, void* tokens, void* projected,
                 long long out_image_stride, void* const* peer_out, int n_peers, void* const* scatter) {
    int rc = check_ready(h, batch);
    if (rc != FVHD_OK) return rc;
    if (!images) return fail(h, FVHD_ERR_INVALID, "images is null");
    if (img_dtype < FVHD_F32 || img_dtype > FVHD_BF16) return fail(h, FVHD_ERR_INVALID, "unsupported image dtype %d", img_dtype);
    const bool has_proj = h->cfg.projector_hidden > 0;
    if (projected && !has_proj) return fail(h, FVHD_ERR_INVALID, "projected output requested but the plan has no projector");
    if (!tokens && !projected) return fail(h, FVHD_ERR_INVALID, "both outputs are null");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const size_t img_stride = (size_t)3 * h->R * h->R * dtype_size(img_dtype);
    const size_t tok_stride = (size_t)h->ntok * FVHD_EMBED_DIM * 2;
    const int nunits = (int)h->units.size();
    // final output (projected tokens, or tower tokens when the plan has no projector): dense, or `out_image_stride`
    // elements between images (>= tokens-per-image * dim) when the destination is an LLM embedding buffer
    const long long dense_final = (long long)h->ntok * (has_proj ? h->cfg.projector_hidden : FVHD_EMBED_DIM);
    if (out_image_stride != 0 && out_image_stride < dense_final)
        return fail(h, FVHD_ERR_INVALID, "out_image_stride %lld < tokens * dim = %lld", out_image_stride, dense_final);
    const long long final_stride = out_image_stride ? out_image_stride : dense_final;
    const size_t prj_stride = (size_t)final_stride * 2;
    const int tok_unit = has_proj ? nunits - 2 : nunits - 1;
    for (int b0 = 0; b0 < batch; b0 += h->cfg.max_batch) {
        const int bc = (batch - b0) < h->cfg.max_batch ? (batch - b0) : h->cfg.max_batch;
        Plan* pl;
        if ((rc = get_plan(h, bc, &pl)) != FVHD_OK) return rc;
        RunCtx ctx;
        ctx.img_dtype = img_dtype;
        const void* img = reinterpret_cast<const uint8_t*>(images) + (size_t)b0 * img_stride;
        uint8_t* tok_dst = tokens ? reinterpret_cast<uint8_t*>(tokens) + (size_t)b0 * (has_proj ? tok_stride : (size_t)final_stride * 2) : nullptr;
        uint8_t* prj_dst = projected ? reinterpret_cast<uint8_t*>(projected) + (size_t)b0 * prj_stride : nullptr;
        if (has_proj) {
            // tokens stay in the workspace (the projector's TMA map points there); copied out if requested
            const int last_unit = projected ? nunits - 1 : nunits - 2;
            PeerList peers{};
            peers.n = n_peers;
            for (int i = 0; i < n_peers; ++i) peers.p[i] = reinterpret_cast<uint8_t*>(peer_out[i]) + (size_t)b0 * prj_stride;
            ScatterList sc{};
            if (scatter) { sc.n = bc; for (int i = 0; i < bc; ++i) sc.p[i] = scatter[b0 + i]; }
            if ((rc = set_io(h, *pl, st, img, prj_dst, tok_dst, final_stride, &peers, &sc)) != FVHD_OK) return rc;
            if ((rc = run_forward(h, *pl, st, ctx, pl->unit_steps[last_unit].second, tok_dst ? pl->unit_out[tok_unit] : nullptr,
                                  (size_t)bc * tok_stride)) != FVHD_OK) return rc;
        } else {
            if ((rc = set_io(h, *pl, st, img, tok_dst, nullptr, final_stride)) != FVHD_OK) return rc;
            if ((rc = run_forward(h, *pl, st, ctx, (int)pl->steps.size(), nullptr, 0)) != FVHD_OK) return rc;
        }
    }
    return FVHD_OK;
}
}  // namespace

extern "C" {

int fvhd_encode_images_host(fvhd_handle h, void* stream, const void* host_images, int img_dtype, int batch, void* host_out) {
    int rc = check_ready(h, batch);
    if (rc != FVHD_OK) return rc;
    if (!host_images || !host_out) return fail(h, FVHD_ERR_INVALID, "null host buffer");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);      // batches above max_batch run in passes inside fvhd_forward
    const size_t img_bytes = (size_t)batch * 3 * h->R * h->R * dtype_size(img_dtype);
    const size_t out_bytes = (size_t)batch * h->ntok * fvhd_out_dim(h) * 2;
    // device staging owned by the handle (grown on demand)
    if (h->stage_in_bytes < img_bytes) {
        if (h->stage_in) cudaFree(h->stage_in);
        h->stage_in = nullptr; h->stage_in_bytes = 0;
        CUDA_TRY(h, cudaMalloc(&h->stage_in, img_bytes));
        h->stage_in_bytes = img_bytes;
    }
    if (h->stage_out_bytes < out_bytes) {
        if (h->stage_out) cudaFree(h->stage_out);
        h->stage_out = nullptr; h->stage_out_bytes = 0;
        CUDA_TRY(h, cudaMalloc(&h->stage_out, out_bytes));
        h->stage_out_bytes = out_bytes;
    }
    void* stage_in = h->stage_in;
    void* stage_out = h->stage_out;
    CUDA_TRY(h, cudaMemcpyAsync(stage_in, host_images, img_bytes, cudaMemcpyHostToDevice, st));
    const bool has_proj = h->cfg.projector_hidden > 0;
    rc = fvhd_forward(h, stream, stage_in, img_dtype, batch, has_proj ? nullptr : stage_out, has_proj ? stage_out : nullptr);
    if (rc != FVHD_OK) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(host_out, stage_out, out_bytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    return FVHD_OK;
}

int fvhd_run_units(fvhd_handle h, void* stream, int first, int last, const void* in, int img_dtype, int batch, void* out) {
    int rc = check_ready(h, batch);
    if (rc != FVHD_OK) return rc;
    const int nunits = (int)h->units.size();
    if (first < 0 || last >= nunits || first > last) return fail(h, FVHD_ERR_INVALID, "bad unit range [%d, %d]", first, last);
    if (batch > h->cfg.max_batch) return fail(h, FVHD_ERR_INVALID, "fvhd_run_units: batch %d > max_batch %d", batch, h->cfg.max_batch);
    if (!in || !out) return fail(h, FVHD_ERR_INVALID, "null buffer");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Plan* pl;
    if ((rc = get_plan(h, batch, &pl)) != FVHD_OK) return rc;
    RunCtx ctx;
    ctx.img_dtype = img_dtype;
    if (first > 0)
        CUDA_TRY(h, cudaMemcpyAsync(pl->unit_in[first], in, (size_t)batch * h->units[first].in_elems * 2, cudaMemcpyDeviceToDevice, st));
    const size_t out_bytes = (size_t)batch * h->units[last].out_elems * 2;
    // the last unit of the plan writes straight to the caller's buffer; earlier units are copied out of the workspace
    if ((rc = set_io(h, *pl, st, in, last == nunits - 1 ? out : nullptr, nullptr, h->units[nunits - 1].out_elems)) != FVHD_OK) return rc;
    if ((rc = run_steps(h, *pl, pl->unit_steps[first].first, pl->unit_steps[last].second, st, ctx)) != FVHD_OK) return rc;
    if (last != nunits - 1) CUDA_TRY(h, cudaMemcpyAsync(out, pl->unit_out[last], out_bytes, cudaMemcpyDeviceToDevice, st));
    return FVHD_OK;
}

int fvhd_profile_units(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch, float* ms, int n_ms) {
    int rc = check_ready(h, batch);
    if (rc != FVHD_OK) return rc;
    const int nunits = (int)h->units.size();
    if (!ms || n_ms < nunits) return fail(h, FVHD_ERR_INVALID, "ms buffer too small (%d < %d)", n_ms, nunits);
    if (batch > h->cfg.max_batch) return fail(h, FVHD_ERR_INVALID, "fvhd_profile_units: batch %d > max_batch %d", batch, h->cfg.max_batch);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Plan* pl;
    if ((rc = get_plan(h, batch, &pl)) != FVHD_OK) return rc;
    std::vector<cudaEvent_t> ev(nunits + 1);
    for (auto& e : ev) CUDA_TRY(h, cudaEventCreate(&e));
    RunCtx ctx;
    ctx.img_dtype = img_dtype;
    if ((rc = set_io(h, *pl, st, images, pl->unit_out[nunits - 1], nullptr, h->units[nunits - 1].out_elems)) != FVHD_OK) return rc;   // result stays in the workspace
    CUDA_TRY(h, cudaEventRecord(ev[0], st));
    for (int u = 0; u < nunits; ++u) {
        if ((rc = run_steps(h, *pl, pl->unit_steps[u].first, pl->unit_steps[u].second, st, ctx)) != FVHD_OK) return rc;
        CUDA_TRY(h, cudaEventRecord(ev[u + 1], st));
    }
    CUDA_TRY(h, cudaStreamSynchronize(st));
    for (int u = 0; u < nunits; ++u) CUDA_TRY(h, cudaEventElapsedTime(&ms[u], ev[u], ev[u + 1]));
    for (auto& e : ev) cudaEventDestroy(e);
    return FVHD_OK;
}

int fvhd_num_steps(fvhd_handle h, int batch) {
    int rc = check_ready(h, batch);
    if (rc != FVHD_OK) return rc;
    Plan* pl;
    if ((rc = get_plan(h, batch, &pl)) != FVHD_OK) return rc;
    return (int)pl->steps.size();
}

int fvhd_step_info(fvhd_handle h, int batch, int i, const char** kernel, int* unit, double* flops, double* bytes) {
    int rc = check_ready(h, batch);
    if (rc != FVHD_OK) return rc;
    Plan* pl;
    if ((rc = get_plan(h, batch, &pl)) != FVHD_OK) return rc;
    if (i < 0 || i >= (int)pl->info.size()) return fail(h, FVHD_ERR_INVALID, "step %d out of range", i);
    if (kernel) *kernel = pl->info[i].kernel;
    if (unit) *unit = pl->info[i].unit;
    if (flops) *flops = pl->info[i].flops;
    if (bytes) *bytes = pl->info[i].bytes;
    return FVHD_OK;
}

int fvhd_profile_steps(fvhd_handle h, void* stream, const void* images, int img_dtype, int batch, float* ms, int n_ms) {
    int rc = check_ready(h, batch);
    if (rc != FVHD_OK) return rc;
    if (batch > h->cfg.max_batch) return fail(h, FVHD_ERR_INVALID, "fvhd_profile_steps: batch %d > max_batch %d", batch, h->cfg.max_batch);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    Plan* pl;
    if ((rc = get_plan(h, batch, &pl)) != FVHD_OK) return rc;
    const int n = (int)pl->steps.size();
    if (!ms || n_ms < n) return fail(h, FVHD_ERR_INVALID, "ms buffer too small (%d < %d)", n_ms, n);
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) CUDA_TRY(h, cudaEventCreate(&e));
    RunCtx ctx;
    ctx.img_dtype = img_dtype;
    if ((rc = set_io(h, *pl, st, images, pl->unit_out[h->units.size() - 1], nullptr, h->units[h->units.size() - 1].out_elems)) != FVHD_OK) return rc;
    CUDA_TRY(h, cudaEventRecord(ev[0], st));
    for (int i = 0; i < n; ++i) {
        if ((rc = run_steps(h, *pl, i, i + 1, st, ctx)) != FVHD_OK) return rc;
        CUDA_TRY(h, cudaEventRecord(ev[i + 1], st));
    }
    CUDA_TRY(h, cudaStreamSynchronize(st));
    for (int i = 0; i < n; ++i) CUDA_TRY(h, cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
    for (auto& e : ev) cudaEventDestroy(e);
    return FVHD_OK;
}

// ---------------------------------------------------------------- row f1: preprocessing
int fvhd_resample_coeffs(int in_size, int out_size, int* bounds, int* kk, int kk_capacity) {
    if (in_size < 1 || out_size < 1) return FVHD_ERR_INVALID;
    std::vector<int> b, k;
    const int ksize = resample_coeffs(in_size, out_size, b, k);
    if (bounds) memcpy(bounds, b.data(), b.size() * sizeof(int));
    if (kk) {
        if ((size_t)kk_capacity < k.size()) return FVHD_ERR_INVALID;
        memcpy(kk, k.data(), k.size() * sizeof(int));
    }
    return ksize;
}

static int rs_get_table(fvhd_handle h, int in_size, int out_size, fvhd_handle_s::RsTable* out) {
    auto key = std::make_pair(in_size, out_size);
    auto it = h->rs_tables.find(key);
    if (it == h->rs_tables.end()) {
        std::vector<int> b, k;
        fvhd_handle_s::RsTable t{};
        t.ksize = resample_coeffs(in_size, out_size, b, k);
        CUDA_TRY(h, cudaMalloc(&t.bounds, b.size() * sizeof(int)));
        CUDA_TRY(h, cudaMalloc(&t.kk, k.size() * sizeof(int)));
        CUDA_TRY(h, cudaMemcpy(t.bounds, b.data(), b.size() * sizeof(int), cudaMemcpyHostToDevice));
        CUDA_TRY(h, cudaMemcpy(t.kk, k.data(), k.size() * sizeof(int), cudaMemcpyHostToDevice));
        it = h->rs_tables.emplace(key, t).first;
    }
    *out = it->second;
    return FVHD_OK;
}

// Shared body of the preprocessing entries: the image (H x W u8 RGB, optionally centred on an Hs x Ws black canvas BEFORE the
// resize = expand2square) is PIL-resized to oh x ow; the result is shown through tiles_y x tiles_x windows of R x R whose first
// one starts at (top, left) of the resized image (pixels outside it are black), x 1/255, NCHW.
static int preprocess_impl(fvhd_handle h, cudaStream_t st, const void* rgb, int src_on_host, int H, int W, int Hs, int Ws, int offy, int offx,
                           int oh, int ow, int top, int left, int tiles_y, int tiles_x, void* out, int out_dtype) {
    int rc;
    const int R = h->R;
    if (!h->rs_lut) {
        float lut[256];
        for (int i = 0; i < 256; ++i) lut[i] = (float)((double)i * (1.0 / 255.0));      // transformers rescale(): float64 multiply
        CUDA_TRY(h, cudaMalloc(&h->rs_lut, sizeof(lut)));
        CUDA_TRY(h, cudaMemcpy(h->rs_lut, lut, sizeof(lut), cudaMemcpyHostToDevice));
    }
    const uint8_t* src = reinterpret_cast<const uint8_t*>(rgb);
    if (src_on_host) {
        const size_t nb = (size_t)H * W * 3;
        if (h->rs_src_bytes < nb) {
            if (h->rs_src) cudaFree(h->rs_src);
            h->rs_src = nullptr; h->rs_src_bytes = 0;
            CUDA_TRY(h, cudaMalloc(&h->rs_src, nb));
            h->rs_src_bytes = nb;
        }
        CUDA_TRY(h, cudaMemcpyAsync(h->rs_src, rgb, nb, cudaMemcpyHostToDevice, st));
        src = h->rs_src;
    }
    const size_t tmp_bytes = (size_t)Hs * ow * 3;
    if (h->rs_tmp_bytes < tmp_bytes) {
        if (h->rs_tmp) cudaFree(h->rs_tmp);
        h->rs_tmp = nullptr; h->rs_tmp_bytes = 0;
        CUDA_TRY(h, cudaMalloc(&h->rs_tmp, tmp_bytes));
        h->rs_tmp_bytes = tmp_bytes;
    }
    fvhd_handle_s::RsTable tx{}, ty{};
    const bool pdl = h->opt.pdl;
    const dim3 g1((ow + 127) / 128, Hs);
    cudaError_t e;
    if (ow != Ws) {
        if ((rc = rs_get_table(h, Ws, ow, &tx)) != FVHD_OK) return rc;
        e = launch_k(pdl, resample_h_kernel, g1, dim3(128), 0, st, src, H, W, offy, offx, Ws, h->rs_tmp, ow, (const int*)tx.bounds, (const int*)tx.kk, tx.ksize);
    } else {
        e = launch_k(pdl, pad_copy_kernel, g1, dim3(128), 0, st, src, H, W, offy, offx, h->rs_tmp, ow);
    }
    if (e != cudaSuccess) return fail(h, FVHD_ERR_CUDA, "preprocess horizontal pass: %s", cudaGetErrorString(e));
    // vertical pass (identity table when oh == Hs: one tap of weight 1 << 22 -> exact copy)
    if ((rc = rs_get_table(h, Hs, oh, &ty)) != FVHD_OK) return rc;
    const int* yb = (const int*)ty.bounds; const int* yk = (const int*)ty.kk; const float* lut = (const float*)h->rs_lut; const uint8_t* tmp = (const uint8_t*)h->rs_tmp;
    if (tiles_y * tiles_x == 1 && top >= 0 && left >= 0 && top + R <= oh && left + R <= ow) {       // one window inside the image
        const dim3 g2((R + 127) / 128, R);
        if (out_dtype == FVHD_F32) e = launch_k(pdl, resample_v_crop_kernel<float>, g2, dim3(128), 0, st, tmp, ow, (float*)out, R, top, left, yb, yk, ty.ksize, lut);
        else if (out_dtype == FVHD_F16) e = launch_k(pdl, resample_v_crop_kernel<__half>, g2, dim3(128), 0, st, tmp, ow, (__half*)out, R, top, left, yb, yk, ty.ksize, lut);
        else e = launch_k(pdl, resample_v_crop_kernel<bf16>, g2, dim3(128), 0, st, tmp, ow, (bf16*)out, R, top, left, yb, yk, ty.ksize, lut);
    } else {                                                                                         // tiles of a canvas: black outside the image
        const dim3 g2((R + 127) / 128, R, tiles_y * tiles_x);
        if (out_dtype == FVHD_F32) e = launch_k(pdl, resample_v_tiles_kernel<float>, g2, dim3(128), 0, st, tmp, ow, oh, (float*)out, R, top, left, tiles_x, yb, yk, ty.ksize, lut);
        else if (out_dtype == FVHD_F16) e = launch_k(pdl, resample_v_tiles_kernel<__half>, g2, dim3(128), 0, st, tmp, ow, oh, (__half*)out, R, top, left, tiles_x, yb, yk, ty.ksize, lut);
        else e = launch_k(pdl, resample_v_tiles_kernel<bf16>, g2, dim3(128), 0, st, tmp, ow, oh, (bf16*)out, R, top, left, tiles_x, yb, yk, ty.ksize, lut);
    }
    if (e != cudaSuccess) return fail(h, FVHD_ERR_CUDA, "preprocess vertical pass: %s", cudaGetErrorString(e));
    return FVHD_OK;
}

int fvhd_preprocess(fvhd_handle h, void* stream, const void* rgb, int src_on_host, int H, int W, int pad_to_square, void* out, int out_dtype) {
    if (!h) return FVHD_ERR_INVALID;
    int rc = ensure_cuda(h);
    if (rc != FVHD_OK) return rc;
    if (!rgb || !out || H < 1 || W < 1) return fail(h, FVHD_ERR_INVALID, "fvhd_preprocess: bad image %dx%d", H, W);
    if (out_dtype < FVHD_F32 || out_dtype > FVHD_BF16) return fail(h, FVHD_ERR_INVALID, "fvhd_preprocess: bad output dtype %d", out_dtype);
    const int R = h->R;
    // expand2square (mm_utils.py:154-165): canvas Hs x Ws with the image at (offy, offx)
    const int Hs = pad_to_square ? (H > W ? H : W) : H, Ws = pad_to_square ? Hs : W;
    const int offy = pad_to_square && W > H ? (W - H) / 2 : 0, offx = pad_to_square && H > W ? (H - W) / 2 : 0;
    // get_resize_output_image_size(size = R, default_to_square = False)
    const int shortE = Ws <= Hs ? Ws : Hs, longE = Ws <= Hs ? Hs : Ws;
    const int new_long = (int)((double)R * longE / shortE);
    const int oh = Ws <= Hs ? new_long : R, ow = Ws <= Hs ? R : new_long;
    const int top = (oh - R) / 2, left = (ow - R) / 2;
    return preprocess_impl(h, reinterpret_cast<cudaStream_t>(stream), rgb, src_on_host, H, W, Hs, Ws, offy, offx, oh, ow, top, left, 1, 1, out, out_dtype);
}

int fvhd_preprocess_tiles(fvhd_handle h, void* stream, const void* rgb, int src_on_host, int H, int W, int new_h, int new_w,
                          int pad_y, int pad_x, int tiles_y, int tiles_x, void* out, int out_dtype) {
    if (!h) return FVHD_ERR_INVALID;
    int rc = ensure_cuda(h);
    if (rc != FVHD_OK) return rc;
    if (!rgb || !out || H < 1 || W < 1 || new_h < 1 || new_w < 1 || tiles_y < 1 || tiles_x < 1 || pad_y < 0 || pad_x < 0)
        return fail(h, FVHD_ERR_INVALID, "fvhd_preprocess_tiles: bad geometry %dx%d -> %dx%d, pad (%d,%d), tiles %dx%d", H, W, new_h, new_w, pad_y, pad_x, tiles_y, tiles_x);
    if (out_dtype < FVHD_F32 || out_dtype > FVHD_BF16) return fail(h, FVHD_ERR_INVALID, "fvhd_preprocess_tiles: bad output dtype %d", out_dtype);
    // the canvas pixel (y, x) shows resized-image pixel (y - pad_y, x - pad_x): the first tile starts at (-pad_y, -pad_x)
    return preprocess_impl(h, reinterpret_cast<cudaStream_t>(stream), rgb, src_on_host, H, W, H, W, 0, 0, new_h, new_w, -pad_y, -pad_x, tiles_y, tiles_x, out, out_dtype);
}

int fvhd_debug_gemm_trace(void* dev_buf_16_u64_per_cta, int force_bn, int max_cs) {
    g_gemm_trace = reinterpret_cast<unsigned long long*>(dev_buf_16_u64_per_cta);
    g_force_bn = force_bn;
    if (max_cs == 1 || max_cs == 2 || max_cs == 4) g_debug_gemm_cs = max_cs;
    return FVHD_OK;
}

int fvhd_debug_mixer_trace(void* dev_buf_8_u64_per_cta) {
    unsigned long long* p = reinterpret_cast<unsigned long long*>(dev_buf_8_u64_per_cta);
    return cudaMemcpyToSymbol(d_mix_trace, &p, sizeof(p)) == cudaSuccess ? FVHD_OK : FVHD_ERR_CUDA;
}

int fvhd_gemm(fvhd_handle h, void* stream, const void* A, const void* W, const void* bias, const void* residual, void* D, int M, int N, int K, int act) {
    if (!h) return FVHD_ERR_INVALID;
    int rc = ensure_cuda(h);
    if (rc != FVHD_OK) return rc;
    Step s;
    if ((rc = make_gemm_step(h, &s, nullptr, 1, (const bf16*)A, K, (const bf16*)W, (const float*)bias, (const bf16*)residual, N, (bf16*)D, N, M, N, K, act)) != FVHD_OK) return rc;
    if (!D) return fail(h, FVHD_ERR_INVALID, "D is null");
    return launch_step(h, s, stream, "gemm");
}

int fvhd_convffn_half(fvhd_handle h, void* stream, const void* z, const void* w1, const void* b1, const void* w2, int w2_is_f16, const void* b2,
                  const void* resid, void* out, int M, int C) {
    if (!h) return FVHD_ERR_INVALID;
    int rc = ensure_cuda(h);
    if (rc != FVHD_OK) return rc;
    if (!z || !w1 || !b1 || !w2 || !b2 || !resid || !out || M <= 0) return fail(h, FVHD_ERR_INVALID, "fvhd_convffn_half: null operand or M <= 0");
    Step s;
    if ((rc = make_convffn2_step(h, &s, (const bf16*)z, (const bf16*)w1, (const float*)b1, w2, w2_is_f16, (const float*)b2,
                                 (const bf16*)resid, (bf16*)out, M, C)) != FVHD_OK) return rc;
    return launch_step(h, s, stream, "convffn2");
}

int fvhd_attention(fvhd_handle h, void* stream, const void* qkv, void* out, int batch, int N, int C) {
    if (!h) return FVHD_ERR_INVALID;
    int rc = ensure_cuda(h);
    if (rc != FVHD_OK) return rc;
    if (!qkv || !out || batch < 1 || N < 1 || C < 32 || C % 32) return fail(h, FVHD_ERR_INVALID, "fvhd_attention: bad arguments");
    const float sl2 = 0.17677669529663687f * 1.4426950408889634f;
    Step s;
    if ((rc = (h->opt.attn == 'u' ? make_attention_umma_step : make_attention_mma_step)(h, &s, (const bf16*)qkv, (bf16*)out, batch, N, C, sl2)) != FVHD_OK)
        return rc;
    return launch_step(h, s, stream, "attention");
}

int fvhd_mixer(fvhd_handle h, void* stream, const void* x, const void* w3, const void* b3, const void* w7, const void* b7,
               void* y, void* z, int batch, int H, int W, int C) {
    if (!h) return FVHD_ERR_INVALID;
    int rc = ensure_cuda(h);
    if (rc != FVHD_OK) return rc;
    if (!x || !w3 || !b3 || !w7 || !b7 || !y || !z || batch < 1 || H < 1 || W < 1) return fail(h, FVHD_ERR_INVALID, "fvhd_mixer: null operand or empty shape");
    const char m = h->opt.mixer;
    const Mixer k = m == '2' ? Mixer::Tc2 : m == 't' ? Mixer::Tc : (m == 0 || m == 'z') ? Mixer::Tz : Mixer::Umma;
    Step s;
    if ((rc = kMixers[(int)k].make(h, &s, (const bf16*)x, (bf16*)y, (bf16*)z, (const float*)w3, (const float*)b3, (const float*)w7,
                                   (const float*)b7, batch, H, W, C)) != FVHD_OK) return rc;
    return launch_step(h, s, stream, "mixer");
}

int fvhd_convffn(fvhd_handle h, void* stream, const void* z, const void* w1, const void* b1, const void* w2, const void* b2,
                 const void* resid, void* out, int M, int C, void* trace_64_u64_per_cta) {
    if (!h) return FVHD_ERR_INVALID;
    int rc = ensure_cuda(h);
    if (rc != FVHD_OK) return rc;
    if (!z || !w1 || !b1 || !w2 || !b2 || !resid || !out || M <= 0) return fail(h, FVHD_ERR_INVALID, "fvhd_convffn: null operand or M <= 0");
    Step s;
    if (C == MLPC_C) {
        rc = make_cluster_mlp_step(h, &s, (const bf16*)z, (const bf16*)w1, (const float*)b1, (const bf16*)w2, (const float*)b2,
                                   (const bf16*)resid, (bf16*)out, M, (unsigned long long*)trace_64_u64_per_cta);
    } else if (C == 96 || C == 192) {
        rc = make_fused_mlp_step(h, &s, (const bf16*)z, (const bf16*)w1, (const float*)b1, (const bf16*)w2, (const float*)b2,
                                 (const bf16*)resid, (bf16*)out, M, C);
    } else {
        return fail(h, FVHD_ERR_INVALID, "fvhd_convffn: fused ConvFFN kernels exist for C in {96, 192, 384}, got %d", C);
    }
    if (rc != FVHD_OK) return rc;
    return launch_step(h, s, stream, "convffn");
}


// ------------------------------------------------------------------ row f3: LLM prefill
int fvhd_llm_load(fvhd_handle h, const fvhd_llm_config* cfg, const void* const* weights, int n_weights) {
    if (!h || !cfg || !weights) return FVHD_ERR_INVALID;
    int rc = ensure_cuda(h);
    if (rc != FVHD_OK) return rc;
    const fvhd_llm_config& c = *cfg;
    if (c.hidden < 8 || c.hidden % 8 || c.layers < 1 || c.heads < 1 || c.kv_heads < 1 || c.heads % c.kv_heads || (c.head_dim != 64 && c.head_dim != 128) ||
        c.intermediate % 8 || c.vocab % 8 || c.max_seq < 1)
        return fail(h, FVHD_ERR_INVALID, "fvhd_llm_load: unsupported config (hidden %d, heads %d / %d, head_dim %d, intermediate %d, vocab %d)", c.hidden, c.heads,
                    c.kv_heads, c.head_dim, c.intermediate, c.vocab);
    if (n_weights != c.layers * 7 + 2) return fail(h, FVHD_ERR_INVALID, "fvhd_llm_load: expected %d weight pointers, got %d", c.layers * 7 + 2, n_weights);
    for (int i = 0; i < n_weights; ++i)
        if (!weights[i] || ((uintptr_t)weights[i] & 15)) return fail(h, FVHD_ERR_INVALID, "fvhd_llm_load: weight %d is null or not 16-byte aligned", i);
    if (h->llm) { llm_free(h->llm); delete h->llm; h->llm = nullptr; }
    LlmState* S = new LlmState();
    S->c = c;
    S->nqkv = (c.heads + 2 * c.kv_heads) * c.head_dim;
    S->w.assign(weights, weights + n_weights);
    const size_t T = (size_t)c.max_seq;
    auto alloc = [&](void** p, size_t bytes) { return cudaMalloc(p, bytes) == cudaSuccess; };
    bool ok = alloc((void**)&S->x0, T * c.hidden * 2) && alloc((void**)&S->x1, T * c.hidden * 2) && alloc((void**)&S->x2, T * c.hidden * 2) &&
              alloc((void**)&S->xn, T * c.hidden * 2) &&
              alloc((void**)&S->qkv, T * S->nqkv * 2) && alloc((void**)&S->att, T * c.heads * c.head_dim * 2) && alloc((void**)&S->gu, T * 2 * c.intermediate * 2) &&
              alloc((void**)&S->hm, T * c.intermediate * 2) && alloc((void**)&S->logits, (size_t)c.vocab * 2) &&
              alloc((void**)&S->kc, (size_t)c.layers * T * c.kv_heads * c.head_dim * 2) && alloc((void**)&S->vc, (size_t)c.layers * T * c.kv_heads * c.head_dim * 2) &&
              alloc((void**)&S->rope, T * (c.head_dim / 2) * sizeof(float2)) && alloc((void**)&S->token, sizeof(int));
    if (!ok) { (void)cudaGetLastError(); llm_free(S); delete S; return fail(h, FVHD_ERR_CUDA, "fvhd_llm_load: out of device memory"); }
    const int n = c.max_seq * (c.head_dim / 2);
    rope_table_kernel<<<(n + 255) / 256, 256>>>(S->rope, c.max_seq, c.head_dim / 2, c.rope_theta);
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaDeviceSynchronize());
    CUDA_TRY(h, set_smem(causal_attn_kernel<64>, LlmAttnSmem<64>::BYTES));
    CUDA_TRY(h, set_smem(causal_attn_kernel<128>, LlmAttnSmem<128>::BYTES));
    CUDA_TRY(h, set_smem(causal_attn_mma_kernel<64>, LlmAttnMmaSmem<64>::BYTES));
    CUDA_TRY(h, set_smem(causal_attn_mma_kernel<128>, LlmAttnMmaSmem<128>::BYTES));
    h->llm = S;
    return FVHD_OK;
}

void* fvhd_llm_input(fvhd_handle h) { return (h && h->llm) ? h->llm->x0 : nullptr; }

int fvhd_llm_kv_cache(fvhd_handle h, void** k_out, void** v_out) {
    if (!h || !h->llm) return FVHD_ERR_INVALID;
    if (k_out) *k_out = h->llm->kc;
    if (v_out) *v_out = h->llm->vc;
    return FVHD_OK;
}

static int llm_plan(fvhd_handle h, int L, Plan** out) {
    LlmState* S = h->llm;
    if (!S) return fail(h, FVHD_ERR_INVALID, "no LLM loaded (fvhd_llm_load)");
    if (L < 1 || L > S->c.max_seq) return fail(h, FVHD_ERR_INVALID, "prefill length %d outside [1, %d]", L, S->c.max_seq);
    auto it = S->plans.find(L);
    if (it == S->plans.end()) {
        Plan pl;
        int rc = build_llm_plan(h, S, L, pl);
        if (rc != FVHD_OK) return rc;
        it = S->plans.emplace(L, std::move(pl)).first;
    }
    *out = &it->second;
    return FVHD_OK;
}

int fvhd_llm_launches(fvhd_handle h, int L) {
    if (!h) return FVHD_ERR_INVALID;
    Plan* pl = nullptr;
    int rc = llm_plan(h, L, &pl);
    return rc != FVHD_OK ? rc : (int)pl->steps.size();
}

int fvhd_llm_prefill(fvhd_handle h, void* stream, int L, void* logits_out, int* token_out) {
    if (!h) return FVHD_ERR_INVALID;
    Plan* pl = nullptr;
    int rc = llm_plan(h, L, &pl);
    if (rc != FVHD_OK) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    RunCtx ctx{};
    if ((rc = run_forward(h, *pl, st, ctx, (int)pl->steps.size(), nullptr, 0)) != FVHD_OK) return rc;
    LlmState* S = h->llm;
    if (logits_out) CUDA_TRY(h, cudaMemcpyAsync(logits_out, S->logits, (size_t)S->c.vocab * 2, cudaMemcpyDeviceToDevice, st));
    if (token_out) CUDA_TRY(h, cudaMemcpyAsync(token_out, S->token, sizeof(int), cudaMemcpyDefault, st));
    return FVHD_OK;
}

}  // extern "C"
