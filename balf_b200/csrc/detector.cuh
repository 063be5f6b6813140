// Detector weights: raw (reference state_dict order) and packed (kernel) layouts.
#pragma once
#include "common.cuh"
#include "../../include/balf_b200.h"

namespace balf {

constexpr int kHeadPad = 128;   // head logits (cell^2+1 = 65) padded to a full output tile

// One ``Down`` stage, in reference registration order (SURVEY.md appendix A).  Every 2-D weight is
// stored TRANSPOSED in the packed blob: wT[in][out], so that a warp reads consecutive outputs.
struct DownW {
    const float *conv0_w, *conv0_b;           // [Cin][C]
    const float *pn_w, *pn_b;                 // LayerNorm before the split projection
    const float *pd1_w, *pd1_b;               // [C][2C]
    struct Branch {
        const float *n_w, *n_b;               // LayerNorm
        const float *d1_w, *d1_b;             // [C][2C]
        const float *gn_w, *gn_b;             // gating-unit LayerNorm
        const float *gd_w, *gd_b;             // [64][64] spatial mixing (transposed: [in token][out token])
        const float *d2_w, *d2_b;             // [C][C]
    } br[2];                                  // 0 = grid (global), 1 = block (local)
    const float *pd2_w, *pd2_b;               // [2C][C]
    const float *rn_w, *rn_b;                 // channel-attention LayerNorm
    const float *rc1_w, *rc1_b, *rc2_w, *rc2_b;   // [C][C]
    const float *ex0_w, *ex0_b;               // [C][C/4]
    const float *ex2_w, *ex2_b;               // [C/4][C]
    const float *c2_w, *c2_b;                 // [C][C] (used by the last stage only)
};
struct HeadW {
    const float *w, *b;                       // [C][kHeadPad], [kHeadPad]  (zero padded)
    const float *alpha, *beta;                // folded eval BatchNorm: logit = z * alpha + beta
};
struct DetW {
    DownW down[4];
    HeadW head;
};

struct Cursor {
    const float* base;
    size_t off;
    const float* take(size_t n) {
        const float* p = base + off;
        off += (n + 3) / 4 * 4;                // keep every tensor 16-byte aligned
        return p;
    }
};

inline size_t walk_packed(const balf_detector_arch& a, const float* base, DetW* out) {
    Cursor c{base, 0};
    DetW w;
    for (int l = 0; l < 4; ++l) {
        const size_t ci = a.dims[l], ch = a.dims[l + 1], red = ch / a.reduction;
        DownW& d = w.down[l];
        d.conv0_w = c.take(ci * ch); d.conv0_b = c.take(ch);
        d.pn_w = c.take(ch); d.pn_b = c.take(ch);
        d.pd1_w = c.take(ch * 2 * ch); d.pd1_b = c.take(2 * ch);
        for (int b = 0; b < 2; ++b) {
            DownW::Branch& r = d.br[b];
            r.n_w = c.take(ch); r.n_b = c.take(ch);
            r.d1_w = c.take(ch * 2 * ch); r.d1_b = c.take(2 * ch);
            r.gn_w = c.take(ch); r.gn_b = c.take(ch);
            r.gd_w = c.take(64 * 64); r.gd_b = c.take(64);
            r.d2_w = c.take(ch * ch); r.d2_b = c.take(ch);
        }
        d.pd2_w = c.take(2 * ch * ch); d.pd2_b = c.take(ch);
        d.rn_w = c.take(ch); d.rn_b = c.take(ch);
        d.rc1_w = c.take(ch * ch); d.rc1_b = c.take(ch);
        d.rc2_w = c.take(ch * ch); d.rc2_b = c.take(ch);
        d.ex0_w = c.take(ch * red); d.ex0_b = c.take(red);
        d.ex2_w = c.take(red * ch); d.ex2_b = c.take(ch);
        d.c2_w = c.take(ch * ch); d.c2_b = c.take(ch);
    }
    const size_t cl = a.dims[4];
    w.head.w = c.take(cl * kHeadPad); w.head.b = c.take(kHeadPad);
    w.head.alpha = c.take(kHeadPad); w.head.beta = c.take(kHeadPad);
    if (out) *out = w;
    return c.off;
}

// tensor-core path, detector_tc.cu: px = 0 single-rounded fp16 / tf32 operands (precision 1), px = 1 split precision (precision 2)
size_t tc_blob_floats(const balf_detector_arch& a);
int tc_pack_weights(const balf_detector_arch& a, const DetW& w, float* blob, cudaStream_t st);
int tc_run_level_dispatch(int level, const float* xin, const DownW& w, const balf_detector_arch& a, const float* blob,
                          int Bc, int h, int wd, float* u, float* v, float* r, float* q, float* partial, cudaStream_t st, int px, int r16);
int tc_run_head(const float* r, const float* q, const float* scale, const balf_detector_arch& a,
                const float* blob, int Bc, int hc, int wc, float* logits, float* prob, cudaStream_t st, int px, int r16);

}  // namespace balf
