// Sampled epipolar cross-attention, fused: for every query ray, gather the S bilinear feature
// samples on its epipolar segment in each other view straight from the (L2-resident) feature
// map, add the depth positional encoding analytically, soft-max the scores and form the
// attention-weighted sums -- without ever materialising the sampled features
// ([b,v,ov,r,s,128] = 0.94 GB at configs[2]) or K/V ([b*v*r, 32, 1024] = 7.5 GB per layer).
//
// Maths (SURVEY.md Appendix B step 7, /root/reference/src/model/transformer/attention.py:54-70,
// epipolar_transformer.py:115-137), restructured with the same result up to fp32 rounding:
//   kv_s   = f_s + W_d PE(rd_s) + b_d (+ emb_ov),        f_s = bilinear(feat_o, xy_s) * valid
//   score  = q_h . (W_k,h kv_s) * scale = qt_h . f_s + pq_h . PE(rd_s) + bias_h,ov + const
//            with qt_h = scale * W_k,h^T q_h (folded by a GEMM outside), pq_h = W_d^T qt_h,
//            bias = qt_h . emb, and const (the b_d term) dropping out of the soft-max;
//   out_h  = W_v,h sum_s a_s kv_s = W_v,h ( z_h + W_d e_h + b_d + sum_ov mass_h,ov emb_ov )
//            with z_h = sum a_s f_s, e_h = sum a_s PE(rd_s), mass_h,ov = sum_{s in ov} a_s.
// The kernel maps (qt, pq, bias) -> (z, e, mass, lse); the small dense projections around it
// stay GEMMs.  One warp per query; lane l owns channels 4l..4l+3 for the gather and sample l
// for the soft-max / PE.  C = 128, S <= 32.
#include <cstdlib>

#include "ps_common.cuh"

namespace ps {

constexpr int kEpiC = 128;
constexpr int kEpiWarps = 4;
constexpr int kMaxPE = 32;

struct EpiParams {
    int B, V, OV, h, w, S, npe;        // npe = 2 * num_octaves
    const float *feat;                 // [B, V, h, w, C] channels-last
    const float *seg;                  // [B, V, OV, R, 4]
    const uint8_t *valid;              // [B, V, OV, R]
    const float *rd;                   // [B, V, OV, R, S]
    const float *qt;                   // [N, H, C]
    const float *pq;                   // [N, H, npe]
    const float *bias;                 // [N, H, OV] or NULL
};

__device__ __forceinline__ float4 ldg4(const float *p) { return __ldg(reinterpret_cast<const float4 *>(p)); }

// Bilinear tap set of grid_sample(align_corners=False, padding_mode="zeros") at normalised (x, y).
struct Taps {
    int off[4];      // element offset of the tap's channel vector inside one view's map, -1 = outside
    float w[4];
};

__device__ __forceinline__ Taps make_taps(float x, float y, int h, int w) {
    const float ix = x * (float)w - 0.5f, iy = y * (float)h - 0.5f;
    const float fx0 = floorf(ix), fy0 = floorf(iy);
    const float ax = ix - fx0, ay = iy - fy0;
    // clamp before the int cast so wild coordinates cannot overflow; they are outside anyway
    const int x0 = (int)fminf(fmaxf(fx0, -2.0f), (float)w + 1.0f);
    const int y0 = (int)fminf(fmaxf(fy0, -2.0f), (float)h + 1.0f);
    Taps t;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int xi = x0 + (k & 1), yi = y0 + (k >> 1);
        const bool in = xi >= 0 && xi < w && yi >= 0 && yi < h;
        t.off[k] = in ? (yi * w + xi) * kEpiC : -1;
        t.w[k] = ((k & 1) ? ax : 1.0f - ax) * ((k >> 1) ? ay : 1.0f - ay);
    }
    return t;
}

// Sum over the 32 lanes of 32 per-lane values v[0..31]; lane l receives sum_lanes v[l].
__device__ __forceinline__ float transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
    for (int half = 16; half >= 1; half >>= 1) {
        const bool up = (lane & half) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float keep = up ? v[i + half] : v[i];
            const float send = up ? v[i] : v[i + half];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
        }
    }
    return v[0];
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_add(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// PE(rd)[2k] = sin(f_k rd), [2k+1] = sin(f_k rd + pi/2), layout "(d f p)"
// (positional_encoding.py:14-33).  The reference's frequency buffer is float32(2 pi) * 2^k, i.e.
// 2 pi (1 + delta) 2^k with delta = 2.78e-8 -- a phase shift of up to 9e-5 rad at k = 9 that is
// part of its semantics (the buffer is non-persistent, so every checkpoint gets it), so it is
// reproduced: phase/pi = u (1 + delta), u = rd 2^(k+1) formed exactly, reduced exactly mod 2, and
// evaluated with sincospif.  (The reference's own fp32 `sin(rd * f_k + phi)` rounds the product,
// up to 2e-4 rad at k = 9; this evaluation is closer to its float64 result.)
__device__ __forceinline__ void positional_encoding(float rd, int npe, float (&pe)[kMaxPE]) {
    constexpr float kTwoPiF32Excess = 2.7827534e-8f;   // float32(2 pi) / (2 pi) - 1
    float scale = 2.0f;
#pragma unroll
    for (int k = 0; k < kMaxPE / 2; ++k) {
        if (2 * k < npe) {
            float s, c;
            const float u = rd * scale;
            const float ur = u - 2.0f * floorf(0.5f * u);
            sincospif(ur + u * kTwoPiF32Excess, &s, &c);
            pe[2 * k] = s;
            pe[2 * k + 1] = c;
            scale *= 2.0f;
        }
    }
}

// Sum over the 32 lanes of SUB per-lane values v[0..SUB-1] (SUB = 4 or 8); every lane receives the total of
// v[lane & (SUB - 1)].  Halving butterflies on the low lane bits, plain butterflies on the rest.
template <int SUB>
__device__ __forceinline__ float transpose_reduce_sub(float (&v)[SUB], int lane) {
#pragma unroll
    for (int half = SUB / 2; half >= 1; half >>= 1) {
        const bool up = (lane & half) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
            const float keep = up ? v[i + half] : v[i];
            const float send = up ? v[i] : v[i + half];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
        }
    }
    float r = v[0];
#pragma unroll
    for (int o = SUB; o < 32; o <<= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
    return r;
}

// max / sum over the SUB distinct values held by an aligned group of SUB lanes (replicated across groups)
template <int SUB>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
    for (int o = SUB / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
template <int SUB>
__device__ __forceinline__ float group_add(float v) {
#pragma unroll
    for (int o = SUB / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Round 2: the S samples of a segment are processed in SUB-CHUNKS of SUB samples (8 forward, 4 backward) instead
// of all 32 at once.  Holding f[32][4] pinned both kernels at 255 registers = 8 warps per SM (12 % occupancy),
// which is what bounded them: they are latency-bound on the bilinear gathers (ncu r01: 22-27 % issue-active).
// With SUB samples in registers the forward needs <= 128 registers (16 warps / SM) and the backward <= 128 too;
// the soft-max is already streaming (online max / sum), so sub-chunks only add rescales.  The positional-
// encoding half of every score (and of d score) is evaluated once per other view with lane = sample, as before,
// and parked in shared memory for the sub-chunks to pick up.
struct __align__(16) EpiWarpSmem {
    float p[8][4];           // soft-max numerators (forward) / probabilities (backward) of the sub-chunk
    float dsub[8][4];        // backward: d score of the sub-chunk
    float scpe[32][4];       // PE half of the scores (+ bias), [sample][head]; -inf beyond S
    float dape[32][4];       // backward: PE half of d a (+ dmass)
    float ds_all[32][4];     // backward: d score of all samples of this other view (for dpq)
    float pe[32][kMaxPE + 1];
    float pq[4][kMaxPE];
    float aux[4][kMaxPE];    // backward: d_e
};

template <int HEADS, int SUB>
__global__ void __launch_bounds__(kEpiWarps * 32, 4)
k_epi_attn_fwd(EpiParams P, int n_queries, float *__restrict__ z_out, float *__restrict__ e_out,
               float *__restrict__ mass_out, float *__restrict__ lse_out) {
    __shared__ EpiWarpSmem sm_all[kEpiWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    EpiWarpSmem &sm = sm_all[warp];
    const int n = blockIdx.x * kEpiWarps + warp;
    if (n >= n_queries) return;
    const int R = P.h * P.w;
    const int r = n % R, bv = n / R;
    const int v = bv % P.V, b = bv / P.V;

    float qt[HEADS][4];
#pragma unroll
    for (int hd = 0; hd < HEADS; ++hd) {
        const float4 q = ldg4(P.qt + ((size_t)n * HEADS + hd) * kEpiC + 4 * lane);
        qt[hd][0] = q.x; qt[hd][1] = q.y; qt[hd][2] = q.z; qt[hd][3] = q.w;
    }
    for (int i = lane; i < HEADS * P.npe; i += 32)
        sm.pq[i / P.npe][i % P.npe] = P.pq[(size_t)n * HEADS * P.npe + i];
    __syncwarp();

    float m_run[HEADS], l_run[HEADS], z[HEADS][4], e_acc[3];   // e_acc: outputs lane, lane+32, lane+64
    float mass_acc[HEADS];                                     // lane ov (< OV) accumulates the mass of view ov
#pragma unroll
    for (int hd = 0; hd < HEADS; ++hd) {
        m_run[hd] = -INFINITY; l_run[hd] = 0.0f; mass_acc[hd] = 0.0f;
        z[hd][0] = z[hd][1] = z[hd][2] = z[hd][3] = 0.0f;
    }
    e_acc[0] = e_acc[1] = e_acc[2] = 0.0f;
    const int nsub = (P.S + SUB - 1) / SUB;
    const int total_e = HEADS * P.npe;

    for (int ov = 0; ov < P.OV; ++ov) {
        const int o_view = ov < v ? ov : ov + 1;
        const size_t ray = ((size_t)(bv * P.OV + ov)) * R + r;
        const float4 sg = ldg4(P.seg + 4 * ray);
        const bool ok = P.valid[ray] != 0;
        const float *fmap = P.feat + (size_t)(b * P.V + o_view) * R * kEpiC + 4 * lane;

        // ---- PE half of the scores and the bilinear taps, lane = sample
        Taps my_taps;
        int my_cell = -0x7ffffffe;
        {
            float pe[kMaxPE];
            const bool has_sample = lane < P.S;
            if (has_sample && ok) {
                const float u = ((float)lane + 0.5f) / (float)P.S;
                const float sx = sg.x + u * (sg.z - sg.x), sy = sg.y + u * (sg.w - sg.y);
                my_taps = make_taps(sx, sy, P.h, P.w);
                const float ix = sx * (float)P.w - 0.5f, iy = sy * (float)P.h - 0.5f;
                const int bx = (int)fminf(fmaxf(floorf(ix), -2.0f), (float)P.w + 1.0f);
                const int by = (int)fminf(fmaxf(floorf(iy), -2.0f), (float)P.h + 1.0f);
                my_cell = by * (P.w + 4) + bx;            // the bilinear cell (backward merges samples that share it)
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) { my_taps.off[k] = -1; my_taps.w[k] = 0.0f; }
            }
            positional_encoding(has_sample ? P.rd[ray * P.S + lane] : 0.0f, P.npe, pe);
#pragma unroll
            for (int j = 0; j < kMaxPE; ++j)
                if (j < P.npe) sm.pe[lane][j] = has_sample ? pe[j] : 0.0f;
#pragma unroll
            for (int hd = 0; hd < HEADS; ++hd) {
                float sc = 0.0f;
#pragma unroll
                for (int j = 0; j < kMaxPE; ++j)
                    if (j < P.npe) sc += sm.pq[hd][j] * pe[j];
                if (P.bias) sc += P.bias[((size_t)n * HEADS + hd) * P.OV + ov];
                sm.scpe[lane][hd] = has_sample ? sc : -INFINITY;
            }
        }
        __syncwarp();

        for (int sub = 0; sub < nsub; ++sub) {
            // ---- gather SUB samples (channels 4*lane..4*lane+3 of each)
            float f[SUB][4];
#pragma unroll
            for (int i = 0; i < SUB; ++i) {
                const int s = sub * SUB + i;
                f[i][0] = f[i][1] = f[i][2] = f[i][3] = 0.0f;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    // the taps of sample s were formed once, by lane s (every lane needs the same four)
                    const int off = __shfl_sync(0xffffffffu, my_taps.off[k], s);
                    const float wk = __shfl_sync(0xffffffffu, my_taps.w[k], s);
                    if (off >= 0) {
                        const float4 a = ldg4(fmap + off);
                        f[i][0] += wk * a.x; f[i][1] += wk * a.y;
                        f[i][2] += wk * a.z; f[i][3] += wk * a.w;
                    }
                }
            }
            // ---- scores: every lane ends up with the score of sample sub*SUB + (lane & (SUB-1))
            const int s_mine = sub * SUB + (lane & (SUB - 1));
            float scale_old[HEADS];
#pragma unroll
            for (int hd = 0; hd < HEADS; ++hd) {
                float part[SUB];
#pragma unroll
                for (int i = 0; i < SUB; ++i)
                    part[i] = qt[hd][0] * f[i][0] + qt[hd][1] * f[i][1] + qt[hd][2] * f[i][2] + qt[hd][3] * f[i][3];
                const float sc = transpose_reduce_sub<SUB>(part, lane) + sm.scpe[s_mine][hd];   // -inf beyond S
                const float m_new = fmaxf(m_run[hd], group_max<SUB>(sc));     // >= one finite score per sub-chunk
                scale_old[hd] = __expf(m_run[hd] - m_new);                     // exp(-inf) = 0 on the first one
                const float pnum = __expf(sc - m_new);                         // exp(-inf) = 0 beyond S
                const float psum = group_add<SUB>(pnum);
                l_run[hd] = l_run[hd] * scale_old[hd] + psum;
                m_run[hd] = m_new;
                if (lane < SUB) sm.p[lane][hd] = pnum;
                if (lane <= ov) mass_acc[hd] = mass_acc[hd] * scale_old[hd] + (lane == ov ? psum : 0.0f);
            }
            __syncwarp();
            // ---- weighted sums
#pragma unroll
            for (int hd = 0; hd < HEADS; ++hd) {
                z[hd][0] *= scale_old[hd]; z[hd][1] *= scale_old[hd];
                z[hd][2] *= scale_old[hd]; z[hd][3] *= scale_old[hd];
            }
#pragma unroll
            for (int i = 0; i < SUB; ++i) {
                float pw[4];
                *reinterpret_cast<float4 *>(pw) = *reinterpret_cast<const float4 *>(sm.p[i]);
#pragma unroll
                for (int hd = 0; hd < HEADS; ++hd) {
                    z[hd][0] += pw[hd] * f[i][0]; z[hd][1] += pw[hd] * f[i][1];
                    z[hd][2] += pw[hd] * f[i][2]; z[hd][3] += pw[hd] * f[i][3];
                }
            }
            // e[h][j] = sum_s p[s][h] * pe[s][j]; output index o = lane + 32*i -> (h, j) = (o / npe, o % npe)
#pragma unroll
            for (int i3 = 0; i3 < 3; ++i3) {
                const int o = lane + 32 * i3;
                if (o < total_e) {
                    const int hd = o / P.npe, j = o % P.npe;
                    float acc = 0.0f;
#pragma unroll
                    for (int i = 0; i < SUB; ++i) acc += sm.p[i][hd] * sm.pe[sub * SUB + i][j];
                    float so = 0.0f;
#pragma unroll
                    for (int q = 0; q < HEADS; ++q) so = (q == hd) ? scale_old[q] : so;
                    e_acc[i3] = e_acc[i3] * so + acc;
                }
            }
            __syncwarp();
        }
    }

    // ---- normalise and store
#pragma unroll
    for (int hd = 0; hd < HEADS; ++hd) {
        const float inv = 1.0f / l_run[hd];
        float4 o = make_float4(z[hd][0] * inv, z[hd][1] * inv, z[hd][2] * inv, z[hd][3] * inv);
        *reinterpret_cast<float4 *>(z_out + ((size_t)n * HEADS + hd) * kEpiC + 4 * lane) = o;
        if (lane == 0) lse_out[(size_t)n * HEADS + hd] = m_run[hd] + __logf(l_run[hd]);
        if (mass_out && lane < P.OV) mass_out[((size_t)n * HEADS + hd) * P.OV + lane] = mass_acc[hd] * inv;
    }
#pragma unroll
    for (int i3 = 0; i3 < 3; ++i3) {
        const int o = lane + 32 * i3;
        if (o < total_e) {
            const int hd = o / P.npe;
            float lr = 1.0f;
#pragma unroll
            for (int q = 0; q < HEADS; ++q) lr = (q == hd) ? l_run[q] : lr;
            e_out[(size_t)n * total_e + o] = e_acc[i3] / lr;
        }
    }
}

// Backward of k_epi_attn_fwd.  Inputs: the forward inputs, lse, the output cotangents (dz, de,
// dmass) and D_h = dz_h.z_h + de_h.e_h + dmass_h.mass_h (flash-attention's row term, formed
// outside by one elementwise pass).  Outputs: dqt, dpq, dbias, and d(feature map) accumulated with
// 16-byte vector atomics (the map gradient is L2-resident; consecutive samples that fall in the
// same bilinear cell are merged in registers first, which removes most of the atomics on short
// epipolar segments).  With lse known every sample is independent, so sub-chunks need no rescaling here.
template <int HEADS, int SUB>
__global__ void __launch_bounds__(kEpiWarps * 32, 4)
k_epi_attn_bwd(EpiParams P, int n_queries, const float *__restrict__ lse, const float *__restrict__ dz,
               const float *__restrict__ de, const float *__restrict__ dmass, const float *__restrict__ Drow,
               float *__restrict__ dqt_out, float *__restrict__ dpq_out, float *__restrict__ dbias_out,
               float *__restrict__ dfeat) {
    __shared__ EpiWarpSmem sm_all[kEpiWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    EpiWarpSmem &sm = sm_all[warp];
    const int n = blockIdx.x * kEpiWarps + warp;
    if (n >= n_queries) return;
    const int R = P.h * P.w;
    const int r = n % R, bv = n / R;
    const int v = bv % P.V, b = bv / P.V;

    float qt[HEADS][4], gz[HEADS][4], dq[HEADS][4], lse_h[HEADS], D_h[HEADS];
#pragma unroll
    for (int hd = 0; hd < HEADS; ++hd) {
        const size_t o = ((size_t)n * HEADS + hd) * kEpiC + 4 * lane;
        const float4 q = ldg4(P.qt + o), g = ldg4(dz + o);
        qt[hd][0] = q.x; qt[hd][1] = q.y; qt[hd][2] = q.z; qt[hd][3] = q.w;
        gz[hd][0] = g.x; gz[hd][1] = g.y; gz[hd][2] = g.z; gz[hd][3] = g.w;
        dq[hd][0] = dq[hd][1] = dq[hd][2] = dq[hd][3] = 0.0f;
        lse_h[hd] = lse[(size_t)n * HEADS + hd];
        D_h[hd] = Drow[(size_t)n * HEADS + hd];
    }
    for (int i = lane; i < HEADS * P.npe; i += 32) {
        sm.pq[i / P.npe][i % P.npe] = P.pq[(size_t)n * HEADS * P.npe + i];
        sm.aux[i / P.npe][i % P.npe] = de[(size_t)n * HEADS * P.npe + i];
    }
    __syncwarp();
    float dpq_acc[3] = {0.0f, 0.0f, 0.0f};
    const int nsub = (P.S + SUB - 1) / SUB;

    for (int ov = 0; ov < P.OV; ++ov) {
        const int o_view = ov < v ? ov : ov + 1;
        const size_t ray = ((size_t)(bv * P.OV + ov)) * R + r;
        const float4 sg = ldg4(P.seg + 4 * ray);
        const bool ok = P.valid[ray] != 0;
        const size_t map_base = (size_t)(b * P.V + o_view) * R * kEpiC + 4 * lane;
        const float *fmap = P.feat + map_base;

        // ---- PE halves of the score and of d a, and the bilinear taps, lane = sample
        Taps my_taps;
        int my_cell = -0x7ffffffe;
        {
            float pe[kMaxPE];
            const bool has_sample = lane < P.S;
            if (has_sample && ok) {
                const float u = ((float)lane + 0.5f) / (float)P.S;
                const float sx = sg.x + u * (sg.z - sg.x), sy = sg.y + u * (sg.w - sg.y);
                my_taps = make_taps(sx, sy, P.h, P.w);
                const float ix = sx * (float)P.w - 0.5f, iy = sy * (float)P.h - 0.5f;
                const int bx = (int)fminf(fmaxf(floorf(ix), -2.0f), (float)P.w + 1.0f);
                const int by = (int)fminf(fmaxf(floorf(iy), -2.0f), (float)P.h + 1.0f);
                my_cell = by * (P.w + 4) + bx;            // the bilinear cell (backward merges samples that share it)
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) { my_taps.off[k] = -1; my_taps.w[k] = 0.0f; }
            }
            positional_encoding(has_sample ? P.rd[ray * P.S + lane] : 0.0f, P.npe, pe);
#pragma unroll
            for (int j = 0; j < kMaxPE; ++j)
                if (j < P.npe) sm.pe[lane][j] = has_sample ? pe[j] : 0.0f;
#pragma unroll
            for (int hd = 0; hd < HEADS; ++hd) {
                float sc = 0.0f, da = 0.0f;
#pragma unroll
                for (int j = 0; j < kMaxPE; ++j)
                    if (j < P.npe) { sc += sm.pq[hd][j] * pe[j]; da += sm.aux[hd][j] * pe[j]; }
                if (P.bias) sc += P.bias[((size_t)n * HEADS + hd) * P.OV + ov];
                if (dmass) da += dmass[((size_t)n * HEADS + hd) * P.OV + ov];
                sm.scpe[lane][hd] = has_sample ? sc : -INFINITY;
                sm.dape[lane][hd] = da;
                sm.ds_all[lane][hd] = 0.0f;
            }
        }
        __syncwarp();

        float dbias_acc[HEADS];
#pragma unroll
        for (int hd = 0; hd < HEADS; ++hd) dbias_acc[hd] = 0.0f;
        int cur_base = -0x7fffffff;
        float tap_acc[4][4];
        int tap_off[4] = {-1, -1, -1, -1};
#pragma unroll
        for (int k = 0; k < 4; ++k) tap_acc[k][0] = tap_acc[k][1] = tap_acc[k][2] = tap_acc[k][3] = 0.0f;
        auto flush = [&]() {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (tap_off[k] >= 0)
                    atomicAdd(reinterpret_cast<float4 *>(dfeat + map_base + tap_off[k]),
                              make_float4(tap_acc[k][0], tap_acc[k][1], tap_acc[k][2], tap_acc[k][3]));
                tap_acc[k][0] = tap_acc[k][1] = tap_acc[k][2] = tap_acc[k][3] = 0.0f;
            }
        };

        for (int sub = 0; sub < nsub; ++sub) {
            float f[SUB][4];
#pragma unroll
            for (int i = 0; i < SUB; ++i) {
                const int s = sub * SUB + i;
                f[i][0] = f[i][1] = f[i][2] = f[i][3] = 0.0f;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    // the taps of sample s were formed once, by lane s (every lane needs the same four)
                    const int off = __shfl_sync(0xffffffffu, my_taps.off[k], s);
                    const float wk = __shfl_sync(0xffffffffu, my_taps.w[k], s);
                    if (off >= 0) {
                        const float4 a = ldg4(fmap + off);
                        f[i][0] += wk * a.x; f[i][1] += wk * a.y;
                        f[i][2] += wk * a.z; f[i][3] += wk * a.w;
                    }
                }
            }
            const int s_mine = sub * SUB + (lane & (SUB - 1));
#pragma unroll
            for (int hd = 0; hd < HEADS; ++hd) {
                float part[SUB];
#pragma unroll
                for (int i = 0; i < SUB; ++i)
                    part[i] = qt[hd][0] * f[i][0] + qt[hd][1] * f[i][1] + qt[hd][2] * f[i][2] + qt[hd][3] * f[i][3];
                const float sc = transpose_reduce_sub<SUB>(part, lane) + sm.scpe[s_mine][hd];
#pragma unroll
                for (int i = 0; i < SUB; ++i)
                    part[i] = gz[hd][0] * f[i][0] + gz[hd][1] * f[i][1] + gz[hd][2] * f[i][2] + gz[hd][3] * f[i][3];
                const float da = transpose_reduce_sub<SUB>(part, lane) + sm.dape[s_mine][hd];
                const float a = __expf(sc - lse_h[hd]);                 // 0 beyond S (score -inf)
                const float dsc = a * (da - D_h[hd]);
                if (lane < SUB) {
                    sm.p[lane][hd] = a;
                    sm.dsub[lane][hd] = dsc;
                    sm.ds_all[s_mine][hd] = dsc;
                }
                dbias_acc[hd] += group_add<SUB>(dsc);
            }
            __syncwarp();

            // dqt += sum_s ds[s] f[s];  d f[s] = sum_h a[s,h] dz_h + ds[s,h] qt_h  -> scatter to the taps
#pragma unroll
            for (int i = 0; i < SUB; ++i) {
                const int s = sub * SUB + i;
                float aw[4], dw[4];
                *reinterpret_cast<float4 *>(aw) = *reinterpret_cast<const float4 *>(sm.p[i]);
                *reinterpret_cast<float4 *>(dw) = *reinterpret_cast<const float4 *>(sm.dsub[i]);
                float df[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
                for (int hd = 0; hd < HEADS; ++hd) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        dq[hd][c] += dw[hd] * f[i][c];
                        df[c] += aw[hd] * gz[hd][c] + dw[hd] * qt[hd][c];
                    }
                }
                if (s < P.S && ok) {
                    Taps t;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        t.off[k] = __shfl_sync(0xffffffffu, my_taps.off[k], s);
                        t.w[k] = __shfl_sync(0xffffffffu, my_taps.w[k], s);
                    }
                    // identify the bilinear cell by its top-left tap position (may be outside)
                    const int base = __shfl_sync(0xffffffffu, my_cell, s);
                    if (base != cur_base) {
                        flush();
                        cur_base = base;
#pragma unroll
                        for (int k = 0; k < 4; ++k) tap_off[k] = t.off[k];
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        tap_acc[k][0] += t.w[k] * df[0]; tap_acc[k][1] += t.w[k] * df[1];
                        tap_acc[k][2] += t.w[k] * df[2]; tap_acc[k][3] += t.w[k] * df[3];
                    }
                }
            }
            __syncwarp();
        }
        flush();
        if (dbias_out && lane == 0) {
#pragma unroll
            for (int hd = 0; hd < HEADS; ++hd) dbias_out[((size_t)n * HEADS + hd) * P.OV + ov] = dbias_acc[hd];
        }
        // dpq[h][j] += sum_s ds[s][h] pe[s][j]
        {
            const int total = HEADS * P.npe;
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const int o = lane + 32 * i;
                if (o < total) {
                    const int hd = o / P.npe, j = o % P.npe;
                    float acc = 0.0f;
                    for (int s = 0; s < 32; ++s) acc += sm.ds_all[s][hd] * sm.pe[s][j];
                    dpq_acc[i] += acc;
                }
            }
        }
        __syncwarp();
    }
#pragma unroll
    for (int hd = 0; hd < HEADS; ++hd)
        *reinterpret_cast<float4 *>(dqt_out + ((size_t)n * HEADS + hd) * kEpiC + 4 * lane) =
            make_float4(dq[hd][0], dq[hd][1], dq[hd][2], dq[hd][3]);
    {
        const int total = HEADS * P.npe;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const int o = lane + 32 * i;
            if (o < total) dpq_out[(size_t)n * total + o] = dpq_acc[i];
        }
    }
}

constexpr int kEpiSubFwd = 8, kEpiSubBwd = 4;

template <int HEADS>
static int launch_epi(bool backward, const EpiParams &P, int n, float *z, float *e, float *mass, float *lse_out,
                      const float *lse, const float *dz, const float *de, const float *dmass, const float *Drow,
                      float *dqt, float *dpq, float *dbias, float *dfeat, cudaStream_t st) {
    const int blocks = (n + kEpiWarps - 1) / kEpiWarps;
    if (!backward) {
        static int sub_fwd = 0;                       // PIXELSPLAT_B200_EPI_SUB_FWD = 4 | 8 (A/B runs)
        if (sub_fwd == 0) {
            const char *e = getenv("PIXELSPLAT_B200_EPI_SUB_FWD");
            sub_fwd = (e && e[0] == '4') ? 4 : kEpiSubFwd;
        }
        if (sub_fwd == 4) k_epi_attn_fwd<HEADS, 4><<<blocks, kEpiWarps * 32, 0, st>>>(P, n, z, e, mass, lse_out);
        else k_epi_attn_fwd<HEADS, kEpiSubFwd><<<blocks, kEpiWarps * 32, 0, st>>>(P, n, z, e, mass, lse_out);
        PS_LAUNCH_CHECK("k_epi_attn_fwd");
    } else {
        k_epi_attn_bwd<HEADS, kEpiSubBwd><<<blocks, kEpiWarps * 32, 0, st>>>(P, n, lse, dz, de, dmass, Drow, dqt, dpq, dbias, dfeat);
        PS_LAUNCH_CHECK("k_epi_attn_bwd");
    }
    return PS_OK;
}

static int epi_check(const ps_epipolar_desc *d) {
    if (!d) { set_error("desc is NULL"); return PS_ERR_INVALID_ARGUMENT; }
    if (d->batch < 1 || d->views < 2 || d->grid_h < 1 || d->grid_w < 1) {
        set_error("ps_epipolar: need batch >= 1, views >= 2, positive grid"); return PS_ERR_INVALID_ARGUMENT;
    }
    if (d->channels != kEpiC) { set_error("ps_epipolar: channels must be %d, got %d", kEpiC, d->channels); return PS_ERR_UNSUPPORTED; }
    if (d->heads < 1 || d->heads > 4) { set_error("ps_epipolar: heads must be in [1, 4], got %d", d->heads); return PS_ERR_UNSUPPORTED; }
    if (d->samples < 1 || d->samples > 32) { set_error("ps_epipolar: samples must be in [1, 32], got %d", d->samples); return PS_ERR_UNSUPPORTED; }
    if (d->pe_dim < 0 || d->pe_dim > kMaxPE || (d->pe_dim & 1) || d->heads * d->pe_dim > 96) {
        set_error("ps_epipolar: pe_dim must be even, <= %d and heads*pe_dim <= 96 (got %d)", kMaxPE, d->pe_dim);
        return PS_ERR_UNSUPPORTED;
    }
    if (d->views - 1 > 32) { set_error("ps_epipolar: at most 33 views"); return PS_ERR_UNSUPPORTED; }
    return PS_OK;
}

static EpiParams epi_params(const ps_epipolar_desc *d, const ps_epipolar_inputs *in) {
    EpiParams P;
    P.B = d->batch; P.V = d->views; P.OV = d->views - 1; P.h = d->grid_h; P.w = d->grid_w; P.S = d->samples;
    P.npe = d->pe_dim; P.feat = in->features; P.seg = in->segments; P.valid = in->valid;
    P.rd = in->rel_disparity; P.qt = in->q_feat; P.pq = in->q_pe; P.bias = in->bias;
    return P;
}

}  // namespace ps

using namespace ps;

extern "C" PS_API int ps_epipolar_attention_forward(const ps_epipolar_desc *d, const ps_epipolar_inputs *in,
                                                    float *z, float *e, float *mass, float *lse, void *stream) {
    int rc = epi_check(d);
    if (rc) return rc;
    if (!in || !in->features || !in->segments || !in->valid || !in->rel_disparity || !in->q_feat ||
        (d->pe_dim > 0 && (!in->q_pe || !e)) || !z || !lse) {
        set_error("ps_epipolar_attention_forward: a required pointer is NULL");
        return PS_ERR_INVALID_ARGUMENT;
    }
    const EpiParams P = epi_params(d, in);
    const int n = d->batch * d->views * d->grid_h * d->grid_w;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (d->heads) {
        case 1: return launch_epi<1>(false, P, n, z, e, mass, lse, 0, 0, 0, 0, 0, 0, 0, 0, 0, st);
        case 2: return launch_epi<2>(false, P, n, z, e, mass, lse, 0, 0, 0, 0, 0, 0, 0, 0, 0, st);
        case 3: return launch_epi<3>(false, P, n, z, e, mass, lse, 0, 0, 0, 0, 0, 0, 0, 0, 0, st);
        default: return launch_epi<4>(false, P, n, z, e, mass, lse, 0, 0, 0, 0, 0, 0, 0, 0, 0, st);
    }
}

extern "C" PS_API int ps_epipolar_attention_backward(const ps_epipolar_desc *d, const ps_epipolar_inputs *in,
                                                     const float *lse, const float *dz, const float *de,
                                                     const float *dmass, const float *d_row, float *dq_feat,
                                                     float *dq_pe, float *dbias, float *dfeatures, void *stream) {
    int rc = epi_check(d);
    if (rc) return rc;
    if (!in || !in->features || !in->segments || !in->valid || !in->rel_disparity || !in->q_feat || !lse ||
        !dz || (d->pe_dim > 0 && (!in->q_pe || !de || !dq_pe)) || !d_row || !dq_feat || !dfeatures) {
        set_error("ps_epipolar_attention_backward: a required pointer is NULL");
        return PS_ERR_INVALID_ARGUMENT;
    }
    const EpiParams P = epi_params(d, in);
    const int n = d->batch * d->views * d->grid_h * d->grid_w;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (d->heads) {
        case 1: return launch_epi<1>(true, P, n, 0, 0, 0, 0, lse, dz, de, dmass, d_row, dq_feat, dq_pe, dbias, dfeatures, st);
        case 2: return launch_epi<2>(true, P, n, 0, 0, 0, 0, lse, dz, de, dmass, d_row, dq_feat, dq_pe, dbias, dfeatures, st);
        case 3: return launch_epi<3>(true, P, n, 0, 0, 0, 0, lse, dz, de, dmass, d_row, dq_feat, dq_pe, dbias, dfeatures, st);
        default: return launch_epi<4>(true, P, n, 0, 0, 0, 0, lse, dz, de, dmass, d_row, dq_feat, dq_pe, dbias, dfeatures, st);
    }
}
