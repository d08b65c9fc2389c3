// Per-row temperature / top-k / top-p sampling + sequence state advance (dots_sample_advance).
//
// Semantics (DESIGN.md section 3, dots_ocr_b200/sampling.py; restated in fp64 by oracle/sampling.py), per row on the bf16 logits l
// in fp32, HF's warper order (transformers generation/logits_process.py: Temperature -> TopK -> TopP):
//   T < 1e-5            greedy: fp32 argmax, lowest index wins ties (the exact loop of argmax_advance_kernel);
//   top-k (k > 0)       keep l >= (k-th largest l); ties at the cut-off are kept;
//   top-p (p < 1)       over the top-k survivors, keep l iff the softmax(l / T) mass of STRICTLY larger logits is < p, so every
//                       token tied with the last kept value is kept too (no sort, no dependence on the batch);
//   draw                Gumbel-max over the kept set: argmax_i l_i / T - log(-log u_i), lowest index wins ties;
//   u_i                 Philox4x32-10, key = the row's 64-bit seed, counter = (i >> 2, step[b], 0, 0), word i & 3,
//                       u = ((x >> 8) + 0.5) * 2^-24 in (0, 1).
// A row's token depends on its logits row, parameters, seed and step only.
//
// One CTA per row.  bf16 logits give a 16-bit monotone sort key, so the exact cut-off takes two 256-bin radix passes (high
// byte, then low byte inside the selected bucket) with a count and a fixed-point exp((l - max) / T) mass per bin: integer
// sums are associative, so the cut-off is the same run to run.  Rows with k = 0, p = 1 skip to the Gumbel pass; greedy rows
// run the argmax pass only.  At decode batch sizes the logits are L2-resident, so the passes re-read them from L2.
#include "common.h"
#include "ptx.cuh"
#include "../../include/dots_ocr_b200.h"

namespace dots {

namespace {

constexpr int kThreads = 1024;
constexpr int kSub = 8;                              // sub-histograms (by warp & 7): spreads shared-atomic contention
constexpr float kGreedyT = 1e-5f;                    // vLLM's threshold: below it a row decodes greedily
constexpr float kMassScale = 1099511627776.0f;       // 2^40: fixed-point scale of the per-bin mass (152k tokens < 2^58)
constexpr float kMassFloor = -30.0f;                 // (l - max) / T below this: exp() * 2^40 < 0.5 rounds to a zero mass
constexpr float kGumbelMax = 17.5f;                  // > -log(-log u) for every u the generator yields (max 17.33)

struct StopIds { long long id[DOTS_MAX_STOP_IDS]; int n; };

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
    f[0] = bf16_lo(u.x); f[1] = bf16_hi(u.x); f[2] = bf16_lo(u.y); f[3] = bf16_hi(u.y);
    f[4] = bf16_lo(u.z); f[5] = bf16_hi(u.z); f[6] = bf16_lo(u.w); f[7] = bf16_hi(u.w);
}

// monotone 16-bit key of a bf16 value (-0 folded onto +0 so that equal values have equal keys)
__device__ __forceinline__ unsigned sort_key(float f) {
    unsigned b = __float_as_uint(f) >> 16;
    if (b == 0x8000u) b = 0;
    return (b & 0x8000u) ? (~b & 0xFFFFu) : (b | 0x8000u);
}

// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
        const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c;
}

// -log(u) for u = ((x >> 8) + 0.5) * 2^-24, with the argument of each log exact in fp32: the upper half goes through
// log1p(-(1 - u)) so that u close to 1 keeps its precision.
__device__ __forceinline__ float neg_log_u(uint32_t x) {
    const uint32_t a = x >> 8;
    if (a < (1u << 23)) return -logf(((float)a + 0.5f) * 5.9604644775390625e-8f);
    const float w = ((float)((1u << 24) - 1u - a) + 0.5f) * 5.9604644775390625e-8f;          // 1 - u
    return -log1pf(-w);
}

__device__ __forceinline__ void better(float& best, int& bidx, float ob, int oi) {
    if (ob > best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
}

// block-wide (value, lowest index) argmax; every thread gets the result
__device__ __forceinline__ void block_argmax(float& best, int& bidx, float* sb, int* si) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        better(best, bidx, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, bidx, o));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) { sb[warp] = best; si[warp] = bidx; }
    __syncthreads();
    best = (lane < (int)(blockDim.x >> 5)) ? sb[lane] : -INFINITY;
    bidx = (lane < (int)(blockDim.x >> 5)) ? si[lane] : 0x7fffffff;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        better(best, bidx, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, bidx, o));
}

struct Smem {
    unsigned sub_c[kSub][256];
    unsigned long long sub_m[kSub][256];
    unsigned hc[256], lc[256];                     // reduced high-byte / low-byte bins: counts
    unsigned long long hm[256], lm[256];           //                                   masses
    unsigned hc_above[256], lc_above[256];         // exclusive sums from the top bin down
    unsigned long long hm_above[256], lm_above[256];
    unsigned long long wsum_c[8], wsum_m[8];
    float sb[32];
    int si[32];
    int pick;
};

// One histogram pass over the row: bins by key >> 8 (hi_sel < 0) or by key & 255 among keys with key >> 8 == hi_sel; values
// below `floor` are left out.  Result reduced into (cnt, mass) and their exclusive sums from the top into (c_above, m_above).
__device__ void histogram(Smem& s, const bf16* row, int V, int hi_sel, float floor, float m, float invT, bool want_mass, unsigned* cnt,
                          unsigned long long* mass, unsigned* c_above, unsigned long long* m_above) {
    for (int i = threadIdx.x; i < kSub * 256; i += blockDim.x) { (&s.sub_c[0][0])[i] = 0; (&s.sub_m[0][0])[i] = 0; }
    __syncthreads();
    unsigned* sc = s.sub_c[(threadIdx.x >> 5) & (kSub - 1)];
    unsigned long long* sm = s.sub_m[(threadIdx.x >> 5) & (kSub - 1)];
    const int nchunks = V >> 3;
    for (int c = threadIdx.x; c < nchunks; c += blockDim.x) {
        float f[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(row) + c), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const unsigned key = sort_key(f[j]);
            if (f[j] < floor || (hi_sel >= 0 && (int)(key >> 8) != hi_sel)) continue;
            const unsigned bin = hi_sel >= 0 ? (key & 255u) : (key >> 8);
            atomicAdd(&sc[bin], 1u);
            if (want_mass) atomicAdd(&sm[bin], (unsigned long long)__float2ull_rn(__expf((f[j] - m) * invT) * kMassScale));
        }
    }
    __syncthreads();
    // threads 0..255 own the bins in DESCENDING order (t -> bin 255 - t) and scan them
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    unsigned long long ic = 0, im = 0, oc = 0, om = 0;
    if (t < 256) {
        const int bin = 255 - t;
#pragma unroll
        for (int k = 0; k < kSub; ++k) { oc += s.sub_c[k][bin]; om += s.sub_m[k][bin]; }
        cnt[bin] = (unsigned)oc; mass[bin] = om;
        ic = oc; im = om;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long xc = __shfl_up_sync(0xffffffffu, ic, o), xm = __shfl_up_sync(0xffffffffu, im, o);
            if (lane >= o) { ic += xc; im += xm; }
        }
        if (lane == 31) { s.wsum_c[warp] = ic; s.wsum_m[warp] = im; }
    }
    __syncthreads();
    if (t < 256) {
        for (int w = 0; w < warp; ++w) { ic += s.wsum_c[w]; im += s.wsum_m[w]; }
        c_above[255 - t] = (unsigned)(ic - oc);
        m_above[255 - t] = im - om;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kThreads) sample_advance_kernel(
        const bf16* __restrict__ logits, long long ldl, int V, long long* __restrict__ next_ids, long long* __restrict__ out_ids,
        long long out_ld, int* __restrict__ step, int* __restrict__ pos, int* __restrict__ ctx_len, int* __restrict__ finished,
        const StopIds stops, long long pad_id, const long long* __restrict__ forced, long long forced_ld,
        const float* __restrict__ temperature, const float* __restrict__ top_p, const int* __restrict__ top_k,
        const unsigned long long* __restrict__ seed) {
    pdl_wait();
    pdl_launch_dependents();
    __shared__ Smem s;
    const int b = blockIdx.x;
    const bf16* row = logits + (long long)b * ldl;
    const int nchunks = V >> 3;
    const float T = temperature[b];
    const int st = step ? step[b] : 0;
    float best = -INFINITY;
    int bidx = 0x7fffffff;
    if (!(T >= kGreedyT)) {
        // greedy: the argmax_advance_kernel loop
        for (int c = threadIdx.x; c < nchunks; c += blockDim.x) {
            float f[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(row) + c), f);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (f[j] > best) { best = f[j]; bidx = c * 8 + j; }
        }
    } else {
        const float invT = 1.0f / T;
        const float p = top_p[b];
        const int k = top_k[b];
        const bool use_k = k > 0 && k < V, use_p = p < 1.0f;
        const uint32_t k0 = (uint32_t)seed[b], k1 = (uint32_t)(seed[b] >> 32);
        // max pass: the row maximum m (top-p masses are exp((l - m) / T)) and its index, which every cut-off keeps
        float m = -INFINITY;
        int amax = 0x7fffffff;
        for (int c = threadIdx.x; c < nchunks; c += blockDim.x) {
            float f[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(row) + c), f);
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (f[j] > m) { m = f[j]; amax = c * 8 + j; }
        }
        block_argmax(m, amax, s.sb, s.si);
        unsigned cut = 0;                                     // kept: sort_key(l) >= cut
        if (use_k || use_p) {
            // top-p alone needs only the tokens with a non-zero fixed-point mass (bin occupancy below them cannot matter)
            const float floor = use_k ? -INFINITY : m + kMassFloor * T;
            histogram(s, row, V, -1, floor, m, invT, use_p, s.hc, s.hm, s.hc_above, s.hm_above);
            int hk = 0, lk = 0;                               // top-k cut-off key (hk << 8 | lk); 0 = none
            unsigned long long Z = s.hm_above[0] + s.hm[0];   // mass of the survivors of top-k
            if (use_k) {
                if (threadIdx.x == 0) s.pick = 0;
                __syncthreads();
                if (threadIdx.x < 256) {
                    const int h = threadIdx.x;
                    if (s.hc_above[h] < (unsigned)k && (unsigned)k <= s.hc_above[h] + s.hc[h]) s.pick = h;
                }
                __syncthreads();
                hk = s.pick;
                histogram(s, row, V, hk, -INFINITY, m, invT, use_p, s.lc, s.lm, s.lc_above, s.lm_above);
                const unsigned kk = (unsigned)k - s.hc_above[hk];
                if (threadIdx.x < 256) {
                    const int l = threadIdx.x;
                    if (s.lc_above[l] < kk && kk <= s.lc_above[l] + s.lc[l]) s.pick = l;
                }
                __syncthreads();
                lk = s.pick;
                Z = s.hm_above[hk] + s.lm_above[lk] + s.lm[lk];
                cut = ((unsigned)hk << 8) | (unsigned)lk;
            }
            if (use_p) {
                const double thr = (double)p * (double)Z;
                // high byte of the top-p cut-off: the lowest occupied bin (at or above the top-k bin) whose strictly-larger mass
                // is below p * Z
                __syncthreads();
                if (threadIdx.x == 0) s.pick = 255;
                __syncthreads();
                if (threadIdx.x < 256) {
                    const int h = threadIdx.x;
                    if (h >= hk && s.hc[h] > 0 && (double)s.hm_above[h] < thr) atomicMin(&s.pick, h);
                }
                __syncthreads();
                const int hp = s.pick;
                __syncthreads();
                if (!(use_k && hp == hk))
                    histogram(s, row, V, hp, floor, m, invT, true, s.lc, s.lm, s.lc_above, s.lm_above);
                const int lo_min = (use_k && hp == hk) ? lk : 0;   // inside the top-k bin only the top-k survivors count
                if (threadIdx.x == 0) s.pick = 255;
                __syncthreads();
                if (threadIdx.x < 256) {
                    const int l = threadIdx.x;
                    if (l >= lo_min && s.lc[l] > 0 && (double)(s.hm_above[hp] + s.lm_above[l]) < thr) atomicMin(&s.pick, l);
                }
                __syncthreads();
                cut = ((unsigned)hp << 8) | (unsigned)s.pick;
            }
        }
        // Gumbel-max over the kept tokens.  The maximum's own key is a lower bound of the winning key, and the noise is below
        // kGumbelMax, so a token with l / T + kGumbelMax below that bound cannot win: Philox and the logs run only for groups
        // of 4 that hold a kept token above it.
        const uint4 xm = philox4x32_10(make_uint4((uint32_t)(amax >> 2), (uint32_t)st, 0u, 0u), k0, k1);
        const uint32_t xw = (amax & 2) ? ((amax & 1) ? xm.w : xm.z) : ((amax & 1) ? xm.y : xm.x);
        const float lo = (m * invT - logf(neg_log_u(xw)) - kGumbelMax) * T;                // candidates: l >= lo
        for (int c = threadIdx.x; c < nchunks; c += blockDim.x) {
            float f[8];
            unpack8(__ldg(reinterpret_cast<const uint4*>(row) + c), f);
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                bool any = false;
#pragma unroll
                for (int j = 0; j < 4; ++j) any |= f[4 * g + j] >= lo && sort_key(f[4 * g + j]) >= cut;
                if (!any) continue;
                const uint4 x = philox4x32_10(make_uint4((uint32_t)(2 * c + g), (uint32_t)st, 0u, 0u), k0, k1);
                const uint32_t xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float l = f[4 * g + j];
                    if (l < lo || sort_key(l) < cut) continue;
                    const float key = l * invT - logf(neg_log_u(xs[j]));
                    if (key > best) { best = key; bidx = c * 8 + 4 * g + j; }       // strictly greater: first index kept
                }
            }
        }
    }
    block_argmax(best, bidx, s.sb, s.si);
    if (threadIdx.x == 0) {
        long long tok = bidx;
        if (forced) tok = forced[(long long)b * forced_ld + st];   // teacher forcing (parity tests)
        if (finished) {
            if (finished[b]) tok = pad_id;
            else {
                bool hit = false;
#pragma unroll
                for (int i = 0; i < DOTS_MAX_STOP_IDS; ++i) hit |= (i < stops.n) && (tok == stops.id[i]);
                if (hit) finished[b] = 1;
            }
        }
        next_ids[b] = tok;
        if (out_ids) out_ids[(long long)b * out_ld + st] = tok;
        if (step) step[b] = st + 1;
        if (pos) pos[b] += 1;
        if (ctx_len) ctx_len[b] += 1;
    }
}

}  // namespace
}  // namespace dots

using namespace dots;
#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" int dots_sample_advance(const void* logits, long long ldl, int batch, int vocab, long long* next_ids, long long* out_ids,
                                   long long out_ld, int* step, int* pos, int* ctx_len, int* finished, const long long* stop_ids,
                                   int n_stops, long long pad_id, const long long* forced_ids, long long forced_ld,
                                   const float* temperature, const float* top_p, const int* top_k, const unsigned long long* seed,
                                   void* stream) {
    DOTS_REQUIRE(batch > 0 && vocab % 8 == 0 && ldl % 8 == 0, "dots_sample_advance: vocab and pitch must be multiples of 8");
    DOTS_REQUIRE(n_stops >= 0 && n_stops <= DOTS_MAX_STOP_IDS && (n_stops == 0 || stop_ids), "dots_sample_advance: at most %d stop ids (got %d)",
                 DOTS_MAX_STOP_IDS, n_stops);
    DOTS_REQUIRE(temperature && top_p && top_k && seed, "dots_sample_advance: temperature, top_p, top_k and seed are required");
    StopIds stops{};
    stops.n = n_stops;
    for (int i = 0; i < n_stops; ++i) stops.id[i] = stop_ids[i];
    DOTS_CHECK_CUDA(launch_ex(sample_advance_kernel, dim3(batch), dim3(kThreads), (size_t)(0), ST(stream), true, (const bf16*)logits, ldl,
                              vocab, next_ids, out_ids, out_ld, step, pos, ctx_len, finished, stops, pad_id, forced_ids, forced_ld,
                              temperature, top_p, top_k, seed));
    return 0;
}
