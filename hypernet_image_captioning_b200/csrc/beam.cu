// Batched, device-resident beam search bookkeeping for HyperNet.test_step (reference hypernet_attention.py:247-326,
// beam_size = 3 at :44).  The reference keeps, per image, k live beams: after every decoder step it adds the rows'
// log-softmax to their running scores, takes the top k_live of the k_live * V candidates (step 1: of row 0 only, :274-275),
// moves the beams that just produced </s> to the "complete" list and shrinks k (:296-303), and carries hidden state,
// score and token history of the others to the next step -- all with host-side lists and .item()/.tolist() round trips.
//
// Here all B images advance together: rows b*k .. b*k+k-1 belong to image b (live beams first), the decoder step runs on
// all B*k rows, and ONE kernel (a CTA per image) does everything between two decoder steps on the device:
//   log-sum-exp of every live row -> top-k_live over (live rows x V) by k_live passes of a block-wide arg-max (ties: lower
//   flat index first, like a stable descending sort) -> completed beams appended to the image's complete list ->
//   surviving beams compacted, their token history / score / hidden state gathered from the parent row -> next input words
//   (-1 = zero embedding: the reference zeroes EVERY row's embedding whenever the first row's previous word is 0, :265-266).
// The host reads results once, after the last step.
#include "common.cuh"

namespace caphn {

constexpr int BS_THREADS = 256, BS_MAXK = 8;

struct BeamArgs {
    const float* logits;     // [B*k, V]
    const float* h_out;      // [B*k, H]  hidden state after this step
    float* h_next;           // [B*k, H]  hidden state of the surviving beams (next step's h_{t-1})
    float* scores;           // [B*k]     running scores of the live beams (in/out)
    int* live;               // [B]       live beams (in/out)
    int* prev_tok;           // [B*k]     token each live beam ended with (out)
    long long* words;        // [B*k]     embedding row to feed next (-1: zero vector) (out)
    const int* seq_in;       // [B*k, L]
    int* seq_out;            // [B*k, L]
    float* comp_score;       // [B*k]
    int* comp_seq;           // [B*k, L]
    int* comp_len;           // [B*k]
    int* ncomp;              // [B]
    int* failed;             // [B]  set when beams are still open after the last step (reference returns no caption)
    int B, k, V, H, L, step, end_tok, last;
};

__device__ __forceinline__ bool better(float s, int i, float bs, int bi) { return s > bs || (s == bs && i < bi); }

__global__ void __launch_bounds__(BS_THREADS) beam_step_kernel(const BeamArgs a) {
    __shared__ float s_lse[BS_MAXK], s_ts[BS_MAXK], s_rv[BS_THREADS / 32];
    __shared__ int s_ri[BS_THREADS / 32];
    __shared__ float s_pick_s[BS_MAXK];
    __shared__ int s_pick_i[BS_MAXK], s_src[BS_MAXK], s_word[BS_MAXK], s_newn, s_zero;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k = a.k, V = a.V, L = a.L;
    const int n = a.live[b];
    const long r0 = (long)b * k;
    if (n == 0) {
        for (int j = tid; j < k; j += BS_THREADS) a.words[r0 + j] = -1;
        return;
    }
    const int nrows = a.step == 1 ? 1 : n;        // step 1 ranks row 0 only
    // ---- log-sum-exp of every candidate row ----
    for (int r = 0; r < nrows; ++r) {
        const float* x = a.logits + (r0 + r) * V;
        float mx = -INFINITY;
        for (int v = tid; v < V; v += BS_THREADS) mx = fmaxf(mx, x[v]);
        mx = warp_max(mx);
        if (lane == 0) s_rv[warp] = mx;
        __syncthreads();
        mx = s_rv[0];
        for (int w = 1; w < BS_THREADS / 32; ++w) mx = fmaxf(mx, s_rv[w]);
        __syncthreads();
        float sum = 0.f;
        for (int v = tid; v < V; v += BS_THREADS) sum += expf(x[v] - mx);
        sum = warp_sum(sum);
        if (lane == 0) s_rv[warp] = sum;
        __syncthreads();
        if (tid == 0) {
            float t = 0.f;
            for (int w = 0; w < BS_THREADS / 32; ++w) t += s_rv[w];
            const float lse = mx + logf(t);
            s_lse[r] = isfinite(lse) ? lse : NAN;      // a NaN / +inf logit or an all -inf row: every score NaN, no candidate
            s_ts[r] = a.scores[r0 + r];
        }
        __syncthreads();
    }
    // ---- top-n of the nrows * V candidates: n passes, pass j takes the best candidate that comes after pick j-1.  A NaN
    //      score is never `after` anything: such candidates are not eligible ----
    float last_s = INFINITY;
    int last_i = -1;
    const int ncand = nrows * V;
    int found = n;
    for (int j = 0; j < n; ++j) {
        float bs = -INFINITY;
        int bi = 0x7fffffff;
        for (int c = tid; c < ncand; c += BS_THREADS) {
            const int r = c / V, v = c - r * V;
            const float s = s_ts[r] + (a.logits[(r0 + r) * V + v] - s_lse[r]);
            const bool after = s < last_s || (s == last_s && c > last_i);      // false for NaN
            if (after && better(s, c, bs, bi)) { bs = s; bi = c; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float os = __shfl_xor_sync(0xffffffffu, bs, o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (better(os, oi, bs, bi)) { bs = os; bi = oi; }
        }
        if (lane == 0) { s_rv[warp] = bs; s_ri[warp] = bi; }
        __syncthreads();
        if (tid == 0) {
            float fs = s_rv[0];
            int fi = s_ri[0];
            for (int w = 1; w < BS_THREADS / 32; ++w)
                if (better(s_rv[w], s_ri[w], fs, fi)) { fs = s_rv[w]; fi = s_ri[w]; }
            s_pick_s[j] = fs;
            s_pick_i[j] = fi;
        }
        __syncthreads();
        last_s = s_pick_s[j];
        last_i = s_pick_i[j];
        if (last_i == 0x7fffffff) { found = j; break; }   // (block-uniform) no eligible candidate left
    }
    if (found < n) {
        // the image ends without a caption, and nothing is read through the missing pick
        if (tid == 0) { a.live[b] = 0; a.failed[b] = 1; }
        for (int j = tid; j < k; j += BS_THREADS) a.words[r0 + j] = -1;
        return;
    }
    // ---- bookkeeping (one thread): completed beams out, survivors compacted ----
    const int len = a.step;                       // tokens in every live history (leading 0 + step-1 words)
    if (tid == 0) {
        int newn = 0, nc = a.ncomp[b];
        for (int j = 0; j < n; ++j) {
            const int idx = s_pick_i[j];
            const int parent = idx / V, word = idx - parent * V;
            if (word != a.end_tok) {
                s_src[newn] = parent;
                s_word[newn] = word;
                s_pick_s[newn] = s_pick_s[j];     // newn <= j: never overwrites an unread pick
                ++newn;
            } else {
                const long c = r0 + nc;
                a.comp_score[c] = s_pick_s[j];
                const int* src = a.seq_in + (r0 + parent) * L;
                int* dst = a.comp_seq + c * L;
                for (int t = 0; t < len && t < L; ++t) dst[t] = src[t];
                if (len < L) dst[len] = word;
                a.comp_len[c] = min(len + 1, L);
                ++nc;
            }
        }
        a.ncomp[b] = nc;
        a.live[b] = newn;
        s_newn = newn;
        s_zero = newn > 0 && s_word[0] == 0;      // reference :265-266: zero EVERY row's embedding when the first row's word is 0
        if (a.last && newn > 0) a.failed[b] = 1;
    }
    __syncthreads();
    const int newn = s_newn;
    for (int j = tid; j < k; j += BS_THREADS) {
        if (j < newn) {
            a.scores[r0 + j] = s_pick_s[j];
            a.prev_tok[r0 + j] = s_word[j];
            a.words[r0 + j] = s_zero ? -1 : (long long)s_word[j];
        } else {
            a.words[r0 + j] = -1;
        }
    }
    for (int i = tid; i < newn * L; i += BS_THREADS) {
        const int j = i / L, t = i - j * L;
        int v = 0;
        if (t < len) v = a.seq_in[(r0 + s_src[j]) * L + t];
        else if (t == len) v = s_word[j];
        a.seq_out[(r0 + j) * L + t] = v;
    }
    for (int i = tid; i < newn * a.H; i += BS_THREADS) {
        const int j = i / a.H, h = i - j * a.H;
        a.h_next[(r0 + j) * a.H + h] = a.h_out[(r0 + s_src[j]) * a.H + h];
    }
}

}  // namespace caphn

using namespace caphn;

extern "C" {

// One beam-search bookkeeping step for B images x k beams (see file header).  step is 1-based; last != 0 marks the final
// permitted step (reference: step > max_steps): images that still have open beams get failed[b] = 1.
// seq_in / seq_out: token histories [B*k, L] (ping-pong between steps), L >= max steps + 2.  k <= V: step 1 ranks V
// candidates.  Rows whose log-sum-exp is not finite offer no candidates; an image left with fewer than its live count of
// candidates ends with failed[b] = 1, live[b] = 0.
int caphn_beam_step(const float* logits, const float* h_out, float* h_next, float* scores, int* live, int* prev_tok,
                    long long* words, const int* seq_in, int* seq_out, float* comp_score, int* comp_seq, int* comp_len,
                    int* ncomp, int* failed, int B, int k, int V, int H, int L, int step, int end_tok, int last,
                    void* stream) {
    if (B <= 0 || k <= 0 || k > BS_MAXK || V <= 0 || k > V || H <= 0 || L < 2 || step < 1) return CAPHN_EINVAL;
    BeamArgs a{logits, h_out, h_next, scores, live, prev_tok, words, seq_in, seq_out, comp_score, comp_seq, comp_len,
               ncomp, failed, B, k, V, H, L, step, end_tok, last};
    beam_step_kernel<<<B, BS_THREADS, 0, (cudaStream_t)stream>>>(a);
    CAPHN_RETURN_LAST();
}

}  // extern "C"
