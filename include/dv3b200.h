/* dv3b200 -- C ABI of the B200-native hot path of r9y9/deepvoice3_pytorch.
 *
 * The reference has no FFI of its own (it is pure Python on ATen): the seam it offers is the Python
 * module API (deepvoice3_pytorch.builder.* -> nn.Module, SURVEY.md section 8b).  This header is the
 * C-ABI layer underneath our mirror of that API; each entry point names the reference code whose GPU
 * work (ATen/cuDNN/cuBLAS calls) it replaces.  See INTEGRATION.md for the reference-side binding.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; dv3_last_error() gives the message of the
 *     most recent failure on the calling thread.  No exceptions, no torch types.
 *   - all pointers are caller-owned DEVICE memory (fp32 unless stated), densely packed, row-major with the
 *     last index fastest; kernels never allocate.  `stream` is a cudaStream_t; every call is asynchronous on
 *     it and re-entrant (no global mutable state besides cached device attributes).
 *   - activations use the reference's conv layout (B, C, T), T fastest.
 *   - dropout: keep(i) is a pure function of (*seed_ptr, salt, element index i); `seed_ptr` points to 8
 *     bytes of device memory (so a captured CUDA graph gets fresh masks by bumping it), `salt` identifies the
 *     call site.  p_drop == 0 or seed_ptr == NULL disables it.
 *   - tensors must have fewer than 2^31 elements.
 */
#ifndef DV3B200_H
#define DV3B200_H

#ifdef __cplusplus
extern "C" {
#endif

const char* dv3_last_error(void);
int dv3_abi_version(void);
/* number of kernels this library has launched in this process (every launch is counted once) */
long long dv3_launch_count(void);

/* ---- weight normalisation: reference modules.py:85,100,109 (nn.utils.weight_norm pre-hook) -------------
 * v is [R][X][k] (k fastest), g is [R]; w = g*v/||v[r]||.  Writes w in up to two packed layouts:
 * out1[r*s1r + x*s1x + j*s1j] and out2[r*s2r + x*s2x + j*s2j] (either may be NULL).
 * inv_norm, scale: [R] outputs (1/||v||, g/||v||), inv_norm is needed by the backward. */
int dv3_weightnorm_fwd(const float* v, const float* g, float* inv_norm, float* scale, float* out1,
                       float* out2, int R, int X, int k, long long s1r, long long s1x, long long s1j,
                       long long s2r, long long s2x, long long s2j, void* stream);
/* dw_partials: [nsplit][R*X*k] partial gradients w.r.t. w (summed here; slot 0 is overwritten with the sum), in
 * v's own layout (r,x,j) when tap_major = 0 or as [j][r][x] when tap_major = 1; outputs dv [R][X][k], dg [R],
 * overwritten (accumulate = 0) or added to (accumulate = 1, e.g. straight into a flat gradient arena). */
int dv3_weightnorm_bwd(float* dw_partials, long long split_stride, int nsplit, int tap_major, const float* v,
                       const float* g, const float* inv_norm, float* dv, float* dg, int R, int X, int k,
                       int accumulate, void* stream);

/* ---- fused ConvBlock forward: reference modules.py:145-164 (Conv1dGLU._forward, mode 0) and
 * modules.py:200-226 (HighwayConv1d._forward, mode 1).
 * x (B,C,T); w_f packed [k][C][2C]; bias [2C]; spk (B,C,T) = softsign(speaker_proj(.)) transposed, or NULL;
 * y (B,C,T); save_a / save_s (B,C,T) = gate pre-activation a(+bias+spk) and sigmoid(b) for the backward, or NULL.
 * causal: left pad (k-1)*dilation; else symmetric (k-1)/2*dilation. Dropout is applied to the conv input only. */
int dv3_convblock_fwd(const float* x, const float* w_f, const float* bias, const float* spk, float* y,
                      float* save_a, float* save_s, int B, int C, int T, int k, int dilation, int causal,
                      int mode, int residual, float p_drop, const unsigned long long* seed_ptr,
                      unsigned salt, void* stream);
/* gate backward: dab (B,2C,T) = [d a ; d b], dbias[2C] += row sums (may be NULL). x only read in mode 1. */
int dv3_convblock_gate_bwd(const float* dy, const float* a, const float* s, const float* x, float* dab,
                           float* dbias, int B, int C, int T, int mode, int residual, void* stream);

/* ---- plain weight-normed Conv1d (+ fused ReLU): reference conv.py:7-15 via modules.py:94-100.
 * x (B,Cin,T); w_f packed [k][Cin][Cout]; y (B,Cout,T). */
int dv3_conv1d_fwd(const float* x, const float* w_f, const float* bias, float* y, int B, int Cin, int Cout,
                   int T, int k, int dilation, int causal, int relu, void* stream);
/* data gradient of a conv with M output rows: dx (B,Cin,T) = mask * convT(dab (B,M,T), w_b [k][M][Cin]) + addend.
 * mask = the forward's input-dropout mask (same seed/salt).  addmode 0: none; 1: + alpha*e1; 2: + e1*(1-e2)
 * (e1, e2 (B,Cin,T)) -- the residual-path gradients of the GLU / highway blocks. */
int dv3_conv1d_dgrad(const float* dab, const float* w_b, float* dx, int B, int M, int Cin, int T, int k,
                     int dilation, int causal, float p_drop, const unsigned long long* seed_ptr,
                     unsigned salt, int addmode, const float* e1, const float* e2, float alpha,
                     void* stream);
/* weight gradient, split over (b,t): writes dv3_conv1d_wgrad_nsplit(...) partials of `split_stride` floats each;
 * element (m, ci, j) of a partial lives at (m%msplit)*s_m + (m/msplit)*s_mh + ci*s_n + j*s_j. */
int dv3_conv1d_wgrad_nsplit(int B, int M, int Cin, int T, int k);
int dv3_conv1d_wgrad(const float* dab, const float* x, float* dw_partials, long long split_stride, int B,
                     int M, int Cin, int T, int k, int dilation, int causal, float p_drop,
                     const unsigned long long* seed_ptr, unsigned salt, int msplit, int s_m, int s_mh,
                     int s_n, int s_j, void* stream);
/* dyr = relu ? dy*(y>0) : (untouched); dbias[C] += sum_{b,t} dyr.  dy,y,dyr (B,C,T). */
int dv3_bias_act_bwd(const float* dy, const float* y, float* dyr, float* dbias, int B, int C, int T,
                     int relu, void* stream);

/* ---- layout change (B,R,C) -> (B,C,R): every x.transpose(1,2) between the attention (B,T,C) and conv (B,C,T)
 * layouts, reference deepvoice3.py:86,93,318,324,340-345,355,359,592,602; nyanko.py:66,206,214-217,230,234,402. */
int dv3_transpose(const float* in, float* out, int B, int R, int C, void* stream);

/* ---- embedding lookup: reference deepvoice3.py:74, nyanko.py:64,201-203,__init__.py:69-71 (F.embedding).
 * ids int64 [N] -> out (N,D); an id outside [0,V) sets *err_flag (device int) to 1 and writes nothing.
 * bwd: dtable[ids[n]] += dy[n] except rows == padding_idx (pass -1 for none); dtable must be pre-zeroed. */
int dv3_embedding_fwd(const long long* ids, const float* table, float* out, int N, int D, int V, int* err_flag,
                      void* stream);
int dv3_embedding_bwd(const long long* ids, const float* dy, float* dtable, int N, int D, int V,
                      long long padding_idx, void* stream);

/* ---- sinusoidal position encoding: reference modules.py:27-31,45-64 (SinusoidalEncoding.forward).
 * pos int64 (B,T) in [0,P); table (P,D) raw (non-sinusoidal) table; w [nw] position rate(s), nw in {1,B};
 * out (B,T,D).  bwd accumulates into pre-zeroed dtable (P,D) and dw [nw] (either may be NULL). */
int dv3_sinusoid_fwd(const long long* pos, const float* table, const float* w, int nw, float* out, int B, int T,
                     int D, int P, int* err_flag, void* stream);
int dv3_sinusoid_bwd(const long long* pos, const float* table, const float* w, int nw, const float* dy,
                     float* dtable, float* dw, int B, int T, int D, int P, void* stream);

/* ---- standalone dropout y = x*mask/(1-p): reference F.dropout at deepvoice3.py:75,80,294,321,588,597.
 * Calling it on the gradient with the same (seed, salt) is the backward. */
int dv3_dropout(const float* x, float* y, long long n, float p, const unsigned long long* seed_ptr, unsigned salt,
                void* stream);

/* ---- masked row softmax + dropout: reference deepvoice3.py:145-148,161-165.
 * s (rows,L); mask (rows/rows_per_b, L) bytes, 1 = padding (-inf), or NULL; probs = softmax (the returned
 * alignment); pd = dropout(probs) (may be NULL).  bwd: ds = P*(g - <g,P>), g = dpd*dropmask + dprobs_ext. */
int dv3_softmax_fwd(const float* s, const unsigned char* mask, float* probs, float* pd, int rows, int L,
                    int rows_per_b, float p, const unsigned long long* seed_ptr, unsigned salt, void* stream);
int dv3_softmax_bwd(const float* probs, const float* dpd, const float* dprobs_ext, float* ds, int rows, int L,
                    float p, const unsigned long long* seed_ptr, unsigned salt, void* stream);

/* ---- ConvTranspose1d(k=2,s=2) time interleave: reference deepvoice3.py:519,527; nyanko.py:372,377.
 * in (B,2C,T) rows ordered (j,co) -> out (B,C,2T), out[b,co,2t+j] = in[b,j*C+co,t]; inverse=1 undoes it. */
int dv3_interleave2(const float* in, float* out, int B, int C, int T, int inverse, void* stream);

/* ---- batched strided GEMM C[b] = alpha*A_b*B_b (+C): the attention contractions, reference
 * deepvoice3.py:143 (bmm(q,k)), :167 (bmm(p,v)) and their gradients.  A_b(m,k)=A[b*sAb+m*sAm+k*sAk],
 * B_b(k,n)=B[b*sBb+k*sBk+n*sBn], C_b(m,n)=C[b*sCb+m*ldc+n]; each operand needs one unit stride. */
int dv3_bgemm(const float* A, long long sAb, long long sAm, long long sAk, const float* B, long long sBb,
              long long sBk, long long sBn, float* C, long long sCb, int ldc, int batch, int M, int N, int K,
              float alpha, int accumulate, void* stream);

/* ---- fused tensor-core attention (tcgen05, split-bf16 operands staged and split in-kernel): reference
 * deepvoice3.py:132-176 between the projections.  q (B,E,Td), k / v (B,E,Ts), mask (B,Ts) bytes (1 = padding) or
 * null -> probs (B,Td,Ts) = softmax(q^T k) (pre-dropout, returned as the alignment), out (B,E,Td) =
 * scale * v . dropout(probs)^T.  Backward: dout (B,E,Td), dprobs (B,Td,Ts) gradient arriving at the returned
 * probabilities (or null) -> dq, dk, dv; ds is a (B,Td,Ts) scratch.  Shapes: dv3_tc_attn_supported (Ts <= 128,
 * E % 16 == 0, E <= 256); others go through dv3_bgemm + dv3_softmax_*.  An utterance whose keys are all masked has
 * no softmax: both paths return NaN for its probabilities and context, as torch's softmax of a row of -inf does, and
 * NaN for its dq, dk and dv (torch's masked_fill backward gives 0 for dq and dk there; the loss is NaN either way).
 * Pinned by tests/test_gpu_attention_core.py. */
int dv3_tc_attn_supported(int B, int E, int Td, int Ts);
int dv3_tc_attn_fwd(const float* q, const float* k, const float* v, const unsigned char* mask, float* probs,
                    float* out, int B, int E, int Td, int Ts, float scale, float p_drop,
                    const unsigned long long* seed_ptr, unsigned salt, void* stream);
int dv3_tc_attn_bwd(const float* dout, const float* q, const float* k, const float* v, const float* probs,
                    const float* dprobs, float* ds, float* dq, float* dk, float* dv, int B, int E, int Td, int Ts,
                    float scale, float p_drop, const unsigned long long* seed_ptr, unsigned salt, void* stream);

/* ---- optimizer step over a flat fp32 arena: reference train.py:756-759 (clip_grad_norm_ + Adam.step).
 * dv3_sumsq: out[0] = sum(x^2), deterministic (per-block partials in `scratch`, summed in index order by the block
 * that finishes last: bit-identical on every data-parallel replica); scratch = dv3_sumsq_scratch_floats() floats,
 * zero-filled once by the caller.  dv3_adam_clip: g' = g*hyper[3]*min(1, max_norm/(||g*hyper[3]||+1e-6))
 * (max_norm <= 0: no clipping), then torch.optim.Adam's update with lr=hyper[0], bias corrections hyper[1], hyper[2].
 * hyper (4 floats) and sumsq live in device memory: no host sync, graph-replayable. */
int dv3_sumsq_scratch_floats(void);
int dv3_sumsq(const float* x, long long n, float* out, float* scratch, void* stream);
int dv3_adam_clip(float* p, const float* g, float* m, float* v, long long n, const float* hyper,
                  const float* sumsq, float beta1, float beta2, float eps, float max_norm, void* stream);

/* ---- fused STFT -> linear + mel front-end: reference audio.py:31-34 (spectrogram) and :46-51 (melspectrogram)
 * incl. preemphasis (:21-23), lws sqrt-Hann STFT 1024/256 with 768-sample zero padding (:54-55), mel basis product
 * (:64-68), dB (:79-81) and normalisation (:88-89).  wav (nclips, max_len) fp32; lengths int32 [nclips];
 * mel_basis (n_mels, 513) dense with mel_start/mel_len [n_mels] giving each filter's non-zero span;
 * linear (nclips, max_frames, 513) and mel (nclips, max_frames, n_mels) -- the transposed (T, F) layout the
 * preprocessors store (ljspeech.py:72-73); either output may be NULL.  Frames >= a clip's own count are zero-filled (outputs need no
 * initialisation); n_mels <= 128; min_level_db < 0.  Fastest when wav is 16-byte aligned and max_len % 4 == 0 (bulk /
 * 16-byte staging copies; any other pitch works through 4-byte copies, bit-identical results).  The first call on a
 * device builds a 2.7 KB table with a one-off kernel on the given stream (synchronised unless the stream is capturing). */
int dv3_stft_num_frames(int n_samples);
int dv3_stft_mel(const float* wav, const int* lengths, const float* mel_basis, const int* mel_start,
                 const int* mel_len, float* linear, float* mel, int nclips, int max_len, int max_frames,
                 int n_mels, float preemph, float min_level_db, float ref_level_db, void* stream);

/* ---- inverse audio path: reference audio.py:37-43 (inv_spectrogram) and :26-28 (inv_preemphasis).  The reference
 * recovers the phase with the un-vendored `lws` package (parity UNPINNED); restated here as Griffin-Lim on the same
 * sqrt-Hann 1024 / hop 256 / 768-pad frame as dv3_stft_mel (sum of squared windows == 1: synthesis window = analysis
 * window).  The iteration x <- istft(mag * exp(i angle(stft(x)))) is driven by the host (audio.inv_spectrogram).
 * dv3_spec_to_amp: normalised dB (n) -> (10^((S*(-min)+min+ref)/20))^power.  dv3_stft_complex: wav (n_samples) ->
 * spec (nframes,513,2) [re,im]; mag (nframes,513) != NULL projects the result onto that magnitude.  dv3_istft: spec ->
 * wav (n_samples) += overlap-added frames (zero wav first).  dv3_deemphasis: y[n] = x[n] + coef*y[n-1] per clip. */
int dv3_spec_to_amp(const float* spec_norm, float* amp, long long n, float min_level_db, float ref_level_db,
                    float power, void* stream);
int dv3_stft_complex(const float* wav, int n_samples, const float* mag, float* spec, int nframes, void* stream);
int dv3_istft(const float* spec, float* wav, int n_samples, int nframes, void* stream);
int dv3_deemphasis(const float* x, float* y, int nclips, int n_samples, long long stride, float coef, void* stream);

/* ================= tensor-core ConvBlock / conv path: tcgen05 + TMA, split-bf16 operands =================
 * Same reference code as dv3_convblock_fwd / dv3_conv1d_fwd / dv3_conv1d_dgrad / dv3_conv1d_wgrad (modules.py:94-100,
 * 145-164, 200-226 and their autograd).  fp32 operands are split into bf16 planes p0 = bf16(x), p1 = bf16(x-p0)
 * [, p2 = bf16(x-p0-p1)]; npl = 2 issues p0*p0 + p0*p1 + p1*p0 ("x3", ~2^-17/operand), npl = 3 adds
 * p1*p1 + p0*p2 + p2*p0 ("x6", fp32-equivalent).  Plane buffers are bf16 device memory laid out [npl][...]; channel
 * pitches are padded to a multiple of 8.  Callers use the exact-fp32 entry points for unsupported shapes. */
int dv3_tc_supported(int B, int C, int T, int k);           /* gated block: C % 128 == 0, k <= 8 */
int dv3_tc_conv_supported(int B, int Cin, int Cout, int T, int k);   /* plain conv: k == 1 or Cout % 128 == 0 */
/* Operand planes: every fp32 operand x travels as hi = rn16(x), lo = rn16((x - hi) * 2^11) (csrc/common.cuh).
 * Forward GEMMs multiply fp16 pairs (22-bit operands: fp32-class results; activations and normalised weights are O(1),
 * values are clamped to +-65504); gradient GEMMs multiply bf16 pairs (gradients need the fp32 exponent range for any
 * loss scale) -- tcgen05 kind::f16 does not mix formats in one MMA, so a conv input is split into both.
 * x (B,C,T) fp32 -> conv-input dropout -> btc: [2][B][T][Cp] fp16 pair (forward operand, Cp = pad8(C)) and
 * bct (may be NULL): [2][B][T][Cp] bf16 pair of the same values (operand of the weight gradient). npl must be 2. */
int dv3_tc_split_input(const float* x, void* btc, int npl, void* bct, int B, int C, int T, int k, int dilation,
                       int causal, float p_drop, const unsigned long long* seed_ptr, unsigned salt, void* stream);
/* gate backward writing dAB = [da ; db] as planes btc: [2][B][T][2C] (dgrad operand), bct: [2][B][2C][T] (wgrad). */
int dv3_tc_gate_bwd_split(const float* dy, const float* a, const float* s, const float* x, void* btc, void* bct,
                          float* dbias, int B, int C, int T, int mode, int residual, void* stream);
/* plain-conv backward prologue: g = dy*(relu ? y>0 : 1) -> btc: [2][B][T][Cp], bct: [2][B][C][T]; dbias[C] += sums. */
int dv3_tc_grad_split(const float* dy, const float* y, void* btc, void* bct, float* dbias, int B, int C, int T,
                      int relu, void* stream);
/* weight norm + split: v (Cout,Cin,k), g [Cout] -> wfwd: [npl][k][Cout][Cinp] (forward), wbwd: [2][k][Cin][Coutp] (dgrad). */
int dv3_tc_weightnorm_fwd(const float* v, const float* g, float* inv_norm, float* scale, void* wfwd, int npl,
                          void* wbwd, int Cout, int Cin, int k, void* stream);
/* ConvTranspose1d(k=2,s=2) weight v (Cin,Cout,2), g [Cin] as a 1x1 conv with 2*Cout rows ordered (j,co):
 * wfwd: [npl][2*Cout][Cinp], wbwd: [2][Cin][pad8(2*Cout)]. */
int dv3_tc_weightnorm_convt_fwd(const float* v, const float* g, float* inv_norm, float* scale, void* wfwd, int npl,
                                void* wbwd, int Cin, int Cout, void* stream);
/* Batched weight norm (csrc/wn_batched.cu): one record per weight-normed conv (v (Cout,Cin,k), g [Cout]); the table
 * lives in DEVICE memory, blk_* are the first block of the record in the batched norm / pack / backward launches
 * (ascending over the table), pack_gx = ceil(Cin*k / 32).  Layouts as dv3_tc_weightnorm_fwd with npl = 2; the
 * backward consumes tap-major partials [nsplit][k][Cout][Cin] (what dv3_tc_wgrad_mn writes; slot 0 is scratch). */
typedef struct Dv3WnEntry {
    const float* v; const float* g; float* inv_norm; float* scale;
    void* wfwd; void* wbwd;
    float* partials; float* dv; float* dg;
    long long split_stride;
    int Cout, Cin, k, nsplit;
    int blk_norm, blk_pack, blk_bwd, pack_gx;
} Dv3WnEntry;
/* norm + pack of every record: 2 launches (replaces 2 launches per layer). */
int dv3_tc_weightnorm_fwd_batched(const Dv3WnEntry* table_dev, int n, int norm_blocks, int pack_blocks,
                                  void* stream);
/* split-K reduction + dg / dv of every record: 1 launch; accumulate = 1 adds into dv / dg. */
int dv3_weightnorm_bwd_batched(const Dv3WnEntry* table_dev, int n, int bwd_blocks, int accumulate, void* stream);
/* gated forward: xd = btc planes of dv3_tc_split_input, w = wfwd planes [npl][k][2C][C].
 * reserved must be NULL (any other value is refused); it keeps the argument list of ABI version 1. */
int dv3_tc_convblock_fwd(const void* xd, const void* w, int npl, const float* bias, const float* spk,
                         const float* res, float* y, float* save_a, float* save_s, int B, int C, int T, int k,
                         int dilation, int causal, int mode, int residual, const void* reserved, void* stream);
/* generic conv / data gradient: out (B,Nc,T) = sum_j A[b,t+off_j,:].W[j,n,:], then *dropmask, +bias, +addend, relu.
 * a: [npl][B][T][pad8(Kc)], w: [npl][k][Nc][pad8(Kc)]; transpose_taps = 1 for a data gradient.
 * reserved must be NULL, as for dv3_tc_convblock_fwd. */
int dv3_tc_conv(const void* a, const void* w, int npl, float* out, int B, int Kc, int Nc, int T, int k, int dilation,
                int causal, int transpose_taps, const float* bias, int relu, float p_drop,
                const unsigned long long* seed_ptr, unsigned salt, int addmode, const float* e1, const float* e2,
                float alpha, const void* reserved, void* stream);
/* weight gradient from the (B,T,C) planes (MN-major operands, tap shift = TMA row coordinate):
 * dy: [2][B][T][pad8(Mw)], xd: [2][B][T][pad8(Nw)]; partial element (m,n,j) of split s at
 * dw_partials + s*split_stride + (m%msplit)*s_m + (m/msplit)*s_mh + n*s_n + j*s_j; dv3_tc_wgrad_nsplit(...) splits. */
int dv3_tc_wgrad_nsplit(int B, int Mw, int Nw, int T, int k);
int dv3_tc_wgrad_mn(const void* dy, const void* xd, float* dw_partials, long long split_stride, int B, int Mw,
                    int Nw, int T, int k, int dilation, int causal, int msplit, long long s_m, long long s_mh,
                    long long s_n, long long s_j, void* stream);

/* ---- fused training losses + gradients: reference train.py:537-601 (spec_loss, guided_attention) and :704-740.
 * dv3_spec_loss: pairs (y_hat[b,t], y[b,t+r]), t < T-r; lengths int64 [B] valid target frames; adds
 * (1-bw)*L1 + bw*binary_divergence (each = w*masked_mean + (1-w)*mean) to loss[0]; grad (B,T,D) = dLoss/dy_hat.
 * priority_bin > 0 and priority_weight > 0: L1 = (1-pw)*L1(all D bins) + pw*L1(bins < priority_bin), train.py:559-567.
 * dv3_aux_loss: adds BCE(done_hat, done) and, if use_attn, mean(attn*W) with the guided-attention mask
 * W[b,t,n] = 1-exp(-(n/in_len[b] - t/dec_len[b])^2/(2 sigma^2)) built on the fly; writes both gradients. */
int dv3_spec_loss(const float* y_hat, const float* y, const long long* lengths, float* grad, float* loss, int B,
                  int T, int D, int r, float masked_loss_weight, float binary_divergence_weight, int priority_bin,
                  float priority_weight, void* stream);
int dv3_aux_loss(const float* done_hat, const float* done, float* d_done, long long n_done, const float* attn,
                 float* d_attn, const long long* in_len, const long long* dec_len, int A, int B, int Td, int Ts,
                 float sigma, int use_attn, float* loss, void* stream);

/* ---- incremental (autoregressive) decoding: reference conv.py:17-46, deepvoice3.py:367-485, nyanko.py:250-338 ----
 * All loop state lives in device memory so that one decoder step is the same launch sequence every time (CUDA-graph
 * replay): *t_ptr is the step counter; every row pointer advances by a per-step stride: row b of step t of operand
 * X is X + b*X_ld + t*X_t (floats). */
typedef struct Dv3IncStep {
    const float* x; long long x_ld, x_t;          /* current input (B, Cin) */
    const float* add; long long add_ld, add_t;    /* optional, added to the input (position encoding) */
    float* ring;                                   /* (B, (k-1)*dilation+1, Cin) zero-initialised history; NULL: k = 1 */
    const float* w; const float* bias;             /* normalised weight linearised as [Cout][k][Cin]; [Cout] */
    const float* spk; long long spk_ld;            /* GLU: softsign(speaker_proj(embed)) (B, C) or NULL */
    const float* res1; long long res1_ld, res1_t;  /* y = (y + res1)*sqrt(.5) if non-NULL, then the same with res2 */
    const float* res2; long long res2_ld, res2_t;
    float* y; long long y_ld, y_t;
    float* y2; long long y2_ld, y2_t;              /* optional second output, see y2_mode */
    const float* yadd; long long yadd_ld, yadd_t;  /* y2_mode 2: y2 = y + yadd (position encoding of the query) */
    const int* t_ptr;
    int B, Cin, Cout, k, dilation;
    int mode;                                      /* 0 plain conv, 1 GLU (a*sigmoid(b)), 2 highway */
    int act;                                       /* plain: 0 none, 1 ReLU, 2 sigmoid */
    int vec4;                                      /* 1: Cin % 4 == 0 and every input row is 16-byte aligned */
    int y2_mode;                                   /* 1: y2 = sigmoid(y); 2: y2 = y + yadd */
} Dv3IncStep;
int dv3_inc_conv_step(const Dv3IncStep* step, void* stream);
typedef struct Dv3IncAttn {
    const float* q; long long q_ld;                /* projected query (B, E) */
    const float* keys; const float* values;        /* (B, E, Ts) pre-transposed, (B, Ts, E): projected once */
    float* ctx; long long ctx_ld;                  /* context * Ts*sqrt(1/Ts) (B, E) */
    float* align; long long align_ld, align_t;     /* probabilities * align_scale, or NULL */
    int* last_attended;                            /* int[2] (slot t&1 read, (t+1)&1 written) or NULL: no window */
    const int* t_ptr;
    float align_scale;
    int B, E, Ts, window_backward, window_ahead;
} Dv3IncAttn;
int dv3_inc_attn_step(const Dv3IncAttn* attn, void* stream);
int dv3_inc_advance(int* t_ptr, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DV3B200_H */
