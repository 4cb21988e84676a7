// kernels.h -- launchers of the HBM-bound kernels of the VBLinear path (elementwise.cu).
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace vbnn {

constexpr int kMaxPartials = 1184;   // 148 SMs x 8 blocks
constexpr int kStatSlots = 16;

// VBLinear:sample (VBLinear.lua:49-64): W_s = mu + sigma .* eps_s for S samples at once.
struct SampleParams {
  const float* mu;          // [O x I]
  const float* sig;         // stdv cache (strict_reference) or lvars
  int sig_is_lvar;
  int O, I, S;
  PhiloxStream ps;          // sample index = ps.sample + s
  const uint32_t* step_ptr;
  const float* eps_in;      // nullable [S x O x I]: injected epsilon
  float* eps_out;           // nullable [S x O x I]: keep epsilon (self.e)
  float* w_f32;             // nullable [S x O x I]
  bf16* w_bf16; int ld_bf16; long long zs_bf16;   // nullable [S x O x ld]
  void* eps16;              // nullable [S x O x ld] (__half, same pitch / stride as w_bf16): epsilon kept for the dW epilogue
};
int launch_sample_w(const SampleParams& p, cudaStream_t st);

// VBLinear:compute_prior (VBLinear.lua:77-88): per-block partial sums of exp(lvar) + mu^2.
int launch_prior_partials(const float* mu, const float* lvar, long long n, double* partials,
                          int* n_partials_out, cudaStream_t st);
// same reduction with a fixed grid, written to the half of a 2 x kMaxPartials ping-pong buffer that
// the next update of the layer will read: partials2 + (*t_dev & 1) * kMaxPartials
int launch_prior_partials_pp(const float* mu, const float* lvar, long long n, double* partials2,
                             const int* t_dev, int grid, cudaStream_t st);
int update_grid(int O, int I);
// The prior N(mu_hat, var_hat) of the KL terms (include/vbnn.h, enum vbnn_prior): Graves' empirical
// (mu_hat = 0, var_hat = mean(sigma^2 + mu^2)), fixed scalars, or per-weight arrays [O x I].
struct PriorArgs {
  int kind;                             // enum vbnn_prior
  float mu0, var0, lvar0;               // VBNN_PRIOR_FIXED (lvar0 = log var0)
  const float *mu, *lvar;               // VBNN_PRIOR_PER_WEIGHT: prior means, prior log-variances
};
// finalise var_hat into a device scalar (+ optional caches stdv, mu_sqe = (mu - mu_hat)^2): EMPIRICAL reduces
// the partials (sum / W), FIXED stores var0, PER_WEIGHT stores NaN (there is no scalar prior)
int launch_prior_finalize(const double* partials, int n_partials, long long W, float* var_hat_dev,
                          const float* mu, const float* lvar, float* stdv, float* mu_sqe, const PriorArgs& pr,
                          cudaStream_t st);

// The hyper-parameters the reference reads at every update (vbnn_layer_set_opts): one block per layer in device
// memory.  The update kernels read it when they run, so a captured step graph follows a change without re-capture.
struct LiveOpts { float B, lr_bias, lr_mu, lr_var, beta1, beta2, eps; };
// *dst = v on the stream, by a one-thread kernel (the values travel as its arguments)
int launch_set_live_opts(LiveOpts* dst, const LiveOpts& v, cudaStream_t st);

// VBLinear:update (VBLinear.lua:124-166) minus the bias SGD: KL + likelihood gradients and both
// Adam steps in one pass.
struct UpdateParams {
  float *mu, *lvar;
  const float *gW, *gS;
  float *m_mu, *v_mu, *m_var, *v_var;
  float *stdv, *mu_sqe;                 // nullable: caches of compute_prior (strict_reference)
  bf16 *mu_bf16, *s2_bf16; int ld_bf16; // nullable: tensor-core operand copies (LRT mode)
  float* s2_f32;                        // nullable: sigma^2 operand for the fp32 LRT path
  int O, I;
  const double* partials; int n_partials;
  int partials_pingpong;                // partials / next_partials are 2 x kMaxPartials halves selected by (*t_dev & 1)
  float* var_hat_dev;                   // out: var_hat used by this update
  const int* t_dev;                     // Adam step counter (t BEFORE this update)
  float S;
  const LiveOpts* hp;                   // B, lr_mu, lr_var, beta1, beta2, eps of the layer
  int lrt;
  double* stat_partials;                // nullable [grid x kStatSlots]
  double* next_partials;                // nullable [grid]: sum(exp(lvar_new) + mu_new^2) per block, i.e.
                                        // the compute_prior partials of the NEXT update (saves a read pass)
  // ---- peer mode (row shard of a layer; all pointers above are pre-offset to the shard, O = its rows) ----
  long long W_total;                    // weights of the WHOLE layer (var_hat denominator); 0 -> O * I
  int n_src; long long src_stride;      // > 0: gW / gS are sums of n_src receive slots, src_stride ELEMENTS apart
  int grads_bf16;                       // the slots hold bf16 tiles (gW / gS point at bf16 data; src_stride in bf16 elements)
  int grid_override;                    // > 0: blocks of this launch
  int part_off;                         // this launch's first index in the next_partials array
  int n_peer; double* peer_partials[7]; // next_partials mirrored into the other ranks' arrays (peer stores)
  // all-gather fused into the update (used for layer 0, whose update is the tail of a minibatch and has
  // idle SMs and idle NVLink to itself): every refreshed operand quad is also stored to the n_push
  // other ranks; pointers pre-offset like their local counterparts, nullptr = not pushed
  int n_push;
  bf16* push_mu16[7]; bf16* push_s216[7]; float* push_mu[7]; float* push_lv[7]; float* push_s2[7];
  // ---- co-resident variant (peer mode, layers > 0): 128-thread blocks with <= 80 registers, one per SM,
  // that fit beside a resident tcgen05 GEMM CTA, so a shard's update starts while the persistent GEMMs
  // of the layers below own every SM ----
  int coresident;
  // ---- prior of the KL terms: EMPIRICAL reads var_hat from `partials`; FIXED uses prior.mu0 / prior.lvar0 and
  // skips that reduction; PER_WEIGHT reads prior.mu / prior.lvar (pre-offset to the shard like mu / lvar) ----
  PriorArgs prior;
};
int launch_update(const UpdateParams& p, int* grid_out, cudaStream_t st);

// compute_mugrads / compute_vargrads (VBLinear.lua:90-98) as standalone tensors (API parity).  EMPIRICAL reads var_hat
// from var_hat_dev (mu_hat = 0); FIXED and PER_WEIGHT take mu_hat and log var_hat from pr, as k_update.  B from hp.
int launch_grads(const float* mu, const float* lvar, float* gW, float* gS, long long n,
                 const float* var_hat_dev, const PriorArgs& pr, const LiveOpts* hp, float S, int lrt, float* mleg,
                 float* mlcg, float* vleg, float* vlcg, cudaStream_t st);

// VBLinear:calc_lc (VBLinear.lua:99-103); mu_is_sq: mu_src is the mu_sqe cache (mu - mu_hat)^2.  Prior as in
// launch_grads, B from hp.
int launch_calc_lc(const float* var_src, int var_kind /*0 lvar, 1 stdv*/, const float* mu_src,
                   int mu_is_sq, long long n, const float* var_hat_dev, const PriorArgs& pr, const LiveOpts* hp,
                   float* lc_out, double* partials, int* n_partials_out, cudaStream_t st);

// x -= lr * g  (optim.sgd, VBLinear.lua:125-128, mlp.lua:120-123) + optional bf16 operand copy; *lr is read on the
// device (LiveOpts::lr_bias)
int launch_sgd(float* x, const float* g, long long n, const float* lr, bf16* x_bf16, int I, int ld_bf16,
               cudaStream_t st);
// peer mode: g = sum of n_src receive slots src_stride floats apart
int launch_sgd_slots(float* x, const float* g, int n_src, long long src_stride, long long n, const float* lr,
                     bf16* x_bf16, int I, int ld_bf16, cudaStream_t st);

// LogSoftMax + ClassNLLCriterion forward/backward + accuracy (mlp.lua:30-32,78-82; utils.lua:11-27)
struct LossParams {
  const float* logits; int ld_logits;   // [Z*N x ld]
  const float* targets;                 // [N] 1-based floats, shared by all z
  int N, C, Z;
  float grad_scale;                     // 1 / N_global
  float* g_f32; bf16* g_bf16; int ld_g; // dLoss/dlogits (one of the two)
  float* logp_out;                      // nullable [Z*N x C]
  float* result;                        // [2*Zslots]: result[2z] += sum nll, result[2z+1] += #correct
  int z_slot0;
  // ---- regression criteria (launch_loss_reg) ----
  int criterion;                        // enum vbnn_criterion: VBNN_CRIT_MSE or VBNN_CRIT_GAUSSIAN_NLL
  const void* r; void* h;               // nullable, typed as the gradient: LRT output layer, h = g .* r [Z*N x ld_g]
};
int launch_loss(const LossParams& p, cudaStream_t st);
// The regression criteria of vbnn_mlp_set_criterion, one warp per row like launch_loss.  targets are dense [N x K]
// (MSE: K = C; GAUSSIAN_NLL: K = C / 2, columns [0, K) of a row are means m, [K, 2K) log-variances s); a NaN target
// adds nothing.  grad_scale = 1 / (N_global K).  Per (z, n) it writes dl/dY into g (padding columns zeroed as
// launch_loss leaves them) and h, and adds {sum of loss terms, sum (y - m)^2} into result[2z], result[2z+1]: MSE's loss
// term is (y - m)^2 itself, GAUSSIAN_NLL's 1/2 (s + q^2) with q = (y - m) e^{-s/2}.
int launch_loss_reg(const LossParams& p, cudaStream_t st);
// A caller-supplied dLoss/dlogits (vbnn_mlp_backward_update), dense fp32 [rows x C], into the output layer's
// gradient operand g [rows x ld_g] (bf16 or fp32, padding columns zeroed as launch_loss leaves them) and, when r is
// set (LRT output layer), h = g .* r [rows x ld_g] in the same pass (launch_mul_act's H).
int launch_grad_logits(const float* grad, long long rows, int C, void* g, int ld_g, const void* r, void* h, int is_bf16,
                       cudaStream_t st);

// Bayesian model average over sampled forward passes (vbnn_mlp_predict), one chunk of zc samples per launch.
// Per (row, class) the state is an online log-sum-exp over samples of logp_t = x_t - lse_t: a running max and
// the sum of exp(logp_t - max), so log p-bar = max + log(sum) - log T stays finite wherever every logp_t is.
// Per row it also keeps the sum over samples of the entropies H[p_t].  The first chunk initialises the state,
// the last one finalises it into the outputs instead of storing it.
struct PredictParams {
  const float* logits; int ld_logits;   // [zc*N x ld]
  int N, C, zc;
  int first, last;                      // this chunk starts / ends the average
  int T;                                // samples averaged in all (last chunk)
  float *st_max, *st_sum;               // [N x C] log-sum-exp state
  float* st_ent;                        // [N] sum_t H[p_t]
  float* logp_out;                      // nullable [N x C] log p-bar (last chunk)
  float* unc_out;                       // nullable [N x 4] {H[p-bar], mean_t H[p_t], mutual information, argmax + 1}
  const float* targets;                 // nullable [N] 1-based floats (last chunk)
  double* partials;                     // [grid x 2] per-block {sum nll, #correct} when targets is set
};
// returns the grid in *grid_out (the number of partial pairs written)
int launch_predict(const PredictParams& p, int* grid_out, cudaStream_t st);

// Moments of the raw outputs over sampled forward passes (vbnn_mlp_predict_outputs), one chunk of zc samples per
// launch.  K output columns (RAW: C = K; GAUSSIAN: C = 2K, columns [0, K) means m, [K, 2K) log-variances s).  Per
// (row, mean column) the state is the first sample's value f0, sum_t (m_t - f0) and sum_t (m_t - f0)^2; per (row,
// log-variance column) sum_t exp(s_t) in st_sum; per row (lse) an online log-sum-exp of sum_k log N(y_k; m_tk, e^s_tk).
// The first chunk initialises the state, the last one writes the outputs instead of storing it.
struct MomentsParams {
  const float* out; int ld_out;         // [zc*N x ld] raw outputs of this chunk
  int N, K, gaussian, zc;
  int first, last;                      // this chunk starts / ends the average
  int T;                                // samples averaged in all
  float *st_f0, *st_sum, *st_sq;        // [N x C]
  float *st_lmax, *st_lsum;             // [N] (lse)
  int lse;                              // GAUSSIAN with targets on every chunk: keep the per-row mixture likelihood
  float *mean_out, *epi_out, *ale_out;  // nullable [N x K] (last chunk)
  const float* targets;                 // nullable dense [N x K]
  double* partials;                     // nullable [grid x 2] per-block {sum_n -log p-bar, sum (y - mean)^2} (last chunk)
};
// returns the grid in *grid_out (the number of partial pairs written)
int launch_predict_moments(const MomentsParams& p, int* grid_out, cudaStream_t st);

// gradBias += column sums of G over all rows (nn.Linear:accGradParameters addmv)
int launch_colsum(const void* G, int is_bf16, long long rows, int cols, int ld, float scale,
                  float* gb, cudaStream_t st);

// fp32 [rows x cols] -> bf16 [rows x ld] (+ squared copy): tensor-core operand staging
int launch_cast(const float* src, int src_ld, long long rows, int cols, bf16* dst, bf16* dst_sq,
                int ld, cudaStream_t st);
// uint8 [rows x cols] -> (x - mean) * inv_std as bf16 [rows x ld] (+ squared copy) or fp32 [rows x ld_f32]
// (+ squared copy): data.lua's normalisation (utils.lua:29-35) fused into the operand staging
int launch_cast_u8(const uint8_t* src, long long rows, int cols, float mean, float inv_std, bf16* dst, bf16* dst_sq,
                   int ld, float* dst_f32, float* dst_sq_f32, int ld_f32, cudaStream_t st);
// dst (+)= scale * sum_z src[z * stride + e]: fixed-order reduction of the per-sample partial products of a
// sample-split dW GEMM (deterministic, unlike atomics)
int launch_sum_partials(const float* src, int Z, long long stride, long long n, float scale, int accumulate, float* dst,
                        cudaStream_t st);
// fp32 x -> x^2 (fp32 LRT path)
int launch_square(const float* src, float* dst, long long n, cudaStream_t st);
// fp32 exp() (sigma^2 operand of the fp32 LRT path / bf16 copies at init)
int launch_param_copies(const float* mu, const float* lvar, int O, int I, bf16* mu_bf16,
                        bf16* s2_bf16, int ld, float* s2_f32, cudaStream_t st);

// out = a .* b on activation-typed matrices with independent leading dims (H = G .* R, A12)
int launch_mul_act(const void* a, int lda, int a_is_bf16, const void* b, int ldb, void* out, int ldo,
                   long long rows, int cols, int is_bf16, cudaStream_t st);
int launch_fill(float* dst, long long n, float v, cudaStream_t st);
int launch_init_normal(float* dst, long long n, float mean, float std, PhiloxStream ps,
                       cudaStream_t st);
int launch_philox_matrix(float* dst, int rows, int cols, int row0, PhiloxStream ps, cudaStream_t st);
int launch_bump(uint32_t* step, int** t_ptrs_dev, int n_t, cudaStream_t st);
int launch_snr(const float* mu, const float* lvar, long long n, float thresh, uint8_t* mask,
               unsigned long long* count_dev, cudaStream_t st);
// result[0] = mean over Z of loss sums / div, result[1] = mean over Z of acc[2z+1] / div * scale1: ClassNLL passes
// div = N, scale1 = 100 (mean accuracy %, main.lua:38-39); the regression criteria div = N K, scale1 = 1
int launch_finalize_result(const float* acc, int Z, float div, float scale1, float* out2, cudaStream_t st);

}  // namespace vbnn
