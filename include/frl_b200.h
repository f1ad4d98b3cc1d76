/*
 * frl_b200.h — C ABI of the B200 (sm_100a) data-parallel training-step kernels.
 *
 * The reference (facebookresearch/FRL-Distributed-ML-Scaffold) has no native boundary of its
 * own: its step arithmetic runs inside PyTorch.  Each entry point below replaces the PyTorch
 * call the reference makes at the cited line; the reference-side binding is the ctypes stub in
 * INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (the library never allocates or
 *     frees caller-visible memory) unless the parameter name ends in `_host`;
 *     `*_mapped` pointers may be pinned, device-mapped host memory;
 *   - every function enqueues work on `stream` (a cudaStream_t passed as void*) and returns
 *     immediately; nothing synchronises;
 *   - return value: 0 = ok, negative = argument error (FRL_E_*), positive = cudaError_t of
 *     the launch; `frl_last_error()` gives a thread-local message;
 *   - no exceptions, no longjmp, no global mutable state except the launch counter.
 *   - dtype codes: FRL_F32 = 0, FRL_BF16 = 1, FRL_U8 = 2, FRL_I64 = 3.
 */
#ifndef FRL_B200_H
#define FRL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FRL_ABI_VERSION 1

enum { FRL_F32 = 0, FRL_BF16 = 1, FRL_U8 = 2, FRL_I64 = 3 };
enum { FRL_E_ARG = -1, FRL_E_ALIGN = -2, FRL_E_DTYPE = -3, FRL_E_TOO_MANY = -4 };

int          frl_abi_version(void);
const char*  frl_last_error(void);
/* number of kernels this library has launched since load / since the last reset */
uint64_t     frl_launch_count(void);
void         frl_launch_count_reset(void);
/* SM count and sm arch (major*10+minor) of the current device; <0 on error */
int          frl_device_sm_count(void);
int          frl_device_arch(void);

/* ------------------------------------------------------------------------------------------
 * K2 — fused optimizer update over a flat bucket of the parameter arena.
 * Replaces torch.optim.{SGD,Adam,AdamW,RMSprop}.step() (reference solver.py:162-188, called at
 * solver_worker.py:592) AND the DDP reducer's scale / copy-out passes (reference
 * solver.py:287-289): the reduced gradient is read once, straight from the bucket.
 *
 *   p        fp32 master weights [n]           (read + written)
 *   g        gradient bucket [n], dtype g_dtype (FRL_F32 or FRL_BF16), read once
 *   p_lp     optional bf16 shadow weights [n] (written), NULL when the model runs in fp32
 *   grad_scale      host scalar multiplied into g (1/world_size for the DDP mean)
 *   grad_scale_dev  optional device scalar multiplied in as well (clip coefficient written
 *                   by frl_grad_sumsq_clip), NULL = 1
 * All arrays must be 16-byte aligned; n is arbitrary (scalar tail).
 * Hyper-parameters are doubles (Python floats): derived constants such as 1-beta2 or the
 * Adam bias corrections are formed in double and rounded to fp32 once, exactly as torch does
 * when it hands Python scalars to fp32 tensor ops.
 *   dyn      optional DEVICE array of per-step scalars that override the by-value arguments,
 *            so a CUDA graph that captured the launch stays valid while they change:
 *            SGD / RMSprop: dyn[0] = lr ;  Adam: dyn[0] = -lr/(1-beta1^t), dyn[1] = sqrt(1-beta2^t) ;
 *            AdamW: dyn[0] = -lr/(1-beta1^t), dyn[1] = sqrt(1-beta2^t), dyn[2] = 1-lr*wd.
 *            The block is 4 floats; a rule reads only its own slots.
 * Update rules are torch 2.11's: L2-coupled weight decay (g += wd * p first) for SGD, Adam and
 * RMSprop; decoupled weight decay (p *= 1-lr*wd first, g not decayed) for AdamW.
 * ---------------------------------------------------------------------------------------- */

/* SGD: buf = first_step ? g : mu*buf + (1-dampening)*g ; p -= lr*buf.   mu == 0: buf may be NULL. */
int frl_sgd_momentum(float* p, const void* g, float* buf, void* p_lp, int64_t n,
                     double lr, double mu, double dampening, double wd,
                     double grad_scale, const float* grad_scale_dev, const float* dyn,
                     int first_step, int g_dtype, void* stream);

/* Adam (coupled L2, optional amsgrad when vmax != NULL).  `step` is the 1-based step count
 * used for the bias corrections (computed in double on the host side of the call). */
int frl_adam(float* p, const void* g, float* m, float* v, float* vmax, void* p_lp, int64_t n,
             double lr, double beta1, double beta2, double eps, double wd, int64_t step,
             double grad_scale, const float* grad_scale_dev, const float* dyn, int g_dtype,
             void* stream);

/* AdamW = torch.optim.AdamW = Adam(decoupled_weight_decay=True): p *= 1-lr*wd (formed in double,
 * rounded to fp32 once), then the Adam update of the decayed p with the undecayed gradient.
 * Same arguments, state and traffic as frl_adam; `wd` is the decoupled coefficient. */
int frl_adamw(float* p, const void* g, float* m, float* v, float* vmax, void* p_lp, int64_t n,
              double lr, double beta1, double beta2, double eps, double wd, int64_t step,
              double grad_scale, const float* grad_scale_dev, const float* dyn, int g_dtype,
              void* stream);

/* RMSprop (not centered): sq = alpha*sq + (1-alpha)*g^2 ; avg = sqrt(sq)+eps ;
 * mu > 0: buf = mu*buf + g/avg ; p -= lr*buf     else: p -= lr*g/avg  (buf may be NULL). */
int frl_rmsprop(float* p, const void* g, float* sq, float* buf, void* p_lp, int64_t n,
                double lr, double alpha, double eps, double wd, double mu,
                double grad_scale, const float* grad_scale_dev, const float* dyn, int g_dtype,
             void* stream);

/* ------------------------------------------------------------------------------------------
 * K2-mt / K1 — multi-tensor forms of the update and the bucket flatten.
 * Replaces the DDP reducer's per-tensor bucket copy-in / copy-out (reference solver.py:287-289 ->
 * torch Reducer) for parameters whose gradients autograd allocates itself (convolutions,
 * normalisation layers): a SEGMENT TABLE in device memory names, per parameter tensor, where its
 * gradient lies, its dtype, its arena offset (a multiple of 8 elements) and its length.
 *   tile_prefix_dev[s] = number of tiles of segments 0..s-1 (int64, n_segs + 1 entries), a tile
 *   being frl_mt_tile_elems() arena elements of ONE segment; n_tiles = tile_prefix_dev[n_segs];
 *   tile_seg_dev[t] = segment index of tile t (int32, n_tiles entries).
 *   Gradient pointers must be 16-byte aligned; tensors contiguous in the parameter's layout.
 * frl_flatten_grads : arena_grad[arena_off + i] = cast(g[i] * scale) for every segment, one launch.
 * frl_*_mt          : the K2 update of the listed segments reading g in place; p / state / p_lp
 *                     are the ARENA BASE pointers (offset 0), other arguments as in K2.
 * ---------------------------------------------------------------------------------------- */
typedef struct frl_grad_seg {
    const void* g;          /* device pointer of the gradient tensor (g_dtype elements) */
    int64_t     arena_off;  /* first arena element of the parameter */
    int64_t     numel;      /* elements of the parameter */
    int32_t     g_dtype;    /* FRL_F32 | FRL_BF16 */
    int32_t     _pad;
} frl_grad_seg;

int64_t frl_mt_tile_elems(void);

int frl_flatten_grads(const frl_grad_seg* segs_dev, const int64_t* tile_prefix_dev,
                      const int32_t* tile_seg_dev, int64_t n_tiles, void* arena_grad, int dst_dtype,
                      double scale, void* stream);

int frl_sgd_momentum_mt(float* p, float* buf, void* p_lp, const frl_grad_seg* segs_dev,
                        const int64_t* tile_prefix_dev, const int32_t* tile_seg_dev, int64_t n_tiles,
                        double lr, double mu, double dampening, double wd, double grad_scale,
                        const float* grad_scale_dev, const float* dyn, int first_step, void* stream);

int frl_adam_mt(float* p, float* m, float* v, float* vmax, void* p_lp, const frl_grad_seg* segs_dev,
                const int64_t* tile_prefix_dev, const int32_t* tile_seg_dev, int64_t n_tiles, double lr, double beta1,
                double beta2, double eps, double wd, int64_t step, double grad_scale,
                const float* grad_scale_dev, const float* dyn, void* stream);

int frl_adamw_mt(float* p, float* m, float* v, float* vmax, void* p_lp, const frl_grad_seg* segs_dev,
                 const int64_t* tile_prefix_dev, const int32_t* tile_seg_dev, int64_t n_tiles, double lr, double beta1,
                 double beta2, double eps, double wd, int64_t step, double grad_scale,
                 const float* grad_scale_dev, const float* dyn, void* stream);

int frl_rmsprop_mt(float* p, float* sq, float* buf, void* p_lp, const frl_grad_seg* segs_dev,
                   const int64_t* tile_prefix_dev, const int32_t* tile_seg_dev, int64_t n_tiles, double lr, double alpha,
                   double eps, double wd, double mu, double grad_scale, const float* grad_scale_dev,
                   const float* dyn, void* stream);

/* ------------------------------------------------------------------------------------------
 * K3 — global gradient norm for clipping.
 * Replaces torch.nn.utils.clip_grad_norm_ (reference solver_worker.py:588-591): one pass
 * over the model-parameter range of the gradient arena.
 *   out[0] = sum(g^2) * pre_scale^2,  out[1] = sqrt(out[0]),
 *   out[2] = min(1, max_norm / (out[1] + 1e-6))   (the coefficient K2 reads)
 * scratch: >= frl_reduce_scratch_floats() floats + 1 uint32 ticket, zero-initialised once.
 * Deterministic: fixed-order two-stage reduction.
 * ---------------------------------------------------------------------------------------- */
int64_t frl_reduce_scratch_bytes(void);
int frl_grad_sumsq_clip(const void* g, int64_t n, int g_dtype, float pre_scale, float max_norm,
                        float* out3, void* scratch, void* stream);

/* ------------------------------------------------------------------------------------------
 * K4 — fused multitask criterion.
 * Replaces ParallelCriterion.compute_split_loss/forward (reference criteria.py:42-61), the
 * nn.MSELoss / nn.CrossEntropyLoss kernels underneath, MaskedLoss's gather
 * (criteria.py:267-287) and the isnan()/item() syncs of the loop (solver_worker.py:486-487,
 * 569).
 * ---------------------------------------------------------------------------------------- */
#define FRL_MAX_TASKS 8
enum { FRL_LOSS_MSE = 0, FRL_LOSS_CE = 1 };

typedef struct frl_task_desc {
    int32_t     kind;         /* FRL_LOSS_MSE | FRL_LOSS_CE */
    int32_t     out_dtype;    /* FRL_F32 | FRL_BF16 : dtype of `out` (and of `dout`) */
    int32_t     tgt_dtype;    /* MSE: FRL_F32 | FRL_BF16 ; CE: FRL_I64 */
    int32_t     ignore_index; /* CE only (torch default -100) */
    const void* out;          /* model output  [rows, cols] row-major contiguous */
    const void* tgt;          /* MSE: [rows, cols] ; CE: int64 class index [rows] */
    const uint8_t* mask;      /* optional (MaskedLoss): nonzero = use ; numel = rows*cols/mask_inner */
    void*       dout;         /* backward only: gradient wrt out, same shape/dtype as out */
    int64_t     rows;
    int64_t     cols;
    int64_t     mask_inner;   /* elements of `out` covered by one mask entry (1 or cols ...) */
    float       weight;       /* loss weight w_i */
    float       _pad;
} frl_task_desc;

/* scratch bytes for T tasks (partials + ticket); zero-initialise once */
int64_t frl_criteria_scratch_bytes(int n_tasks);

/* forward: losses[0] = sum_i w_i*L_i (left-to-right), losses[1+i] = w_i*L_i.
 *   aux[i]      = 1/count_i (0 if nothing selected) for the backward
 *   lse[...]    = per-row log-sum-exp of every CE task, rows concatenated in task order
 *   sink_mapped = optional second destination of losses[0..T] (e.g. a row of a pinned loss
 *                 log), nan_flag_mapped = optional int set to 1 when losses[0] is NaN. */
int frl_criteria_forward(const frl_task_desc* tasks_host, int n_tasks,
                         float* losses, float* aux, float* lse,
                         float* sink_mapped, int32_t* nan_flag_mapped,
                         void* scratch, void* stream);

/* backward: dout_i = (gl[0] + gl[1+i]) * w_i * dL_i/dout_i, gl = gradient wrt losses[0..T]
 * (device, fp32 [1+T]); reads aux / lse written by the forward. */
int frl_criteria_backward(const frl_task_desc* tasks_host, int n_tasks,
                          const float* grad_losses, const float* aux, const float* lse,
                          void* stream);

/* ------------------------------------------------------------------------------------------
 * K5 — device-side batch preprocessing.
 * Batched replacement of the per-sample MultifieldTransform arithmetic (reference
 * transform.py:25-38, multitask_problem.py:56-71): dst = (src * scale[c] + bias[c]), with
 * c = (i / inner) % channels, converting FRL_U8|FRL_F32|FRL_BF16 -> FRL_F32|FRL_BF16.
 * scale/bias: device fp32 [channels]; NULL scale = 1, NULL bias = 0.
 * ---------------------------------------------------------------------------------------- */
int frl_preproc_affine(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n,
                       int64_t inner, int64_t channels, const float* scale, const float* bias,
                       void* stream);

/* dtype conversion / scaled copy used by the arena (master -> shadow refresh after a
 * checkpoint load, gradient flatten for modules the arena cannot write into directly):
 * dst = src * scale. */
int frl_cast_scale(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n,
                   float scale, void* stream);

/* ------------------------------------------------------------------------------------------
 * K6 — column sum: out[c] (+)= sum_r x[r, c], x row-major [rows, cols].
 * The bias gradient of a linear layer, written straight into the gradient arena; replaces the
 * generic reduction autograd runs inside `total_loss.backward()` (reference
 * solver_worker.py:586).  accumulate != 0 adds to `out` (a layer applied twice in one step).
 * scratch: frl_colsum_scratch_bytes(rows, cols) bytes, zero-initialised once; deterministic.
 * ---------------------------------------------------------------------------------------- */
int64_t frl_colsum_scratch_bytes(int64_t rows, int64_t cols);
int frl_colsum(const void* x, int x_dtype, int64_t rows, int64_t cols, void* out, int out_dtype,
               int accumulate, void* scratch, void* stream);
/* K6b — the same pass with ReLU's backward folded in, for a Linear+ReLU pair: dz[r,c] =
 * act[r,c] > 0 ? dy[r,c] : 0 (act = the layer's forward output; dy, act, dz share dtype and the
 * [rows, cols] layout; dz may alias dy) and out[c] (+)= sum_r dz[r,c].  Replaces autograd's
 * threshold_backward kernel plus the bias-gradient reduction (reference solver_worker.py:586). */
int frl_drelu_colsum(const void* dy, const void* act, void* dz, int dtype, int64_t rows, int64_t cols,
                     void* out, int out_dtype, int accumulate, void* scratch, void* stream);

/* ------------------------------------------------------------------------------------------
 * K7 — fused gradient all-reduce + optimizer update + weight broadcast over NVSwitch multicast
 * (world_size > 1).  Replaces, per gradient bucket, the DDP reducer's ncclAllReduce
 * (reference solver.py:287-289, run inside solver_worker.py:586) AND optimizer.step()
 * (solver_worker.py:592) with one kernel: barrier | g = multimem.ld_reduce over all ranks'
 * bucket copies | update this rank's 1/world shard | multimem.st the new weights into every
 * replica | barrier.
 *
 *   p, state...        LOCAL fp32 master / optimizer-state slices of the bucket [n]
 *   mc_g               MULTICAST address of the bucket's gradient slice (symmetric allocation)
 *   mc_out             MULTICAST address of the slice every rank's module reads its weights
 *                      from: bf16 shadow weights (g_dtype FRL_BF16) or the fp32 master
 *                      (g_dtype FRL_F32, where p is that same memory, locally addressed)
 *   signal_pads_dev    device array [world] of pointers to each rank's uint32 signal pad;
 *                      slots [pad_base, pad_base + 64) are used
 *   local_scratch      rank-local uint32[8 + max_blocks], zero-initialised once
 *   max_blocks         grid size (1..1024; with in-kernel barriers all blocks must be co-resident)
 *   flags              0: the kernel carries both barriers itself.
 *                      FRL_NVLS_EXTERNAL_SYNC: no barrier inside; the caller issues, on the same
 *                      stream, frl_nvls_barrier(slot 0) before and frl_nvls_barrier(slot 1) after.
 *                      A rank that waits for slower peers then holds one warp instead of a grid
 *                      of spinning CTAs (which would keep its own backward GEMMs off the SMs).
 * n must be a multiple of 8; launch order must be identical on all ranks.
 * ---------------------------------------------------------------------------------------- */
enum { FRL_NVLS_EXTERNAL_SYNC = 1 };
/* 1-CTA cross-GPU rendezvous over the signal pads (slots [32*pad_slot, 32*pad_slot + world)). */
int frl_nvls_barrier(void* const* signal_pads_dev, int rank, int world, int pad_slot, void* stream);
int frl_nvls_sgd(float* p, float* buf, const void* mc_g, void* mc_out, int64_t n, int rank,
                 int world, void* const* signal_pads_dev, int pad_base, void* local_scratch,
                 int max_blocks, double lr, double mu, double dampening, double wd, double grad_scale,
                 const float* dyn, int first_step, int g_dtype, int flags, void* stream);
int frl_nvls_adam(float* p, float* m, float* v, float* vmax, const void* mc_g, void* mc_out,
                  int64_t n, int rank, int world, void* const* signal_pads_dev, int pad_base,
                  void* local_scratch, int max_blocks, double lr, double beta1, double beta2,
                  double eps, double wd,
                  int64_t step, double grad_scale, const float* dyn, int g_dtype, int flags, void* stream);
int frl_nvls_adamw(float* p, float* m, float* v, float* vmax, const void* mc_g, void* mc_out,
                   int64_t n, int rank, int world, void* const* signal_pads_dev, int pad_base,
                   void* local_scratch, int max_blocks, double lr, double beta1, double beta2,
                   double eps, double wd,
                   int64_t step, double grad_scale, const float* dyn, int g_dtype, int flags, void* stream);
int frl_nvls_rmsprop(float* p, float* sq, float* buf, const void* mc_g, void* mc_out, int64_t n,
                     int rank, int world, void* const* signal_pads_dev, int pad_base,
                     void* local_scratch, int max_blocks, double lr, double alpha, double eps,
                     double wd, double mu,
                     double grad_scale, const float* dyn, int g_dtype, int flags, void* stream);

/* ------------------------------------------------------------------------------------------
 * K8 — gather the rows of a minibatch from a pinned, device-mapped host dataset into HBM:
 * dst[i, :] = src[idx[i], :].  Replaces the per-sample __getitem__/collate/H2D sequence of the
 * loop (reference solver_worker.py:462-469): the kernel's PCIe reads are the transfer.
 * src_mapped: host pointer valid on the device (cudaHostAlloc / torch pin_memory); idx_dev:
 * int64 [n_rows] (device or mapped).  Rows that are multiples of 16 bytes take the wide path,
 * narrower rows (labels) an element-wise one.  max_blocks <= 0 -> 64 CTAs.
 * ---------------------------------------------------------------------------------------- */
int frl_gather_rows(const void* src_mapped, int64_t src_rows, const int64_t* idx_dev, void* dst,
                    int64_t n_rows, int64_t row_bytes, int max_blocks, void* stream);
/* K8w — rows of a window of retained minibatches (device tensors that are NOT contiguous with
 * one another): window row w lives in batch b at row w - sum(batch_rows[:b]).  dst[i, :] = that
 * row for w = idx_dev[i]; rows whose index is outside the window are left untouched.  Replaces
 * the per-sample slicing of retained minibatches in the loop's SamplerState (reference
 * solver_worker.py:254-262, 321-351: random picks and the worst-k heap keep data[i] slices)
 * where the indices only exist on the device.  batch_ptrs / batch_rows are HOST arrays (copied
 * into the kernel's parameter block, 64 batches per launch); idx_dev int64 [n_rows] on the device. */
int frl_gather_window_rows(const void* const* batch_ptrs, const int64_t* batch_rows, int n_batches,
                           const int64_t* idx_dev, void* dst, int64_t n_rows, int64_t row_bytes,
                           void* stream);
/* Same contract, moved by the SMs' bulk-copy engine (cp.async.bulk: host -> shared memory -> HBM,
 * one elected thread per CTA, 8 x 16 KB stages in flight).  Rows and pointers must be multiples
 * of 16 bytes.  max_blocks <= 0 -> one CTA per SM. */
int frl_gather_rows_tma(const void* src_mapped, int64_t src_rows, const int64_t* idx_dev, void* dst,
                        int64_t n_rows, int64_t row_bytes, int max_blocks, void* stream);

/* ------------------------------------------------------------------------------------------
 * Host gather pool — the host half of the input path (no CUDA calls inside).
 * Replaces the reference's per-sample __getitem__ + transform + default_collate on the host
 * (reference solver_worker.py:805-832, transform.py:25-38) with native worker threads that copy
 * the raw rows of a minibatch, dst[i, :] = src[idx[i], :], into a pinned staging buffer with
 * non-temporal stores; the caller then moves the staging buffer to HBM with one DMA and runs the
 * per-sample arithmetic on the device (K5).
 *   create(n_threads)            -> pool or NULL (frl_last_error)
 *   submit(...)                  -> ticket >= 1, or a negative FRL_E_* code; returns immediately;
 *                                   idx is copied, src/dst must stay valid until the job completes;
 *                                   an index outside [0, src_rows) rejects the whole job
 *   wait(pool, ticket)           -> blocks until every job up to and including `ticket` is done
 *                                   and its stores are globally visible (sfence)
 * Thread-safe; jobs run FIFO.
 * ---------------------------------------------------------------------------------------- */
typedef struct frl_gather_pool frl_gather_pool;
frl_gather_pool* frl_gather_pool_create(int n_threads);
void frl_gather_pool_destroy(frl_gather_pool* pool);
int frl_gather_pool_threads(const frl_gather_pool* pool);
int64_t frl_gather_pool_submit(frl_gather_pool* pool, const void* src_host, int64_t src_rows,
                               const int64_t* idx_host, void* dst_host, int64_t n_rows,
                               int64_t row_bytes);
/* Same gather with the PCIe hop in bf16: src rows are fp32 [row_elems], dst rows bf16 [row_elems],
 * converted round-to-nearest-even (NaN -> quiet NaN), bit-identical to the device cast, while the
 * worker threads touch the bytes anyway.  Halves the H2D payload of a bf16-compute run. */
int64_t frl_gather_pool_submit_f32_to_bf16(frl_gather_pool* pool, const void* src_host,
                                           int64_t src_rows, const int64_t* idx_host, void* dst_host,
                                           int64_t n_rows, int64_t row_elems);
int frl_gather_pool_wait(frl_gather_pool* pool, int64_t ticket);

#ifdef __cplusplus
}
#endif
#endif /* FRL_B200_H */
