/*
 * distrifuser_b200 -- C ABI of the B200-native patch-parallel UNet hot path.
 *
 * The reference (mit-han-lab/distrifuser) has no FFI: its "plugin API" is Python class substitution
 * (distrifuser/models/distri_sdxl_unet_pp.py:18-40).  Each entry point below replaces the torch / NCCL
 * call sites of one reference function; the Python classes of the same names as the reference's
 * (distrifuser_b200/*.py) are thin shims over these calls.  INTEGRATION.md shows the binding a reference
 * maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; df_last_error() gives the message
 *     (thread-local).  Nothing here owns or frees caller memory except df_symm_alloc/df_symm_free.
 *   - all pointers are DEVICE pointers unless the name ends in _host; `stream` is a cudaStream_t.
 *   - no entry point synchronises the host or allocates device memory (graph-capturable), except the
 *     df_symm_* / df_tensormap_* set-up calls.
 *   - activations are fp16, NHWC ("channels_last") for 4-D tensors, [b, tokens, C] for sequences.
 *
 * Symmetric arena layout (one per rank, mapped into every peer with CUDA IPC):
 *   bank k in [0, DF_NBANKS): byte offset k * bank_stride; inside a bank every registered tensor has
 *   one source slot per patch-group member: slot(k, idx, src) = base + k*bank_stride + tensor_off[idx] + src*slot_bytes[idx].
 *   Epoch e (one per UNet call) publishes into bank e % DF_NBANKS and stamps flags[idx*world + src] = e
 *   on the destination rank.  The epoch clock lives in device memory so captured CUDA graphs replay.
 */
#ifndef DISTRIFUSER_B200_H
#define DISTRIFUSER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DF_NBANKS 3
#define DF_MAX_WORLD 8
#define DF_IPC_HANDLE_BYTES 64
#define DF_TENSORMAP_BYTES 128
#define DF_AR_RING 2               /* depth of the all-reduce slot ring of the tensor-parallel path */

/* ---- errors / info ------------------------------------------------------------------------------ */
const char* df_last_error(void);
int df_version(void);                       /* ABI version, currently 2 */
int df_device_sm_count(int* out);

/* ---- symmetric memory: replaces the flat NCCL buffers of PatchParallelismCommManager.create_buffer
 *      (distrifuser/utils.py:151-164) ------------------------------------------------------------- */
int df_symm_alloc(size_t bytes, void** dptr, void* ipc_handle_out_host /* DF_IPC_HANDLE_BYTES */);
int df_symm_open(const void* ipc_handle_host, void** peer_dptr);
int df_symm_close(void* peer_dptr);
int df_symm_free(void* dptr);

/* Communicator descriptor, filled by the host shim and passed BY VALUE to the kernels.  A communicator describes
 * one GROUP of ranks and indexes its members 0..world-1: the host builds one for the patch group (the ranks that share a
 * CFG branch: K/V, halo and GroupNorm traffic) and one for the whole world (final epsilon gather); both point into the
 * same arenas but use separate flag regions.  Every "rank" / mask bit below is an index inside the communicator. */
typedef struct {
  void* base[DF_MAX_WORLD];        /* arena base of every member, as mapped in THIS process (own = local)  */
  uint32_t* flags[DF_MAX_WORLD];   /* flag array of every member (inside its arena): flags[idx*world+src]  */
  uint32_t* clock;                 /* this rank's epoch clock: [0]=publish, [1]=read, [2]=output epoch     */
  uint32_t* tickets;               /* this rank's per-tensor CTA ticket counters (local scratch, zeroed)   */
  uint64_t bank_stride;            /* bytes between banks                                                   */
  uint64_t spin_timeout_ns;        /* device-side flag waits trap after this long (0 = default 30 s)       */
  int32_t world;                   /* members in this communicator                                          */
  int32_t rank;                    /* this rank's index in the communicator                                 */
} df_comm_t;

/* ---- epoch clock: replaces the host-side counter / handle bookkeeping of the comm manager
 *      (distrifuser/utils.py:170-199).  kind: 0 = synchronous step (read what is published this step),
 *      1 = asynchronous step (read previous epoch, publish a new one), 2 = frozen (no_sync after warm-up:
 *      neither advances).  One thread, one launch per UNet call. ---------------------------------- */
int df_step_begin(uint32_t* clock, int kind, void* stream);

/* ---- activation publication: replaces enqueue()+batched async all_gather (utils.py:170-190) and the
 *      blocking all_gather of synchronous steps (attn.py:133).  Copies `rows` rows of `row_bytes` bytes
 *      (source pitch `src_pitch`) into slot(pub%NB, idx, src=comm.rank) of every rank in `peer_mask`
 *      (bit i = member i of the communicator; may include comm.rank itself) and then stamps their flags with
 *      the pub epoch (release, system scope).  rows > 1 publishes a strided [rows, row_bytes] view. ------- */
int df_slot_publish(df_comm_t comm, const void* src, uint64_t rows, uint64_t row_bytes, uint64_t src_pitch,
                    uint64_t tensor_off, uint64_t slot_bytes, int idx, uint32_t peer_mask, int num_ctas,
                    void* stream);

/* Blocks the stream until flags[idx][s] >= read epoch for every s in src_mask (acquire, system scope).
 * Replaces handle.wait() (attn.py:179-182, conv2d.py:46-49, groupnorm.py:19-22). */
int df_slot_wait(df_comm_t comm, int idx, uint32_t src_mask, void* stream);

/* ---- GroupNorm with exchanged sufficient statistics: replaces DistriGroupNorm.forward
 *      (distrifuser/modules/pp/groupnorm.py:14-97).  x,y: [b,h,w,C] NHWC fp16.
 *      mode: 0 local statistics only (n==1, or separate_gn/no_sync after warm-up, groupnorm.py:92-93)
 *            1 synchronous exchange   (groupnorm.py:45-47 and :74-80)
 *            2 corrected_async_gn     (groupnorm.py:49-51,60-63)
 *            3 stale_gn               (groupnorm.py:52-55)
 *      bessel != 0 multiplies the variance by ne/(ne-1) with the LOCAL element count (groupnorm.py:65-66);
 *      neg_var_fallback != 0 replaces negative variance by the local variance (groupnorm.py:60-63).
 *      group_mask selects the patch-group members (bit i = group rank i); stats slots hold 2*b*G fp32
 *      (mean, mean of squares).  `scratch` >= df_groupnorm_scratch_bytes(). ---------------------------- */
size_t df_groupnorm_scratch_bytes(int b, int groups, int h, int w, int C);
/* `addend` (nullable): [b, C] fp16 (row pitch `addend_pitch` elements, 0 = C) added to every pixel before the statistics and the normalisation, i.e. the
 * kernel computes GroupNorm(x + addend[:, :, None, None]) -- ResnetBlock2D's time-embedding add, fused.
 * `scratch` must be zero-filled once when it is allocated (it carries a self-resetting CTA ticket). */
int df_groupnorm_fwd(df_comm_t comm, const void* x, const void* addend, int64_t addend_pitch, void* y, const void* gamma, const void* beta,
                     int b, int h, int w, int C, int groups, float eps, int mode, int bessel,
                     int neg_var_fallback, int fuse_silu, int idx, uint64_t tensor_off, uint64_t slot_bytes,
                     uint32_t group_mask, void* scratch, void* stream);

/* GroupNorm -> (SiLU) -> 3x3 conv in one pass over the activation (the ResnetBlock2D / conv_norm_out pattern): like
 * df_groupnorm_fwd, but y_padded is [b, h+2, w, C]; the normalised rows go to rows 1..h, this rank's first / last output rows
 * are also stored into the patch neighbours' slots of the CONV's comm tensor `halo_idx` (when push != 0; replaces
 * df_halo_push) and rows 0 / h+1 are filled from the neighbours' slots of the read epoch, zeros at the image border (replaces
 * df_halo_assemble and its copy of the whole activation; distrifuser/modules/pp/conv2d.py:72-93).  comm must be the patch
 * group even when the statistics mode is 0. */
int df_groupnorm_halo_fwd(df_comm_t comm, const void* x, const void* addend, int64_t addend_pitch, void* y_padded, const void* gamma, const void* beta,
                          int b, int h, int w, int C, int groups, float eps, int mode, int bessel, int neg_var_fallback,
                          int fuse_silu, int idx, uint64_t tensor_off, uint64_t slot_bytes, uint32_t group_mask, void* scratch,
                          int halo_idx, uint64_t halo_off, uint64_t halo_slot_bytes, int up_rank, int down_rank, int push,
                          int wait_flags, void* stream);

/* ---- conv halo exchange: replaces the boundary stack + all_gather + cat/pad of DistriConv2dPP.forward
 *      (distrifuser/modules/pp/conv2d.py:72-93).  x: [b,h,w,C] NHWC fp16, one halo row (padding 1).
 *      df_halo_push sends x's first row to patch-neighbour `up_rank` (its bottom halo) and x's last row to
 *      `down_rank` (its top halo); a rank of -1 means image border.  df_halo_assemble builds
 *      xp[b,h+2,w,C] = [halo from up | x | halo from down] reading the read-epoch bank (zero rows at the
 *      border) after waiting for the neighbours' flags. ------------------------------------------ */
int df_halo_push(df_comm_t comm, const void* x, int b, int h, int w, int C, int idx, uint64_t tensor_off,
                 uint64_t slot_bytes, int up_rank, int down_rank, void* stream);
int df_halo_assemble(df_comm_t comm, const void* x, void* xp, int b, int h, int w, int C, int idx,
                     uint64_t tensor_off, uint64_t slot_bytes, int up_rank, int down_rank, int wait_flags,
                     void* stream);

/* ---- fused multi-head attention over per-rank K/V segments: replaces torch.cat(full_kv)+split+SDPA of
 *      DistriSelfAttentionPP._forward (distrifuser/modules/pp/attn.py:127-153) and the SDPA of
 *      DistriCrossAttentionPP.forward (attn.py:79-87).
 *      q:[b,lq,heads*d] fp16 (row pitch q_pitch elements); out same shape (pitch o_pitch).
 *      K/V live in `nseg` segments, each [b, lseg, 2*heads*d] (K at column h*d, V at heads*d + h*d).
 *      Segment `own_seg` is read from kv_own (this step's fresh projection, pitch kv_pitch elements); every
 *      other segment s is read from the arena slot(read%NB, idx, src=seg_rank[s]) through the tensor maps
 *      prepared by df_attn_make_kvmaps.  wait_flags != 0 makes the kernel wait for the peers' flags itself.
 *      d: any multiple of 8 up to 192 (SDXL 64; SD1.x 40 / 80 / 160), zero-padded to 64-column blocks by TMA;
 *      softmax scale is 1/sqrt(d) unless scale > 0. ------------------------------------------------- */
int df_attn_make_kvmaps(df_comm_t comm, uint64_t tensor_off, uint64_t slot_bytes, int b, int lseg, int heads,
                        int d, void* maps_out /* device, DF_NBANKS*world*DF_TENSORMAP_BYTES */, void* stream);
/* Scratch of a launch: df_attn_workspace_bytes() bytes, ZERO-INITIALISED ONCE by the caller and then reusable by any number of
 * stream-ordered launches (every counter in it resets itself).  It holds the ticket counter from which the persistent CTAs
 * of a grid that fills the SMs draw their work units and, for small grids (short per-rank Q at n >= 2), the fp32 partials and
 * arrival tickets of units whose K/V range is cut over several CTAs (merged in-kernel by the last part to arrive).  Passing a
 * null / too small workspace is legal: every CTA then walks a static list of whole units. */
size_t df_attn_workspace_bytes(int b, int lq, int lseg, int nseg, int heads, int d);
int df_attn_fwd(df_comm_t comm, const void* q, const void* kv_own, void* out, const void* kvmaps,
                int b, int lq, int lseg, int heads, int d, int64_t q_pitch, int64_t kv_pitch, int64_t o_pitch,
                int nseg, int own_seg, const int32_t* seg_rank_host, int idx, int wait_flags, float scale,
                void* workspace, size_t workspace_bytes, void* stream);

/* ---- final epsilon gather: replaces the blocking world all_gather + cat(dim=2) at the end of
 *      DistriUNetPP.forward (distrifuser/models/distri_sdxl_unet_pp.py:162-169,186-193).
 *      strip: this rank's [bs,C,hs,W] NCHW fp16 output; it is written into slot(pub%NB, idx, 0) of every
 *      world rank at batch offset `batch0`, row offset `row0` of a [B,C,H,W] image, then every rank waits for
 *      all `world` flags and copies the assembled image to `out`. ---------------------------------- */
int df_output_gather(df_comm_t comm, const void* strip, void* out, int B, int C, int H, int W, int bs, int hs,
                     int batch0, int row0, int idx, uint64_t tensor_off, void* stream);

/* ---- fused GEGLU gate of the transformer feed-forward: out[r, c] = in[r, c] * gelu_erf(in[r, cols + c]).
 *      Not one of the reference's wrapped modules (diffusers FeedForward, SURVEY Appendix A) but on the per-step
 *      path inside DistriUNetPP.forward; in:[rows, 2*cols] fp16 (pitch in_pitch elements), out:[rows, cols]. ---- */
int df_geglu(const void* in, void* out, int64_t rows, int cols, int64_t in_pitch, int64_t out_pitch, void* stream);

/* ---- out = a + bias[c] (+ residual) on NHWC fp16 activations [rows = b*h*w, C], in one pass (out may alias a).
 *      Replaces the broadcast bias `add_` that torch runs after every cudnn_convolution (F.conv2d, used by
 *      distrifuser/modules/pp/conv2d.py:41,110) and the residual add of diffusers' ResnetBlock2D.forward. -------------- */
int df_bias_residual_add(const void* a, const void* residual /* nullable */, const void* bias, void* out, int64_t rows, int C,
                         void* stream);

/* ---- fused residual add + LayerNorm of BasicTransformerBlock: s = x + r (fp16, written to s_out when non-null; r may
 *      be null = plain LayerNorm), y = LayerNorm(s) * gamma + beta.  x, r, s_out, y: [rows, C] contiguous fp16. ---- */
int df_add_layernorm(const void* x, const void* r, void* s_out, void* y, const void* gamma, const void* beta,
                     int64_t rows, int C, float eps, void* stream);

/* ---- Linear layers of the transformer blocks as a tcgen05 GEMM with fused epilogues (SURVEY 8f N1; reference call sites
 *      distrifuser/modules/pp/attn.py:121-125,159 and the diffusers FeedForward between the wrappers):
 *        out[M,N] = a[M,K] . w[N,K]^T (+ bias[N]) (+ residual[M,N])                         epilogue 0
 *        out[M,N/2] = (a.Wh^T + bh) * gelu_erf(a.Wg^T + bg), rows of w (and bias) interleaved in blocks of
 *                     80 or 128 (df_linear_geglu_block): [hidden block t | gate block t]  (diffusers GEGLU without its [M,8C] intermediate)   epilogue 1
 *      All matrices fp16 row-major with pitches lda / ldw / ldr / ldo in elements; N % 8 == 0, K % 64 == 0 (GEGLU: N % 160 == 0 or N % 256 == 0):
 *      df_linear_supported() tells; unsupported shapes stay library calls.
 *      publish != 0 (epilogue 0 only): the columns >= pub_col0 are ALSO stored into slot(pub % NB, idx, src = comm.rank) of every
 *      member in peer_mask, row-major [M, N - pub_col0], and the peers' flags are stamped with the publish epoch -- the k|v
 *      half of the fused q|k|v projection goes straight into the peers' arenas (replaces enqueue, utils.py:181-190).
 *      max_ctas: 0 = all SMs. ------------------------------------------------------------------------------- */
int df_linear_supported(int64_t M, int N, int K, int epilogue);
/* rows per hidden / gate block of the interleaved GEGLU weight for this problem (80 or 128 = half the pair-tile width the
 * kernel will use); pass the same value as `geglu_block` (0 = let the kernel pick, must then match the interleave). */
int df_linear_geglu_block(int64_t M, int N, int K);
int df_linear_fwd(df_comm_t comm, const void* a, const void* w, const void* bias, const void* residual, void* out,
                  int64_t M, int N, int K, int64_t lda, int64_t ldw, int64_t ldr, int64_t ldo, int epilogue,
                  int geglu_block, int publish, int pub_col0, int idx, uint32_t peer_mask, uint64_t tensor_off,
                  uint64_t slot_bytes, int max_ctas, void* stream);

/* ---- tensor parallelism: fused all-reduce over peer memory.  Replaces the blocking dist.all_reduce + bias (+ residual)
 *      adds of the reference's tensor-parallel modules (distrifuser/modules/tp/attention.py:159, feed_forward.py:77,
 *      resnet.py:189, conv2d.py:52).
 *      out[rows, C] = sum over members s in contrib_mask of partial_s + bias[C] (+ residual), fp32 in member order 0..n-1,
 *      rounded to fp16 once: bit-identical on every member.  4-D NHWC tensors are passed as [b*h*w, C]; rows*C % 8 == 0.
 *      partial == NULL: this member contributes nothing (it owns no heads); its bit in contrib_mask must then be clear.
 *      One-shot: the partial goes to ring slot (seq % DF_AR_RING, src = comm.rank) of every peer, at arena offset
 *      ring_off + (ring*world + src)*ring_slot_bytes, and the peer's flag u32 at flags_off + 4*(ring*world + src) is stamped
 *      with seq = clock[0]*nsites + site (release, system scope); every member waits for all peers' flags (acquire) and
 *      reduces locally.  After each df_step_begin the sites must be issued in order 0..nsites-1 on one stream, so that
 *      consecutive all-reduces carry consecutive seq.  comm.tickets[ticket] is the CTA ticket.  comm.world == 1: no exchange.
 *      Never launched with programmatic dependent launch (the ring reuse relies on stream order). ------------- */
int df_allreduce_fwd(df_comm_t comm, const void* partial, void* out, int64_t rows, int C, const void* bias,
                     const void* residual, uint32_t contrib_mask, int site, int nsites, uint64_t ring_off,
                     uint64_t ring_slot_bytes, uint64_t flags_off, int ticket, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DISTRIFUSER_B200_H */
