/*
 * mot_b200.h -- C ABI of the B200-native byte-mix embedding path of
 * mixture-of-tokenizers (libmot_b200.so, sm_100a only).
 *
 * The reference has no FFI: the path is inline PyTorch module code.  Each entry
 * point below names the reference lines whose work it replaces (paths relative
 * to the reference checkout; "spt" = scaled-pre-train, "runs/N" =
 * modded-nanogpt/runs/N_mot-in_toks-valemb.py).  INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller; nothing is allocated
 *     or freed by the library; outputs, gradients and workspace are caller-provided;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no
 *     host synchronisation, no host reads of device data (CUDA-graph capturable);
 *   - return value: 0 = MOT_OK, otherwise an error code for mot_strerror();
 *   - token ids are int32; byte ids are int32 or int64 (MOT_F_IDS_I64);
 *   - tables, outputs and dense gradients share one element type (MotDesc.dtype);
 *   - tok_dim, byte_dim and out_dim must be multiples of 8 elements and all table /
 *     output pointers 16-byte aligned (128-bit accesses).
 */
#ifndef MOT_B200_H
#define MOT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MOT_B200_ABI_VERSION 7

/* ---- error codes ------------------------------------------------------- */
enum {
  MOT_OK = 0,
  MOT_ERR_BAD_ARG = 1,     /* null pointer / non-positive size / inconsistent dims   */
  MOT_ERR_UNSUPPORTED = 2, /* a reference option this library refuses (no fallback)  */
  MOT_ERR_MISALIGNED = 3,  /* pointer not 16-byte aligned / dim not a multiple of 8  */
  MOT_ERR_WORKSPACE = 4,   /* workspace smaller than mot_embed_workspace_bytes()     */
  MOT_ERR_CUDA = 5,        /* launch failed; see mot_last_cuda_error()               */
  MOT_ERR_NO_DEVICE = 6    /* no sm_100 device is current                            */
};

/* ---- element / id types ------------------------------------------------ */
enum { MOT_BF16 = 0, MOT_F32 = 1 };
/* storage of the ttb table: int16 (native), or the reference's float containers:
 * fp32 nn.Embedding (spt/data_creation.py:51-58) and the bf16-cast table of the
 * runs (runs/7:441) whose ids > 256 are rounded -- read back with truncation like
 * `.to(int64)` (spt/data_creation.py:63). */
enum { MOT_TTB_I16 = 0, MOT_TTB_F32 = 1, MOT_TTB_BF16 = 2 };

/* ---- how token and byte rows are combined (SURVEY.md 2.4) -------------- */
enum {
  MOT_ADD = 0,        /* z = u + concat_k(w_k)        tok_dim == bpt*byte_dim == out_dim (runs/71:228-230) */
  MOT_CONCAT = 1,     /* z = [u | concat_k(w_k)]      out_dim == tok_dim + bpt*byte_dim  (runs/711:224-232,
                         the A operand of the projection variants runs/7:226-234, spt/train_gpt.py:439-443) */
  MOT_TOK_ONLY = 2,   /* z = u                        (spt/train_gpt.py:342-348)          */
  MOT_BYTES_ONLY = 3, /* z = concat_k(w_k)            (runs/4_bytes-in_toks-valemb.py:313) */
  MOT_MEAN = 4        /* z = u + mean_k(w_k)          byte_dim == tok_dim (inference/inference.py:267) */
};

enum {
  MOT_F_TOK_NORM = 1 << 0,     /* u = lam_tok * rms_norm(E_tok[tok])          (runs/7:317)            */
  MOT_F_BYTE_NORM = 1 << 1,    /* w_k = lam_byte * rms_norm(E_byte[id_k])     (runs/7:318, over byte_dim) */
  MOT_F_OUT_NORM = 1 << 2,     /* out = rms_norm(z)                           (runs/71:230)           */
  MOT_F_BYTES_FIRST = 1 << 3,  /* MOT_CONCAT order [bytes | tok]              (mathblations/model.py:267) */
  MOT_F_SLOT_MAJOR = 1 << 4,   /* byte ids are [bpt, n_tokens] (runs/71:479 `.view(16,-1)`), else [n_tokens, bpt] */
  MOT_F_IDS_FROM_TTB = 1 << 5, /* no byte-id tensor: ids are read from the ttb table inside the kernel */
  MOT_F_TTB_SCRAMBLE = 1 << 6, /* with IDS_FROM_TTB: slot i of position s is flat byte i*seq_len + s of its
                                  row of seq_len tokens (the `.view(bpt,-1)` of runs/71:479)           */
  MOT_F_IDS_I64 = 1 << 7,      /* byte-id tensors hold int64 (spt), else int32 (runs)                  */
  MOT_F_HAS_LAMBDAS = 1 << 8,  /* lam[0] = lam_tok, lam[1] = lam_byte (runs/74:314-315)                */
  MOT_F_TTB_PULL_LEFT = 1 << 9, /* with IDS_FROM_TTB: the ids are the PULLED ids of pull_from_left (mot_pull) over rows of
                                  seq_len tokens (n_tokens % seq_len == 0, bpt <= 32, tok_vocab = the ttb table's rows
                                  also for MOT_BYTES_ONLY), pad_id / eot_id as there;
                                  with TTB_SCRAMBLE the scramble picks (token, slot) and the id comes from the pulled row */
  MOT_F_TTB_PULL_RIGHT = 1 << 10, /* the same rules with the pulled ids of pull_from_right (rows right-padded); not
                                     together with TTB_PULL_LEFT */
  MOT_F_TTB_NEXT_TOK = 1 << 11    /* with TTB_PULL_RIGHT only: row r has one more token, the lookahead, at
                                     tok[n_tokens + r] for r < n_tokens / seq_len (the loader's window of seq_len + 1
                                     tokens, whose last token the right pull of the row's end reads).  Only the pull
                                     reads this tail: the token gathers, the sort plan and the touched-rows bitmap see
                                     tok[0, n_tokens) */
};

typedef struct MotDesc {
  int32_t abi_version; /* MOT_B200_ABI_VERSION */
  int32_t dtype;       /* MOT_BF16 | MOT_F32 */
  int64_t n_tokens;    /* positions in this call (B*S) */
  int64_t seq_len;     /* tokens per row (only used by MOT_F_TTB_SCRAMBLE; n_tokens % seq_len == 0) */
  int32_t tok_vocab;   /* rows of E_tok  (50257) */
  int32_t byte_vocab;  /* rows of E_byte (458; 14 for mathblations digits) */
  int32_t bpt;         /* bytes (digits) per token, 1..32 */
  int32_t tok_dim;
  int32_t byte_dim;
  int32_t out_dim;
  int32_t combine;     /* MOT_ADD ... */
  int32_t flags;       /* MOT_F_* */
  int32_t ttb_dtype;   /* MOT_TTB_* (only with MOT_F_IDS_FROM_TTB) */
  float eps;           /* rms_norm eps; the reference uses torch's default, finfo(float32).eps */
  int64_t row_stride;  /* elements between consecutive rows of `out` (forward) / `grad_out` (backward); 0 = out_dim.
                          With col_offset it lets a call produce or consume a column slice of wider rows, e.g. the
                          token half of the [tok | bytes] operand next to mot_byte_pair_fwd's byte half. */
  int32_t col_offset;  /* first column of this call's slice inside those rows (multiple of 8) */
  int32_t dp_slabs;    /* 0 / 1: the backward runs in one piece.  n > 1: the caller will run it as n vocabulary slabs
                          (mot_embed_bwd_slab); only sizes the workspace (one fp32 slot per finer stream chunk) */
  int32_t pad_id;      /* with MOT_F_TTB_PULL_LEFT / _RIGHT: the pad byte (456) and the end-of-text byte (457) of the ttb table,
                          each in the int16 range */
  int32_t eot_id;
} MotDesc;

const char* mot_strerror(int rc);
int mot_abi_version(void);
/* cudaGetErrorString of the last failed launch on this thread ("" if none). */
const char* mot_last_cuda_error(void);
/* Number of kernels this library launched since load / since the last reset (process-wide). */
int64_t mot_launch_count(void);
void mot_launch_count_reset(void);
/* Measurement hook (bench.py): cudaEvent_t pairs recorded on the launch stream immediately around the
 * main forward kernel and the main backward kernel of the following calls; NULL disables a pair. */
void mot_profile_events(void* fwd_start, void* fwd_stop, void* bwd_start, void* bwd_stop);

/* Measurement hook (tools/trace_timeline.py): a device buffer of 64 x int64 per warp of the main forward / backward kernel
 * that receives %globaltimer stamps of the warp's phases.  Only libraries built with -DMOT_TRACE write it (the shipped
 * build compiles the stamps out); NULL disables. */
void mot_profile_trace(void* device_buffer);

/* tokens -> padded byte ids.
 * Replaces tokens_to_bytes (spt/data_creation.py:61-67, runs/7:444-450): gather ttb rows
 * and cast to integer.  out is [n, bpt] token-major, int64 when out_i64 != 0 else int32. */
int mot_ttb_expand(const int32_t* tok, int64_t n, const void* ttb, int32_t tok_vocab, int32_t bpt,
                   int32_t ttb_dtype, void* out, int32_t out_i64, void* stream);

/* ttb table build as an integer gather.  Replaces the loop body of create_ttb (modded-nanogpt/create_ttb.py:18-31):
 * row v = the FIRST min(bpt, len_v) character ids of token v (`chars[offs[v] .. offs[v+1])`, the ids byte_to_int
 * gives the characters of `encoding.decode([v])`), padded with pad_byte on the left (pad_left != 0) or on the right;
 * rows with is_eot[v] != 0 (string "<|endoftext|>", :20-22) are bpt copies of eot_byte.  is_eot may be NULL.
 * out: int16 [n_rows, bpt]. */
int mot_ttb_build(const int16_t* chars, const int32_t* offs, const uint8_t* is_eot, int32_t n_rows, int32_t bpt,
                  int32_t pad_left, int32_t pad_byte, int32_t eot_byte, int16_t* out, void* stream);

/* The same table under another (bpt, pad side): the scaled-pre-train files ttb_{16,18,20}_{left,right}_pad.json
 * (spt/train_gpt.py:665-672) are create_ttb of the same strings.  A row's characters are its non-pad entries in order
 * (first min(count, bpt_out) kept, as create_ttb.py:24); all-eot rows stay all-eot.  bpt_in, bpt_out <= 32; out != table. */
int mot_ttb_repad(const int16_t* table, int32_t n_rows, int32_t bpt_in, int32_t bpt_out, int32_t pad_left,
                  int32_t pad_byte, int32_t eot_byte, int16_t* out, void* stream);

/* uint16 shard tokens -> int32 ids on the device.  Replaces the host-side `.to(torch.int32)` of load_data_shard
 * (spt/train_gpt.py:640-648) so that the upload moves the shard's own 2 bytes per token.  Pointers 16-byte aligned. */
int mot_tokens_widen_u16(const void* tok_u16, int64_t n, int32_t* out, void* stream);

/* tokens -> padded digit ids, the arithmetic ttb analogue of mathblations (GenerateEquations.tokens_to_digits,
 * mathblations/data.py:92-109): decimal digits right-aligned in dpt slots, pad 13; op / eq / pad tokens -> 10 / 11 / 12
 * in the last slot.  tok int32 or int64 (tok_i64), out [n, dpt] int32 or int64 (out_i64). */
int mot_tokens_to_digits(const void* tok, int64_t n, int32_t tok_i64, int32_t dpt, int64_t op_token, int64_t eq_token,
                         int64_t pad_token, void* out, int32_t out_i64, void* stream);

/* Workspace needed by mot_embed_bwd for this descriptor (bytes, 256-aligned). */
size_t mot_embed_workspace_bytes(const MotDesc* d);

/* State of a caller-owned workspace, passed as `ws_flags`.
 *   MOT_WS_PLAN_READY : the workspace holds mot_embed_plan() for these tokens.
 *   MOT_WS_CLEAN      : the head of the workspace (histogram, byte-gradient accumulators) is all zero, which is the
 *                       state mot_embed_workspace_init() and every completed mot_embed_bwd() leave it in; a caller
 *                       that keeps one workspace per stream passes it from the second step on and saves a memset.
 *                       Without the flag the library clears what it needs itself.
 *   MOT_WS_PLAN_JOINED: (with MOT_WS_PLAN_READY) the plan ran on ANOTHER stream and this stream waited for its event
 *                       (mot_embed_plan_async + mot_stream_wait_event), i.e. it was complete before this call's kernels were
 *                       launched: the backward may then read the plan before its programmatic-launch wait, while the
 *                       previous kernel of this stream is still draining.  Never pass it when mot_embed_plan() ran on the
 *                       same stream right before the backward. */
enum { MOT_WS_PLAN_READY = 1, MOT_WS_CLEAN = 2, MOT_WS_PLAN_JOINED = 4 };
int mot_embed_workspace_init(const MotDesc* d, void* workspace, size_t ws_bytes, void* stream);

/* Fused forward: out[n_tokens, out_dim] =
 *   f_out( combine( lam_tok * f_tok(E_tok[tok]),  lam_byte * f_byte(E_byte[byte ids]) ) ).
 * Replaces the embedding + mixin lines of GPT.forward (runs/71:312-314 + mixin_bytes :228-230 and
 * every variant of SURVEY.md 2.4 without a dense projection; spt/train_gpt.py:342-379).  For the
 * projection variants it produces the A operand [tok | bytes] that mot_linear_* consumes.
 *   byte_ids : int32/int64, NULL with MOT_F_IDS_FROM_TTB (then `ttb` is used), ignored for TOK_ONLY
 *   lam      : device float[2] or NULL (== {1,1}) */
int mot_embed_fwd(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                  const void* E_tok, const void* E_byte, const float* lam, void* out, void* stream);

/* Extended forward.
 *   rstd_out : optional fp32 [n_tokens]; receives the reciprocal rms of every mixed row when MOT_F_OUT_NORM is set,
 *              i.e. what F.rms_norm's autograd node keeps (spt/train_gpt.py:172-173); with `out` it lets
 *              mot_embed_bwd_ex skip rebuilding the mixed row.
 *   addend   : optional dense [n_tokens, out_dim] rows (table dtype) added to the mixed row before the output norm:
 *              z = combine(...) + addend.  With MOT_TOK_ONLY this is `norm(token_embs + F.linear(byte_embs, byte_fc))`
 *              of runs/71051:226-229 (the product comes from mot_linear_fwd).  Not with split concat / strided rows. */
int mot_embed_fwd_ex(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                     const void* E_tok, const void* E_byte, const float* lam, const void* addend, void* out,
                     float* rstd_out, void* stream);

/* Sort plan for the backward (token ids only; reusable by every table gathered with `tok`). */
int mot_embed_plan(const MotDesc* d, const int32_t* tok, void* workspace, size_t ws_bytes, int32_t ws_flags,
                   void* stream);

/* The same plan on a second stream, beside the forward: records ev_fork on main_stream, makes side_stream wait for it,
 * runs the plan there and records ev_join; the stream that later runs mot_embed_bwd (MOT_WS_PLAN_READY) must wait for
 * ev_join first (mot_stream_wait_event).  Streams are cudaStream_t, events cudaEvent_t, all owned by the caller. */
int mot_embed_plan_async(const MotDesc* d, const int32_t* tok, void* workspace, size_t ws_bytes, int32_t ws_flags,
                         void* main_stream, void* side_stream, void* ev_fork, void* ev_join);
int mot_stream_wait_event(void* stream, void* event);

/* Fused backward: the autograd graph of the lines above (rms_norm bwd, split, and the two
 * embedding_dense_backward scatter-adds).  gE_tok [tok_vocab, tok_dim] and gE_byte
 * [byte_vocab, byte_dim] are DENSE and fully overwritten (rows never gathered get zeros), so a
 * caller can all-reduce / feed them to the optimizer exactly like the reference's param.grad.
 *   g_lam    : device float[2], overwritten (d lam_tok, d lam_byte), or NULL
 *   ws_flags : MOT_WS_* state of `workspace`; on return the workspace is MOT_WS_CLEAN again */
int mot_embed_bwd(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                  const void* E_tok, const void* E_byte, const float* lam, const void* grad_out,
                  void* gE_tok, void* gE_byte, float* g_lam, void* workspace, size_t ws_bytes,
                  int32_t ws_flags, void* stream);

/* Extended backward.
 *   out_saved / rstd_saved : the `out` and `rstd_out` of mot_embed_fwd_ex (both NULL = rebuild the mixed row).  For the
 *       MoT-sum variant (MOT_ADD + MOT_F_OUT_NORM only, runs/71) the backward then reads two rows per occurrence
 *       (grad_out and out, same position) instead of the token row plus bpt byte rows:
 *       dz = rstd*g - out*(rstd*mean(g.out)).  Other variants ignore them.  Same results within the rounding of `out`
 *       (bf16: one extra 2^-9 relative rounding inside the second term).
 *   addend / d_addend : the dense rows of mot_embed_fwd_ex and the buffer [n_tokens, out_dim] that receives their
 *       gradient d z (table dtype), which the caller feeds to mot_linear_bwd_* (runs/71051). */
int mot_embed_bwd_ex(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                     const void* E_tok, const void* E_byte, const float* lam, const void* addend,
                     const void* grad_out, const void* out_saved, const float* rstd_saved, void* gE_tok,
                     void* gE_byte, float* g_lam, void* d_addend, void* workspace, size_t ws_bytes, int32_t ws_flags,
                     void* stream);

/* The backward as `n_slabs` vocabulary slabs, so that the data-parallel exchange of slab k (mot_dp_exchange on a second
 * stream) runs beside the backward of slab k + 1 -- the overlap the reference gets from its asynchronous per-parameter
 * all-reduces (runs/7:697-711).  Call k = 0 .. n_slabs - 1 in order with the same arguments: call k writes rows
 * [row_lo, row_hi) = mot_embed_slab_rows(tok_vocab, k, n_slabs) of gE_tok (final when the call's kernels have run);
 * gE_byte and g_lam are final after the last call.  d->dp_slabs must equal n_slabs (workspace layout); calls k > 0 need
 * MOT_WS_PLAN_READY.  reserve_sms (0..16): SMs the launch leaves free for a concurrently running exchange kernel.
 * Only where mot_embed_bwd_uses_saved(d) holds (the MoT-sum variant with out_saved / rstd_saved); MOT_ERR_UNSUPPORTED
 * otherwise -- run mot_embed_bwd_ex and one exchange instead. */
int mot_embed_bwd_slab(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                       const void* E_tok, const void* E_byte, const float* lam, const void* grad_out,
                       const void* out_saved, const float* rstd_saved, void* gE_tok, void* gE_byte, float* g_lam,
                       void* workspace, size_t ws_bytes, int32_t ws_flags, int32_t slab, int32_t n_slabs,
                       int32_t reserve_sms, void* stream);
int mot_embed_slab_rows(int32_t tok_vocab, int32_t slab, int32_t n_slabs, int32_t* row_lo, int32_t* row_hi);

/* 1 when mot_embed_bwd_ex would use out_saved / rstd_saved for this descriptor (so a caller knows whether keeping
 * them pays), else 0: only the MoT-sum variant, widths 512 / 768 / 1024, and at most 4 positions per vocabulary row
 * (beyond that the token rows of the recompute kernel are L2 hits and it is the faster one). */
int mot_embed_bwd_uses_saved(const MotDesc* d);

/* ---- split residual (runs/71081:302-304,315, V3g) ----------------------------------------------------------------
 * One gather, three outputs ([n_tokens, out_dim] each, table dtype, 16-byte aligned):
 *   x0t = rms_norm(E_tok[tok]),  x0b = the per-byte-normed byte rows C'_n,  x = lam[0] * x0t + lam[1] * x0b,
 * every element bit-identical to the separate tok-only / bytes-only / MOT_ADD launches.  d must be the V3c descriptor:
 * MOT_ADD with MOT_F_TOK_NORM | MOT_F_BYTE_NORM | MOT_F_HAS_LAMBDAS, no MOT_F_OUT_NORM / MOT_F_TTB_PULL_RIGHT, no
 * row_stride / col_offset / dp_slabs (else MOT_ERR_BAD_ARG); ids explicit, or from the ttb table (scramble, left pull).
 * out_dim 512 or 1024 (else MOT_ERR_UNSUPPORTED).
 * The backward forms g_nt = lam[0] * gx + gx0t and g_nb = lam[1] * gx + gx0b in fp32 and runs the per-input norm
 * backwards from them: one sort plan, one token-row gather per occurrence, one dense write of each table; g_lam =
 * (sum gx . x0t, sum gx . x0b).  gx0t / gx0b may be NULL (zero: the output was not used).  Workspace, plan and
 * ws_flags as for mot_embed_bwd (mot_embed_workspace_bytes(d), mot_embed_plan(_async)). */
int mot_split_residual_fwd(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                           const void* E_tok, const void* E_byte, const float* lam, void* x, void* x0t, void* x0b,
                           void* stream);
int mot_split_residual_bwd(const MotDesc* d, const int32_t* tok, const void* byte_ids, const void* ttb,
                           const void* E_tok, const void* E_byte, const float* lam, const void* gx, const void* gx0t,
                           const void* gx0b, void* gE_tok, void* gE_byte, float* g_lam, void* workspace, size_t ws_bytes,
                           int32_t ws_flags, void* stream);

/* ---- byte half of `--add-padded-and-pulled` (spt/train_gpt.py:371-379) ----------------------------------------
 * rows[pos, col_offset + k*byte_dim : +byte_dim] = rms_norm(E_byte[ids_a[pos,k]] + E_byte[ids_b[pos,k]]) for k < bpt:
 * two gathers summed BEFORE the per-byte norm (`norm(self.embed_bytes(byte_tensor) + self.embed_bytes(byte_tensor_pulled))`).
 * d: MOT_BYTES_ONLY with MOT_F_BYTE_NORM, out_dim = bpt*byte_dim; row_stride / col_offset locate the byte columns of the
 * [tok | bytes] projection operand, whose token columns mot_embed_fwd writes with MOT_TOK_ONLY and the same row_stride.
 * bpt <= 32, byte_dim a multiple of 8 with byte_dim <= 64 * G, G = the largest power of two <= 32 / bpt.  The ids:
 *   explicit : ids_a / ids_b token-major [n_tokens, bpt], int32 or int64 (MOT_F_IDS_I64); tok and ttb may be NULL;
 *   derived  : MOT_F_IDS_FROM_TTB with MOT_F_TTB_PULL_LEFT, or MOT_F_TTB_PULL_RIGHT optionally with MOT_F_TTB_NEXT_TOK:
 *              ids_a = the padded ids (the ttb rows of `tok`, mot_ttb_expand), ids_b = the pulled ids over rows of seq_len
 *              tokens, both derived inside the kernels; tok int32 [n_tokens] (+ the lookahead tail), ttb [tok_vocab, bpt]
 *              of ttb_dtype, pad_id / eot_id; ids_a and ids_b are NULL.
 * Any other combine or flag: MOT_ERR_BAD_ARG. */
int mot_byte_pair_fwd(const MotDesc* d, const int32_t* tok, const void* ids_a, const void* ids_b, const void* ttb,
                      const void* E_byte, void* out, void* stream);
/* Backward: gE_byte [byte_vocab, byte_dim] dense, fully overwritten, = the norm backward of every (position, slot)
 * added to BOTH gathered rows.  workspace: mot_byte_pair_workspace_bytes() bytes (cleared by the call). */
size_t mot_byte_pair_workspace_bytes(int32_t byte_vocab, int32_t byte_dim);
int mot_byte_pair_bwd(const MotDesc* d, const int32_t* tok, const void* ids_a, const void* ids_b, const void* ttb,
                      const void* E_byte, const void* grad_out, void* gE_byte, void* workspace, size_t ws_bytes,
                      void* stream);

/* ---- data-parallel exchange: average the gradient bucket across ranks through NVLink / NVSwitch -----------------
 * Replaces the per-parameter dist.all_reduce(param.grad, AVG) of spt/train_gpt.py:1320-1321 and runs/7:697-700 (launched
 * asynchronously and waited per optimizer in the runs, :697-711) for the tensors this path owns.
 * The bucket is one symmetric-memory buffer per rank (same size everywhere):
 *   multicast_ptr    : this rank's multicast mapping of all copies (NVLS), or NULL
 *   peer_ptrs_dev    : device array of `world` pointers, entry q = rank q's copy as addressable from this rank (P2P), or NULL
 *   signal_pads_dev  : device array of `world` pointers to the ranks' zero-initialised uint32 signal pads (>= 9216 bytes)
 *   work_area        : 256 bytes of ordinary device memory of this rank, zero-initialised once (tile counters of the launches)
 * mot_dp_exchange averages the byte range [byte_offset, byte_offset + n_bytes) of the bucket in place on every rank
 * (both multiples of 16).  Every rank makes the same sequence of calls.  `epoch` is the caller's barrier counter: the
 * call uses `epoch` for its entry barrier and, when `last` != 0, `epoch + 1` for an exit barrier -- so it grows by 1
 * per call and by 2 after a `last` call (start at 1).  A step that exchanges its bucket in several ranges (one per
 * mot_embed_bwd_slab) sets `last` on the final one only: ranges of one step are disjoint, and the exit barrier is what
 * lets every rank reuse the bucket afterwards.  Ordered on `stream` after the local backward of the range.
 *   algo MOT_DP_NVLS : multimem.ld_reduce / multimem.st through the multicast mapping (reduction inside the switch)
 *        MOT_DP_P2P  : loads / stores through the peer pointers, fp32 accumulation in rank order (world 2, 4 or 8) */
enum { MOT_DP_NVLS = 0, MOT_DP_P2P = 1 };
int mot_dp_exchange(void* multicast_ptr, void* const* peer_ptrs_dev, void* const* signal_pads_dev, void* work_area,
                    int32_t rank, int32_t world, int64_t byte_offset, int64_t n_bytes, int32_t dtype, uint32_t epoch,
                    int32_t last, int32_t algo, void* stream);
/* Touched-rows exchange.  A vocabulary row that no rank gathered is zero in every copy and needs no exchange.
 * mot_embed_touched_rows writes this rank's bitmap (bit v of word v/32: the batch of the planned workspace contains token
 * v; ceil(tok_vocab/32) uint32 words) -- call it after the backward, into the bucket's symmetric memory.
 * mot_dp_exchange_rows ORs the ranks' bitmaps through the fabric and averages only the rows of the union of the table at
 * [table_byte_offset, + n_rows*row_bytes), then the dense range [dense_byte_offset, + dense_bytes) (the byte table, other
 * parameters); both barriers: `epoch` grows by 2.  Rows that are zero everywhere stay untouched.
 * Precondition (the dense-gradient contract of mot_embed_bwd): a row whose bit is clear in a rank's bitmap is all zeros in
 * that rank's copy -- the peer-to-peer variant does not read such a copy at all (MOT_DP_PEER_BITS=0 reads every copy of a
 * union row, as the in-switch reduction necessarily does). */
int mot_embed_touched_rows(const MotDesc* d, const void* workspace, size_t ws_bytes, uint32_t* bitmap, void* stream);
int mot_dp_exchange_rows(void* multicast_ptr, void* const* peer_ptrs_dev, void* const* signal_pads_dev, void* work_area,
                         int32_t rank, int32_t world, int64_t table_byte_offset, int32_t n_rows, int32_t row_bytes,
                         int64_t bitmap_byte_offset, int64_t dense_byte_offset, int64_t dense_bytes, int32_t dtype,
                         uint32_t epoch, int32_t algo, void* stream);
/* Touched-rows exchange of several row tables.  Tables gathered with the same token ids (the front's token table and
 * the value embeddings, runs/7:252,308) touch the same rows, so ONE bitmap describes them all; the kernel moves row v of
 * every table for each row v of the union.  Tables may differ in width. */
#define MOT_DP_MAX_ROW_TABLES 8
typedef struct MotRowTable {
  int64_t byte_offset;  /* row 0 of the table in the bucket */
  int32_t row_bytes;
  int32_t reserved;     /* 0 */
} MotRowTable;
/* mot_dp_exchange_rows for n_tables row tables of n_rows rows each, all indexed by the token ids the bitmap describes.
 * `tables` is a HOST array read during the call.  Offsets and row_bytes are multiples of 16; the tables, the bitmap and
 * the dense range must not overlap.  mot_dp_exchange_rows is this call with one table (same bits, same summation
 * order).  Precondition as above, for every table: a row whose bit is clear in a rank's bitmap is all zeros in every
 * table of that rank's copy.  Errors, all before any CUDA call: n_tables outside 1..MOT_DP_MAX_ROW_TABLES, a NULL
 * `tables`, a nonzero `reserved` or overlapping ranges -> MOT_ERR_BAD_ARG; misaligned offsets or widths ->
 * MOT_ERR_MISALIGNED; MOT_DP_P2P at a world other than 2 or 4 -> MOT_ERR_UNSUPPORTED. */
int mot_dp_exchange_rows_multi(void* multicast_ptr, void* const* peer_ptrs_dev, void* const* signal_pads_dev,
                               void* work_area, int32_t rank, int32_t world, const MotRowTable* tables, int32_t n_tables,
                               int32_t n_rows, int64_t bitmap_byte_offset, int64_t dense_byte_offset, int64_t dense_bytes,
                               int32_t dtype, uint32_t epoch, int32_t algo, void* stream);
/* The whole bucket as one NVLS range with both barriers (= mot_dp_exchange(..., 0, n_bytes, ..., last = 1, MOT_DP_NVLS)):
 * `epoch` grows by 2 per call. */
int mot_dp_allreduce_avg(void* multicast_ptr, void* const* signal_pads_dev, void* work_area, int32_t rank, int32_t world,
                         int64_t n_bytes, int32_t dtype, uint32_t epoch, void* stream);

/* ---- byte pull across tokens ------------------------------------------------------------------------------
 * Replaces pull_from_left / pull_from_right (spt/data_creation.py:179-305 / :71-176, runs/7:351-428).
 * bytes_in / bytes_out: [n_rows, tokens_per_row * bpt] int32 or int64 (ids_i64), rows independent; a token whose bpt
 * bytes all equal eot_byte passes through and resets the pool; from_right == 0: rows are left-padded, every token
 * receives the last bpt non-pad bytes of its segment up to itself (right-aligned); != 0: the mirror image. */
size_t mot_pull_workspace_bytes(int64_t n_rows, int64_t tokens_per_row, int32_t bpt);
int mot_pull(const void* bytes_in, void* bytes_out, int64_t n_rows, int64_t tokens_per_row, int32_t bpt,
             int32_t ids_i64, int32_t pad_byte, int32_t eot_byte, int32_t from_right, void* workspace,
             size_t ws_bytes, void* stream);

/* ---- output side: token rows -> byte rows (the mirror image of the input mix) ------------------------------------
 * y[(t*bpt + k), :] = x[t, :] for k < bpt: ByteMixoutCopy's `einops.repeat(x, "... T D -> ... (T bpt) D")`
 * (spt/train_gpt.py:493); the backward sums the bpt copies in fp32: grad_x[t] = sum_k grad_y[t*bpt + k].
 * (ByteMixoutSplit's `rearrange "... T (bpt D) -> ... (T bpt) D"`, :516, is a view of contiguous rows: no kernel.)
 * x / grad_x: [n_rows, dim]; y / grad_y: [n_rows*bpt, dim]; dim a multiple of 16 bytes; pointers 16-byte aligned. */
int mot_mixout_copy_fwd(const void* x, void* y, int64_t n_rows, int32_t dim, int32_t bpt, int32_t dtype, void* stream);
int mot_mixout_copy_bwd(const void* grad_y, void* grad_x, int64_t n_rows, int32_t dim, int32_t bpt, int32_t dtype,
                        void* stream);

/* ---- dense projection of the concat+projection variants (tcgen05 tensor cores) -------------------------------
 * dtype = MOT_BF16: bf16 operands (kind::f16); MOT_F32: fp32 operands read in place on the TF32 path (kind::tf32, the
 * precision mathblations selects with set_float32_matmul_precision('high'), main.py:522); fp32 accumulation in tensor
 * memory either way.  in_dim = tok_dim + bpt*byte_dim (the row width of the
 * [tok | bytes] operand mot_embed_fwd produces with MOT_CONCAT), out_dim = model_dim; both multiples of 8. */

/* y[n_tokens, out_dim] = x[n_tokens, in_dim] . w[out_dim, in_dim]^T (+ bias[out_dim], fp32, or NULL).
 * Replaces F.linear of mixin_bytes (runs/7:233-234), CastedLinear (spt/train_gpt.py:185-186,443) and
 * DigitMixinConcat.fc (mathblations/model.py:261,268).  y is bf16, or fp32 when y_f32 != 0 (always with MOT_F32). */
int mot_linear_fwd(const void* x, const void* w, const float* bias, void* y, int64_t n_tokens, int32_t in_dim,
                   int32_t out_dim, int32_t dtype, int32_t y_f32, void* stream);
/* dx[n_tokens, in_dim] = dy[n_tokens, out_dim] . w[out_dim, in_dim]   (autograd of F.linear w.r.t. its input) */
/* The two backward products read bf16 operands in place; with MOT_F32 they run on transposed fp32 copies built in a
 * caller-provided workspace of mot_linear_workspace_bytes() bytes (0 for bf16: pass NULL). */
size_t mot_linear_workspace_bytes(int64_t n_tokens, int32_t in_dim, int32_t out_dim, int32_t dtype);
int mot_linear_bwd_input(const void* dy, const void* w, void* dx, int64_t n_tokens, int32_t in_dim, int32_t out_dim,
                         int32_t dtype, void* workspace, size_t ws_bytes, void* stream);
/* dw[out_dim, in_dim] = dy^T . x, reduced in fp32 into dw_f32 (overwritten; the fp32 master-weight gradient of
 * spt/train_gpt.py:1155-1156) and, when dw_bf16 != NULL, also cast to bf16 (the bf16 mixin weight of runs/7:249). */
int mot_linear_bwd_weight(const void* dy, const void* x, float* dw_f32, void* dw_bf16, int64_t n_tokens, int32_t in_dim,
                          int32_t out_dim, int32_t dtype, void* workspace, size_t ws_bytes, void* stream);

/* fp32 -> bf16, round to nearest even: CastedLinear's per-call `self.weight.type_as(x)` (spt/train_gpt.py:185-186) for the
 * fp32 master weight of the mixin projection.  Pointers 16-byte aligned. */
int mot_cast_f32_bf16(const float* in, void* out_bf16, int64_t n, void* stream);
/* out[dim] (fp32) = column sums of x [n_rows, dim] (bf16 or fp32): the bias gradient of F.linear
 * (mathblations/model.py:261,268).  Fixed summation order (no atomics).  dim even. */
int mot_colsum(const void* x, float* out, int64_t n_rows, int32_t dim, int32_t dtype, void* stream);

/* Row-wise rms_norm without weight (F.rms_norm(x, (x.size(-1),)), spt/train_gpt.py:172-173) over [n_rows, dim] and
 * its backward dy = rs*g - y*rs^3*mean(g.y): the `norm(...)` around the projection (runs/7:234, train_gpt.py:443). */
int mot_rmsnorm_fwd(const void* y, void* out, int64_t n_rows, int32_t dim, int32_t dtype, float eps, void* stream);
int mot_rmsnorm_bwd(const void* y, const void* grad_out, void* dy, int64_t n_rows, int32_t dim, int32_t dtype, float eps,
                    void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MOT_B200_H */
