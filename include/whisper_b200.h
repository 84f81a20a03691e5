/* whisper_b200 — C ABI of the B200-native Whisper hot path.
 *
 * This is the thin extern-"C" layer BASELINE.json's north_star asks for: plain pointers and sizes, no C++ or torch types.
 * The COM-style iModel / iContext shells of the reference (include/whisper_b200_com.h) sit on top of it, exactly where the
 * reference's own back-ends sit behind Whisper/modelFactory.cpp:5-20.
 *
 * Each entry point names the reference interface it stands in for (paths relative to the reference tree):
 *   wsp_model_open            Whisper/Whisper/WhisperModel.cpp:434-492 (WhisperModel::load) == Whisper/source/whisper.cpp:451-1072
 *   wsp_engine_create         Whisper/Whisper/WhisperModel.cpp:257-340 (loadGpu: tensors -> VRAM)
 *   wsp_context_create        Whisper/Whisper/ModelImpl.cpp:14 (createContext), KV sizing Whisper/Whisper/WhisperContext.cpp:291-308
 *   wsp_pcm_to_mel            Whisper/source/whisper.h:97 whisper_pcm_to_mel      (Whisper/Whisper/Spectrogram.cpp:64-121)
 *   wsp_pcm_to_mel_window     Whisper/Whisper/MelStreamer.cpp:128-236 (MelStreamer::makeTransposedBuffer / makeBuffer: one window of a streamed clip)
 *   wsp_set_mel               Whisper/source/whisper.h:107 whisper_set_mel
 *   wsp_encode                Whisper/source/whisper.h:117 whisper_encode          (Whisper/Whisper/WhisperContext.cpp:310 encode)
 *   wsp_decode                Whisper/source/whisper.h:128 whisper_decode + :140-150 whisper_sample_best/timestamp
 *                             (Whisper/Whisper/WhisperContext.cpp:578 decode, Whisper/Whisper/ContextImpl.cpp:71-157 sampleBest)
 *   wsp_get_logits/probs      Whisper/source/whisper.h:166 whisper_get_probs
 *   wsp_run_chunks            the fixed-length greedy chunk loop of BASELINE.md §2 (mel + encode + n_decode x (decode + sample))
 *   wsp_get_tensor            the reference's named trace points, Whisper/Utils/Trace/tracing.h (names as in whisper.cpp:1121-1869)
 *
 * Error handling mirrors the reference's HRESULT convention (SURVEY.md §8b): every function returns a wsp_status that the COM
 * shell maps 1:1 to an HRESULT; no exception crosses this boundary.  There is NO CPU fallback: if the CUDA device or the
 * sm_100a kernels are unavailable the calls fail with WSP_E_CUDA.
 *
 * Threading: a wsp_model / wsp_engine is immutable after creation and may be shared; a wsp_context is single-threaded state
 * (KV memories, workspaces), one per concurrent stream — the same contract as iModel / iContext (Whisper/Whisper/WhisperModel.h:28-31).
 */
#ifndef WHISPER_B200_H
#define WHISPER_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef int32_t wsp_status;
enum
{
	WSP_OK = 0,
	WSP_S_FALSE = 1,          /* "did nothing" (S_FALSE) */
	WSP_E_INVALIDARG = -1,
	WSP_E_POINTER = -2,
	WSP_E_FILE = -3,          /* cannot open / truncated */
	WSP_E_FORMAT = -4,        /* not a ggml whisper file, missing or mis-shaped tensors */
	WSP_E_CUDA = -5,          /* CUDA runtime / driver failure, or no sm_100a device */
	WSP_E_OUTOFMEMORY = -6,
	WSP_E_BOUNDS = -7,        /* batch, token count or context length beyond what the context was created for */
	WSP_E_NOTIMPL = -8,
};

typedef struct wsp_model wsp_model;
typedef struct wsp_engine wsp_engine;
typedef struct wsp_context wsp_context;

/* whisper_token_data (Whisper/source/whisper.h:71-85) without the token-level timestamp fields */
typedef struct wsp_token_data
{
	int32_t id;      /* sampled token */
	int32_t tid;     /* most probable timestamp token */
	float p;         /* probability of `id` */
	float pt;        /* probability of `tid` among timestamp tokens */
	float ptsum;     /* total probability of all timestamp tokens */
} wsp_token_data;

/* decode flags */
enum
{
	WSP_DECODE_FORCE_TIMESTAMP = 1,   /* whisper_sample_timestamp */
	WSP_DECODE_INITIAL = 2,           /* is_initial: first timestamp <= 1.00 s */
	WSP_DECODE_ALL_LOGITS = 4,        /* keep logits/probs for every prompt token (n_tokens <= 8), as the oracle does */
	WSP_DECODE_DEVICE_TOKENS = 8,     /* feed the tokens sampled by the previous call (no host round trip); n_past continues */
	WSP_DECODE_NO_SAMPLE = 16,
};

/* ---- library ---- */
const char* wsp_version( void );
const char* wsp_last_error( void );              /* thread-local text of the last failure */
int32_t wsp_device_count( void );
wsp_status wsp_device_name( int32_t device, char* dst, size_t cap );   /* replaces listGPUs (Whisper/D3D/listGPUs.cpp) */
/* number of kernels this library has launched since load (bench.py's gpu_launches evidence) */
uint64_t wsp_launch_count( void );

/* ---- model file (host) ---- */
wsp_status wsp_model_open( const char* path_utf8, wsp_model** out );
void wsp_model_close( wsp_model* m );
/* n_vocab, n_audio_ctx, n_audio_state, n_audio_head, n_audio_layer, n_text_ctx, n_text_state, n_text_head, n_text_layer, n_mels, f16 */
wsp_status wsp_model_hparams( const wsp_model* m, int32_t out11[ 11 ] );
/* eot, sot, prev, solm, not, beg, translate, transcribe */
wsp_status wsp_model_special_tokens( const wsp_model* m, int32_t out8[ 8 ] );
const char* wsp_model_token_text( const wsp_model* m, int32_t id );
int32_t wsp_model_is_multilingual( const wsp_model* m );
/* raw file image, for broadcasting to peer GPUs before wsp_engine_create_from_image */
const void* wsp_model_file_data( const wsp_model* m, uint64_t* size );
/* the small host-side part (hparams, filters, vocabulary, tensor directory) as a relocatable blob */
wsp_status wsp_model_meta_serialize( const wsp_model* m, void* dst, uint64_t cap, uint64_t* size );
wsp_status wsp_model_from_meta( const void* meta, uint64_t size, wsp_model** out );

/* ---- engine: weights resident on one device ---- */
wsp_status wsp_engine_create( const wsp_model* m, int32_t device, wsp_engine** out );
/* same, but the tensor data is taken from a device-resident copy of the file image (e.g. received by an NCCL broadcast) */
wsp_status wsp_engine_create_from_image( const wsp_model* m, int32_t device, const void* dev_file_image, uint64_t size, wsp_engine** out );
void wsp_engine_destroy( wsp_engine* e );
uint64_t wsp_engine_weight_bytes( const wsp_engine* e );

/* ---- context: per-stream state for up to max_batch independent 30 s chunks ---- */
wsp_status wsp_context_create( wsp_engine* e, int32_t max_batch, wsp_context** out );
void wsp_context_destroy( wsp_context* c );
wsp_status wsp_synchronize( wsp_context* c );
/* device memory held by the context: workspaces, KV caches, mel slots (ContextImpl::getMemoryUse, Whisper/Whisper/ContextImpl.misc.cpp:170-182) */
uint64_t wsp_context_device_bytes( const wsp_context* c );

/* a1: 16 kHz mono f32 PCM (host) -> log-mel of chunk slot `slot`, kept on the device.  n_len = n_samples / 160 frames. */
wsp_status wsp_pcm_to_mel( wsp_context* c, int32_t slot, const float* pcm, int32_t n_samples );
/* a1, streamed flavour (iContext::runStreamed): log-mel of frames [0, n_frames) of `pcm` — which should extend 240 samples past the
 * last frame unless the stream ends there — normalised by the maximum over these frames only, floored at 1e-20; `forced_max` (may be
 * NULL) replaces that maximum, `max_out` (may be NULL) receives the maximum found.  The slot then holds n_frames frames. */
wsp_status wsp_pcm_to_mel_window( wsp_context* c, int32_t slot, const float* pcm, int32_t n_samples, int32_t n_frames, const float* forced_max, float* max_out );
wsp_status wsp_set_mel( wsp_context* c, int32_t slot, const float* mel, int32_t n_len );     /* [80][n_len] */
int32_t wsp_mel_len( wsp_context* c, int32_t slot );
wsp_status wsp_get_mel( wsp_context* c, int32_t slot, float* dst, size_t cap_floats );

/* a2-a12: encoder + cross-KV for slots [0,batch); mel_offsets[b] = first frame of the 3000-frame window (NULL = 0) */
wsp_status wsp_encode( wsp_context* c, const int32_t* mel_offsets, int32_t batch );

/* a13-a18: one decoder call for `batch` chunks, n_tokens new tokens each (tokens[b*n_tokens + i]), after n_past cached ones.
 * sampled (nullable) receives the greedy choice per chunk from the last token's distribution. */
wsp_status wsp_decode( wsp_context* c, const int32_t* tokens, int32_t n_tokens, int32_t n_past, int32_t batch, uint32_t flags, wsp_token_data* sampled );
/* logits / probabilities of the last wsp_decode: [batch][n_vocab], or [batch*n_tokens][n_vocab] after WSP_DECODE_ALL_LOGITS */
wsp_status wsp_get_logits( wsp_context* c, float* dst, size_t cap_floats );
wsp_status wsp_get_probs( wsp_context* c, float* dst, size_t cap_floats );

/* whisper_lang_auto_detect (Whisper/source/whisper.cpp:2428-2495): encode slot 0's window at mel frame `offset_frames`, decode [sot],
 * then — like the reference — a softmax over the language tokens' PROBABILITIES; lang_probs[n_langs] (nullable), *lang_id = the arg-max */
wsp_status wsp_detect_language( wsp_context* c, int32_t offset_frames, int32_t n_langs, float* lang_probs, int32_t* lang_id );

/* The measured path: for `batch` chunks of host PCM — mel, encode, then n_decode greedy steps (first step samples with
 * is_initial timestamp rules, as whisper_full does, whisper.cpp:2943) entirely on the device with sampled tokens fed back
 * without host round trips.  tokens_out[b*n_decode + i].  stage_ms (nullable): { h2d+mel, encode, decode } from CUDA events. */
wsp_status wsp_run_chunks( wsp_context* c, const float* const* pcm, const int32_t* n_samples, int32_t batch,
	const int32_t* prompt, int32_t n_prompt, int32_t n_decode, int32_t* tokens_out, float* stage_ms );
/* keep a chunk's PCM resident in HBM (slot-owned copy) ... */
wsp_status wsp_upload_pcm( wsp_context* c, int32_t slot, const float* pcm, int32_t n_samples );
/* ... and run the same path from it: mel + encode + decode with no host->device input copy inside (bench.py's `value` leg) */
wsp_status wsp_run_chunks_resident( wsp_context* c, int32_t batch, const int32_t* prompt, int32_t n_prompt, int32_t n_decode, int32_t* tokens_out, float* stage_ms );

/* ---- several devices in one process (csrc/replicas.cpp) ----
 * Chunks are independent (SURVEY.md §8e): one engine + context per listed device (a device may be listed twice: two contexts on one
 * GPU), the model file read ONCE and its image copied device-to-device from devices[0] (cudaMemcpyPeer over NVLink) — the C++ form of
 * bench.py's NCCL broadcast; reference analogues: iModel::clone (Whisper/Whisper/ModelImpl.cpp:40-60), whisper_full_parallel
 * (Whisper/source/whisper.cpp:3127-3268). */
typedef struct wsp_replicas wsp_replicas;
typedef struct wsp_replica_stats
{
	int32_t device;
	int32_t batches_done, chunks_done;
	int32_t failed;          /* the replica returned an error and was retired; its batch went back to the queue */
	float busy_ms;           /* host wall time spent inside wsp_run_chunks */
	float load_ms;           /* engine + context creation, including the image copy */
} wsp_replica_stats;
wsp_status wsp_replicas_create( const wsp_model* m, const int32_t* devices, int32_t n_devices, int32_t max_batch, wsp_replicas** out );
int32_t wsp_replicas_count( const wsp_replicas* r );
/* n_chunks clips through a host work queue: batches of <= max_batch chunks go to whichever replica is free; a batch whose replica fails
 * is re-queued for the others.  tokens_out[chunk * n_decode + i]; stats (nullable) [n_devices]. */
wsp_status wsp_replicas_run_chunks( wsp_replicas* r, const float* const* pcm, const int32_t* n_samples, int32_t n_chunks, const int32_t* prompt,
	int32_t n_prompt, int32_t n_decode, int32_t* tokens_out, wsp_replica_stats* stats );
/* test hook: replica i fails its next batch (exercises retire + re-queue) */
wsp_status wsp_replicas_debug_fail_next( wsp_replicas* r, int32_t replica );
void wsp_replicas_destroy( wsp_replicas* r );

/* CUDA-event stopwatch on the context's stream (the stream every kernel of this library is launched on) */
wsp_status wsp_timer_start( wsp_context* c );
wsp_status wsp_timer_stop( wsp_context* c, float* ms );
/* instrumented decoder pass for roofline accounting: n_steps more single-token steps, launched kernel by kernel with an event pair
 * around every launch.  kinds: 0 skinny GEMM, 1 cross-attention, 2 self-attention, 3 other (embedding, sampler) */
wsp_status wsp_profile_decode( wsp_context* c, int32_t batch, int32_t n_steps, float ms_by_kind[ 4 ], int32_t launches_by_kind[ 4 ] );

/* test hook: named intermediates of chunk `slot` as f32.  Names:
 *   "mel" ([80][n_len]), "enc.input" ([3000][80] f16 encoder input), "enc.conv1" ([3000][d] after GELU),
 *   "enc.x" ([T][d] residual stream: input of layer 0, or the output of the last layer run, see wsp_debug_set_encoder_layers),
 *   "encode-out" / "enc.xn" ([T][d] ln_post, f16-rounded), "enc.q", "enc.k" ([H][T][64] of the last layer run), "enc.vt" ([H][64][T
 *   padded]), "enc.attn" ([T][d] attention output of the last layer run),
 *   "cross_k", "cross_v" ([L][H][T][64] cross-attention memories), "self_k", "self_v" ([L][H][n_text_ctx][64] self-KV cache; rows
 *   at and past the decoder's n_past hold whatever earlier calls wrote there),
 *   "dec.x" ([8][d] first rows of the decoder's residual stream, for any slot; step mode 2 does not write it). */
wsp_status wsp_get_tensor( wsp_context* c, const char* name, int32_t slot, float* dst, size_t cap_floats, size_t* n_floats );
/* debug: run only the first n encoder layers (negative = all) */
wsp_status wsp_debug_set_encoder_layers( wsp_context* c, int32_t n );
/* The CPU reference accumulates the decoder's V^T*P product in f16, per thread (Whisper/source/ggml.c:4680-4722), so its logits
 * depend on its thread count.  n = the cpuThreads the reference would be run with (sFullParams::cpuThreads; default 4 =
 * whisper_full_default_params, Whisper/source/whisper.cpp:2605); the decoder reproduces that arithmetic for n = 1..16 (the
 * single-launch step kernel covers all of them; WSP_E_INVALIDARG above 16).  n = 0: plain f32 accumulation (per-op kernels). */
wsp_status wsp_set_reference_threads( wsp_context* c, int32_t n );
/* debug: 0 = launch the N = 1 decoder step kernel by kernel instead of replaying the captured CUDA graph */
wsp_status wsp_debug_set_graph( wsp_context* c, int32_t on );
/* debug: how the single-token decoder step runs: 2 = one dataflow kernel (decode_flow.cu, default), 1 = round 1's persistent kernel with
 * grid barriers (decode_mega.cu, kept for same-box A/B runs), 0 = one kernel per op */
wsp_status wsp_debug_set_step_mode( wsp_context* c, int32_t mode );
/* debug: record %globaltimer marks (ns) of CTA 0 at every phase boundary of the decoder-step kernel; read them back after a step */
wsp_status wsp_debug_enable_step_timing( wsp_context* c, int32_t on );
wsp_status wsp_debug_step_timing( wsp_context* c, uint64_t* dst, int32_t cap );
/* pinned host memory for callers that want asynchronous H2D copies of PCM (bench.py's e2e leg) */
void* wsp_host_alloc( size_t bytes );
void wsp_host_free( void* p );
/* per-phase device time accumulated by the context (CUDA events): { mel, encode, decode, sample } in ms, and call counts */
wsp_status wsp_timings( wsp_context* c, float ms4[ 4 ], int32_t calls4[ 4 ], int32_t reset );

/* ---- kernel-level test hooks (tests/ only) ---- */
/* D[M][N] = A[M][K] * B[N][K]^T with the tcgen05 GEMM; A,B f16 bit patterns (uint16), D f32; all host pointers */
wsp_status wsp_test_gemm( int32_t device, int32_t M, int32_t N, int32_t K, const uint16_t* A, const uint16_t* B, float* D, int32_t bn, int32_t iters, float* ms );
/* encoder attention: Q,K [BH][T][64], V [BH][T][64] f16 bit patterns -> out f32 [BH][T][64] */
wsp_status wsp_test_attention( int32_t device, int32_t BH, int32_t T, const uint16_t* Q, const uint16_t* K, const uint16_t* V, float* out, int32_t iters, float* ms );
/* skinny GEMM: out[cols][nOut] = x[cols][K] * W[nOut][K]^T */
wsp_status wsp_test_skinny( int32_t device, int32_t nOut, int32_t K, int32_t cols, const uint16_t* W, const uint16_t* X, float* out, int32_t iters, float* ms );
/* sampler alone: rows of logits -> probs (softmax with the reference's f16-table exp, may be NULL) and one sampled token per row under
 * the rules of whisper_sample_best / whisper_sample_timestamp (whisper.cpp:1875-1964); special4 = { beg, sot, solm, not } */
wsp_status wsp_test_sample( int32_t device, int32_t rows, int32_t n_vocab, const float* logits, const int32_t special4[ 4 ], int32_t force_timestamp,
	int32_t is_initial, float* probs, wsp_token_data* out );
/* LayerNorm rows x d f32 -> f16 bit patterns */
wsp_status wsp_test_layernorm( int32_t device, int32_t rows, int32_t d, const float* x, const float* gamma, const float* beta, uint16_t* out );

#ifdef __cplusplus
}
#endif
#endif
