// extern "C" surface (include/whisper_b200.h) + kernel-level test hooks.
#include "engine.h"
#include <algorithm>
#include <math.h>
#include <math.h>
#include <memory>
#include <string.h>

using namespace wsp;

struct wsp_model { ModelFile* m; };
struct wsp_engine { Engine* e; };
struct wsp_context { Context* c; };

namespace
{
	template<class F> wsp_status guarded( F f )
	{
		try { return f(); }
		catch( const std::bad_alloc& ) { return fail( WSP_E_OUTOFMEMORY, "host allocation failed" ); }
		catch( const std::exception& ex ) { return fail( WSP_E_INVALIDARG, ex.what() ); }
		catch( ... ) { return fail( WSP_E_INVALIDARG, "unknown exception" ); }
	}
	template<class T> struct DevTmp
	{
		T* p = nullptr;
		~DevTmp() { if( p ) cudaFree( p ); }
		cudaError_t alloc( size_t n, bool zero = false )
		{
			cudaError_t e = cudaMalloc( (void**)&p, n * sizeof( T ) );
			if( e == cudaSuccess && zero ) e = cudaMemset( p, 0, n * sizeof( T ) );
			return e;
		}
	};
}

extern "C" {

const char* wsp_version( void ) { return "whisper_b200 0.1 (sm_100a: tcgen05 + TMA)"; }
const char* wsp_last_error( void ) { return g_lastError.c_str(); }
int32_t wsp_device_count( void )
{
	int n = 0;
	if( cudaGetDeviceCount( &n ) != cudaSuccess ) { cudaGetLastError(); return 0; }
	return n;
}
wsp_status wsp_device_name( int32_t device, char* dst, size_t cap )
{
	if( !dst || cap == 0 ) return fail( WSP_E_POINTER, "dst" );
	cudaDeviceProp p;
	WSP_CUDA( cudaGetDeviceProperties( &p, device ) );
	snprintf( dst, cap, "%s (sm_%d%d, %d SMs, %.0f GB)", p.name, p.major, p.minor, p.multiProcessorCount, (double)p.totalGlobalMem / 1e9 );
	return WSP_OK;
}
uint64_t wsp_launch_count( void ) { return g_launchCount.load(); }

// ---- model ----
wsp_status wsp_model_open( const char* path, wsp_model** out )
{
	if( !path || !out ) return fail( WSP_E_POINTER, "path/out" );
	return guarded( [ & ]() -> wsp_status {
		ModelFile* m = nullptr;
		std::string err;
		const int rc = openModelFile( path, &m, err );
		if( rc != WSP_OK ) return fail( rc, err );
		*out = new wsp_model{ m };
		return WSP_OK;
	} );
}
void wsp_model_close( wsp_model* m )
{
	if( !m ) return;
	delete m->m;
	delete m;
}
wsp_status wsp_model_hparams( const wsp_model* m, int32_t out11[ 11 ] )
{
	if( !m || !out11 ) return fail( WSP_E_POINTER, "model/out" );
	memcpy( out11, &m->m->hp, sizeof( int32_t ) * 11 );
	return WSP_OK;
}
wsp_status wsp_model_special_tokens( const wsp_model* m, int32_t out8[ 8 ] )
{
	if( !m || !out8 ) return fail( WSP_E_POINTER, "model/out" );
	const Vocab& v = m->m->vocab;
	const int32_t t[ 8 ] = { v.token_eot, v.token_sot, v.token_prev, v.token_solm, v.token_not, v.token_beg, Vocab::token_translate, Vocab::token_transcribe };
	memcpy( out8, t, sizeof( t ) );
	return WSP_OK;
}
const char* wsp_model_token_text( const wsp_model* m, int32_t id )
{
	if( !m || id < 0 || id >= (int32_t)m->m->vocab.id_to_token.size() ) return nullptr;
	return m->m->vocab.id_to_token[ id ].c_str();
}
int32_t wsp_model_is_multilingual( const wsp_model* m ) { return m && m->m->vocab.multilingual() ? 1 : 0; }
const void* wsp_model_file_data( const wsp_model* m, uint64_t* size )
{
	if( !m ) return nullptr;
	if( size ) *size = m->m->imageSize;
	return m->m->image;
}
wsp_status wsp_model_meta_serialize( const wsp_model* m, void* dst, uint64_t cap, uint64_t* size )
{
	if( !m || !size ) return fail( WSP_E_POINTER, "model/size" );
	return guarded( [ & ]() -> wsp_status {
		std::vector<uint8_t> blob;
		serializeMeta( *m->m, blob );
		*size = blob.size();
		if( !dst ) return WSP_OK;
		if( cap < blob.size() ) return fail( WSP_E_BOUNDS, "meta buffer too small" );
		memcpy( dst, blob.data(), blob.size() );
		return WSP_OK;
	} );
}
wsp_status wsp_model_from_meta( const void* meta, uint64_t size, wsp_model** out )
{
	if( !meta || !out ) return fail( WSP_E_POINTER, "meta/out" );
	return guarded( [ & ]() -> wsp_status {
		ModelFile* m = nullptr;
		std::string err;
		const int rc = modelFromMeta( static_cast<const uint8_t*>( meta ), size, &m, err );
		if( rc != WSP_OK ) return fail( rc, err );
		*out = new wsp_model{ m };
		return WSP_OK;
	} );
}

// ---- engine ----
wsp_status wsp_engine_create( const wsp_model* m, int32_t device, wsp_engine** out )
{
	if( !m || !out ) return fail( WSP_E_POINTER, "model/out" );
	return guarded( [ & ]() -> wsp_status {
		Engine* e = nullptr;
		WSP_CHECK( createEngine( *m->m, device, nullptr, 0, &e ) );
		*out = new wsp_engine{ e };
		return WSP_OK;
	} );
}
wsp_status wsp_engine_create_from_image( const wsp_model* m, int32_t device, const void* dev_file_image, uint64_t size, wsp_engine** out )
{
	if( !m || !out || !dev_file_image ) return fail( WSP_E_POINTER, "model/image/out" );
	return guarded( [ & ]() -> wsp_status {
		Engine* e = nullptr;
		WSP_CHECK( createEngine( *m->m, device, dev_file_image, size, &e ) );
		*out = new wsp_engine{ e };
		return WSP_OK;
	} );
}
void wsp_engine_destroy( wsp_engine* e )
{
	if( !e ) return;
	delete e->e;
	delete e;
}
uint64_t wsp_engine_weight_bytes( const wsp_engine* e ) { return e ? e->e->arenaUsed : 0; }

uint64_t wsp_context_device_bytes( const wsp_context* c ) { return c ? c->c->devBytes : 0; }

// ---- context ----
wsp_status wsp_context_create( wsp_engine* e, int32_t max_batch, wsp_context** out )
{
	if( !e || !out ) return fail( WSP_E_POINTER, "engine/out" );
	return guarded( [ & ]() -> wsp_status {
		Context* c = nullptr;
		WSP_CHECK( createContext( e->e, max_batch, &c ) );
		*out = new wsp_context{ c };
		return WSP_OK;
	} );
}
void wsp_context_destroy( wsp_context* c )
{
	if( !c ) return;
	delete c->c;
	delete c;
}
wsp_status wsp_synchronize( wsp_context* c )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	WSP_CUDA( cudaStreamSynchronize( c->c->stream ) );
	return WSP_OK;
}
wsp_status wsp_pcm_to_mel( wsp_context* c, int32_t slot, const float* pcm, int32_t n_samples )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	return guarded( [ & ]() -> wsp_status { return ctxPcmToMel( *c->c, slot, pcm, n_samples ); } );
}
wsp_status wsp_pcm_to_mel_window( wsp_context* c, int32_t slot, const float* pcm, int32_t n_samples, int32_t n_frames, const float* forced_max, float* max_out )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	return guarded( [ & ]() -> wsp_status { return ctxPcmToMelWindow( *c->c, slot, pcm, n_samples, n_frames, forced_max, max_out ); } );
}
wsp_status wsp_set_mel( wsp_context* c, int32_t slot, const float* mel, int32_t n_len )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	return guarded( [ & ]() -> wsp_status { return ctxSetMel( *c->c, slot, mel, n_len ); } );
}
int32_t wsp_mel_len( wsp_context* c, int32_t slot )
{
	if( !c || slot < 0 || slot >= c->c->maxB ) return -1;
	return c->c->slots[ slot ].nLen;
}
wsp_status wsp_get_mel( wsp_context* c, int32_t slot, float* dst, size_t cap )
{
	if( !c || !dst ) return fail( WSP_E_POINTER, "context/dst" );
	if( slot < 0 || slot >= c->c->maxB ) return fail( WSP_E_BOUNDS, "slot" );
	const MelSlot& s = c->c->slots[ slot ];
	const size_t n = (size_t)80 * s.nLen;
	if( cap < n ) return fail( WSP_E_BOUNDS, "dst too small" );
	WSP_CUDA( cudaSetDevice( c->c->e->device ) );
	WSP_CUDA( cudaStreamSynchronize( c->c->stream ) );
	if( n ) WSP_CUDA( cudaMemcpy( dst, s.mel, n * 4, cudaMemcpyDeviceToHost ) );
	return WSP_OK;
}
wsp_status wsp_encode( wsp_context* c, const int32_t* mel_offsets, int32_t batch )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	return guarded( [ & ]() -> wsp_status { return ctxEncode( *c->c, mel_offsets, batch ); } );
}
wsp_status wsp_decode( wsp_context* c, const int32_t* tokens, int32_t n_tokens, int32_t n_past, int32_t batch, uint32_t flags, wsp_token_data* sampled )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	return guarded( [ & ]() -> wsp_status { return ctxDecode( *c->c, tokens, n_tokens, n_past, batch, flags, sampled ); } );
}
static wsp_status copyRows( wsp_context* c, const float* src, float* dst, size_t cap )
{
	if( !c || !dst ) return fail( WSP_E_POINTER, "context/dst" );
	const size_t n = (size_t)c->c->lastLogitRows * c->c->e->hp.n_vocab;
	if( cap < n ) return fail( WSP_E_BOUNDS, "dst too small" );
	WSP_CUDA( cudaSetDevice( c->c->e->device ) );
	WSP_CUDA( cudaStreamSynchronize( c->c->stream ) );
	if( n ) WSP_CUDA( cudaMemcpy( dst, src, n * 4, cudaMemcpyDeviceToHost ) );
	return WSP_OK;
}
wsp_status wsp_get_logits( wsp_context* c, float* dst, size_t cap ) { return copyRows( c, c ? c->c->logits : nullptr, dst, cap ); }
wsp_status wsp_get_probs( wsp_context* c, float* dst, size_t cap ) { return copyRows( c, c ? c->c->probs : nullptr, dst, cap ); }

wsp_status wsp_run_chunks( wsp_context* c, const float* const* pcm, const int32_t* n_samples, int32_t batch, const int32_t* prompt, int32_t n_prompt,
	int32_t n_decode, int32_t* tokens_out, float* stage_ms )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	return guarded( [ & ]() -> wsp_status { return ctxRunChunks( *c->c, pcm, n_samples, batch, prompt, n_prompt, n_decode, tokens_out, stage_ms, false ); } );
}
wsp_status wsp_run_chunks_resident( wsp_context* c, int32_t batch, const int32_t* prompt, int32_t n_prompt, int32_t n_decode, int32_t* tokens_out, float* stage_ms )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	return guarded( [ & ]() -> wsp_status { return ctxRunChunks( *c->c, nullptr, nullptr, batch, prompt, n_prompt, n_decode, tokens_out, stage_ms, true ); } );
}

wsp_status wsp_upload_pcm( wsp_context* c, int32_t slot, const float* pcm, int32_t n_samples )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	return guarded( [ & ]() -> wsp_status { return ctxUploadPcm( *c->c, slot, pcm, n_samples ); } );
}
wsp_status wsp_profile_decode( wsp_context* c, int32_t batch, int32_t n_steps, float ms_by_kind[ 4 ], int32_t launches_by_kind[ 4 ] )
{
	if( !c || !ms_by_kind || !launches_by_kind ) return fail( WSP_E_POINTER, "context/out" );
	return guarded( [ & ]() -> wsp_status { return ctxProfileDecode( *c->c, batch, n_steps, ms_by_kind, launches_by_kind ); } );
}
wsp_status wsp_timer_start( wsp_context* c )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	WSP_CUDA( cudaSetDevice( c->c->e->device ) );
	WSP_CUDA( cudaEventRecord( c->c->timerEv[ 0 ], c->c->stream ) );
	return WSP_OK;
}
wsp_status wsp_timer_stop( wsp_context* c, float* ms )
{
	if( !c || !ms ) return fail( WSP_E_POINTER, "context/ms" );
	WSP_CUDA( cudaEventRecord( c->c->timerEv[ 1 ], c->c->stream ) );
	WSP_CUDA( cudaEventSynchronize( c->c->timerEv[ 1 ] ) );
	WSP_CUDA( cudaEventElapsedTime( ms, c->c->timerEv[ 0 ], c->c->timerEv[ 1 ] ) );
	return WSP_OK;
}

__global__ void half_to_float_kernel( const __half* src, float* dst, size_t n )
{
	const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
	if( i < n ) dst[ i ] = __half2float( src[ i ] );
}

wsp_status wsp_get_tensor( wsp_context* cc, const char* name, int32_t slot, float* dst, size_t cap, size_t* n_floats )
{
	if( !cc || !name || !n_floats ) return fail( WSP_E_POINTER, "context/name/n" );
	Context& c = *cc->c;
	if( slot < 0 || slot >= c.maxB ) return fail( WSP_E_BOUNDS, "slot" );
	const HParams& hp = c.e->hp;
	const int d = hp.n_audio_state, T = hp.n_audio_ctx, L = hp.n_text_layer, H = hp.n_audio_head;
	WSP_CUDA( cudaSetDevice( c.e->device ) );
	WSP_CUDA( cudaStreamSynchronize( c.stream ) );
	const std::string nm( name );
	const float* f32 = nullptr;
	const __half* f16 = nullptr;
	size_t n = 0;
	if( nm == "mel" ) { f32 = c.slots[ slot ].mel; n = (size_t)80 * c.slots[ slot ].nLen; }
	else if( nm == "enc.input" ) { f16 = c.melF16 + ( (size_t)slot * kFramesPad + 1 ) * 80; n = (size_t)kFrames * 80; }       // [3000][80]
	else if( nm == "enc.conv1" ) { f16 = c.conv1 + ( (size_t)slot * kFramesPad + 1 ) * d; n = (size_t)kFrames * d; }           // [3000][d]
	else if( nm == "enc.x" ) { f32 = c.x + (size_t)slot * T * d; n = (size_t)T * d; }                                             // [1500][d]
	else if( nm == "enc.xn" || nm == "encode-out" ) { f16 = c.xn + (size_t)slot * T * d; n = (size_t)T * d; }
	else if( nm == "enc.attn" ) { f16 = c.attn + (size_t)slot * T * d; n = (size_t)T * d; }
	else if( nm == "enc.q" ) { f16 = c.q + (size_t)slot * T * d; n = (size_t)T * d; }                                             // [H][T][64]
	else if( nm == "enc.k" ) { f16 = c.k + (size_t)slot * T * d; n = (size_t)T * d; }
	else if( nm == "enc.vt" ) { f16 = c.vt + (size_t)slot * H * 64 * c.Tp; n = (size_t)H * 64 * c.Tp; }                            // [H][64][Tp]
	else if( nm == "cross_k" || nm == "cross_v" || nm == "self_k" || nm == "self_v" )
	{
		// gathered per layer below: [L][H][rows][64] of this slot, rows = T (cross-attention memories) or n_text_ctx (self-KV cache)
		const bool self = nm[ 0 ] == 's';
		const size_t per = (size_t)( self ? hp.n_text_ctx : T ) * hp.n_text_state;
		n = (size_t)L * per;
		if( n_floats ) *n_floats = n;
		if( !dst ) return WSP_OK;
		if( cap < n ) return fail( WSP_E_BOUNDS, "dst too small" );
		DevTmp<float> tmp;
		WSP_CUDA( tmp.alloc( per ) );
		const __half* base = nm == "cross_k" ? c.crossK : nm == "cross_v" ? c.crossV : nm == "self_k" ? c.selfK : c.selfV;
		for( int l = 0; l < L; l++ )
		{
			const __half* src = base + ( (size_t)l * c.maxB + slot ) * per;
			half_to_float_kernel<<<(unsigned)( ( per + 255 ) / 256 ), 256, 0, c.stream>>>( src, tmp.p, per );
			WSP_CUDA( cudaMemcpyAsync( dst + (size_t)l * per, tmp.p, per * 4, cudaMemcpyDeviceToHost, c.stream ) );
			WSP_CUDA( cudaStreamSynchronize( c.stream ) );
		}
		return WSP_OK;
	}
	else if( nm == "dec.x" ) { f32 = c.xd; n = (size_t)d * 8; }
	else return fail( WSP_E_INVALIDARG, "unknown tensor name " + nm );
	*n_floats = n;
	if( !dst ) return WSP_OK;
	if( cap < n ) return fail( WSP_E_BOUNDS, "dst too small" );
	if( n == 0 ) return WSP_OK;
	if( f32 ) WSP_CUDA( cudaMemcpy( dst, f32, n * 4, cudaMemcpyDeviceToHost ) );
	else
	{
		DevTmp<float> tmp;
		WSP_CUDA( tmp.alloc( n ) );
		half_to_float_kernel<<<(unsigned)( ( n + 255 ) / 256 ), 256>>>( f16, tmp.p, n );
		WSP_CUDA( cudaMemcpy( dst, tmp.p, n * 4, cudaMemcpyDeviceToHost ) );
	}
	return WSP_OK;
}
// whisper_lang_auto_detect (Whisper/source/whisper.cpp:2428-2495)
wsp_status wsp_detect_language( wsp_context* c, int32_t offset_frames, int32_t n_langs, float* lang_probs, int32_t* lang_id )
{
	if( !c || !lang_id ) return fail( WSP_E_POINTER, "context/lang_id" );
	return guarded( [ & ]() -> wsp_status {
		Context& cx = *c->c;
		const Engine& e = *cx.e;
		const int nVocab = e.hp.n_vocab;
		if( n_langs < 1 || e.tokSot + n_langs >= nVocab ) return fail( WSP_E_INVALIDARG, "n_langs" );
		const int32_t off = offset_frames;
		WSP_CHECK( ctxEncode( cx, &off, 1 ) );
		const int32_t sot = e.tokSot;
		WSP_CHECK( ctxDecode( cx, &sot, 1, 0, 1, WSP_DECODE_ALL_LOGITS, nullptr ) );
		std::vector<float> row( (size_t)n_langs );
		WSP_CUDA( cudaMemcpy( row.data(), cx.probs + ( e.tokSot + 1 ), (size_t)n_langs * 4, cudaMemcpyDeviceToHost ) );
		// the reference sorts (probability, id) descending, then takes a softmax OVER THE PROBABILITIES (sic), summing in that order
		std::vector<std::pair<float, int>> pid;
		for( int i = 0; i < n_langs; i++ ) pid.emplace_back( row[ (size_t)i ], i );
		std::stable_sort( pid.begin(), pid.end(), []( const std::pair<float, int>& a, const std::pair<float, int>& b ) { return a.first > b.first; } );
		float sum = 0;
		for( const auto& kv : pid ) sum += (float)exp( (double)kv.first );
		if( lang_probs )
			for( const auto& kv : pid ) lang_probs[ kv.second ] = (float)( exp( (double)kv.first ) / sum );
		*lang_id = pid[ 0 ].second;
		return WSP_OK;
	} );
}
wsp_status wsp_debug_set_encoder_layers( wsp_context* c, int32_t n )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	c->c->debugEncLayers = n;
	return WSP_OK;
}
wsp_status wsp_set_reference_threads( wsp_context* c, int32_t n )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	if( n < 0 || n > 16 ) return fail( WSP_E_INVALIDARG, "reference thread count must be in [0, 16]" );
	if( n != c->c->refThreads && c->c->stepGraph ) { cudaGraphExecDestroy( c->c->stepGraph ); c->c->stepGraph = nullptr; }
	c->c->refThreads = n;
	return WSP_OK;
}
wsp_status wsp_debug_step_timing( wsp_context* c, uint64_t* dst, int32_t cap )
{
	if( !c || !dst ) return fail( WSP_E_POINTER, "context/dst" );
	WSP_CUDA( cudaStreamSynchronize( c->c->stream ) );
	WSP_CUDA( cudaMemcpy( dst, c->c->megaTiming, sizeof( uint64_t ) * (size_t)( cap < 4608 ? cap : 4608 ), cudaMemcpyDeviceToHost ) );
	return WSP_OK;
}
wsp_status wsp_debug_set_step_mode( wsp_context* c, int32_t on )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	// 0 = one kernel per op, 1 = round 1's barrier kernel, 2 = dataflow kernel (default)
	if( on < 0 || on > 2 ) return fail( WSP_E_INVALIDARG, "step mode" );
	if( on != c->c->stepMode && c->c->stepGraph ) { cudaGraphExecDestroy( c->c->stepGraph ); c->c->stepGraph = nullptr; }
	c->c->stepMode = on;
	return WSP_OK;
}
wsp_status wsp_debug_enable_step_timing( wsp_context* c, int32_t on )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	if( ( on != 0 ) != c->c->stepTiming && c->c->stepGraph ) { cudaGraphExecDestroy( c->c->stepGraph ); c->c->stepGraph = nullptr; }
	c->c->stepTiming = on != 0;
	return WSP_OK;
}
wsp_status wsp_debug_set_graph( wsp_context* c, int32_t on )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	c->c->useGraph = on != 0;
	return WSP_OK;
}
wsp_status wsp_timings( wsp_context* c, float ms4[ 4 ], int32_t calls4[ 4 ], int32_t reset )
{
	if( !c ) return fail( WSP_E_POINTER, "context" );
	for( int i = 0; i < 4; i++ )
	{
		if( ms4 ) ms4[ i ] = c->c->ms[ i ];
		if( calls4 ) calls4[ i ] = c->c->calls[ i ];
		if( reset ) { c->c->ms[ i ] = 0; c->c->calls[ i ] = 0; }
	}
	return WSP_OK;
}

// pinned host memory for callers that want truly asynchronous H2D (bench.py's e2e leg)
void* wsp_host_alloc( size_t bytes )
{
	void* p = nullptr;
	if( cudaMallocHost( &p, bytes ) != cudaSuccess ) { cudaGetLastError(); return nullptr; }
	return p;
}
void wsp_host_free( void* p ) { if( p ) cudaFreeHost( p ); }

// ===================================================================================================================
// kernel-level test hooks
// ===================================================================================================================
static wsp_status requireSm100( int device )
{
	int count = 0;
	WSP_CUDA( cudaGetDeviceCount( &count ) );
	if( device < 0 || device >= count ) return fail( WSP_E_INVALIDARG, "no such CUDA device" );
	WSP_CUDA( cudaSetDevice( device ) );
	cudaDeviceProp prop;
	WSP_CUDA( cudaGetDeviceProperties( &prop, device ) );
	if( prop.major != 10 ) return fail( WSP_E_CUDA, "needs an sm_100a device" );
	return WSP_OK;
}

wsp_status wsp_test_gemm( int32_t device, int32_t M, int32_t N, int32_t K, const uint16_t* A, const uint16_t* B, float* D, int32_t bn, int32_t iters, float* ms )
{
	if( !A || !B || !D ) return fail( WSP_E_POINTER, "A/B/D" );
	if( M < 1 || N < 1 || K < 8 || ( K % 8 ) != 0 || ( bn != 128 && bn != 256 ) ) return fail( WSP_E_INVALIDARG, "shape (K must be a multiple of 8)" );
	WSP_CHECK( requireSm100( device ) );
	cudaDeviceProp prop;
	WSP_CUDA( cudaGetDeviceProperties( &prop, device ) );
	DevTmp<__half> dA, dB;
	DevTmp<float> dD;
	WSP_CUDA( dA.alloc( (size_t)M * K ) );
	WSP_CUDA( dB.alloc( (size_t)N * K ) );
	WSP_CUDA( dD.alloc( (size_t)M * N, true ) );
	WSP_CUDA( cudaMemcpy( dA.p, A, (size_t)M * K * 2, cudaMemcpyHostToDevice ) );
	WSP_CUDA( cudaMemcpy( dB.p, B, (size_t)N * K * 2, cudaMemcpyHostToDevice ) );
	gemm::Launch g;
	if( !gemm::makeMap2D( &g.mapA, dA.p, K, M, (uint64_t)K * 2, gemm::BM ) || !gemm::makeMap2D( &g.mapB, dB.p, K, N, (uint64_t)K * 2, bn ) )
		return fail( WSP_E_CUDA, "cuTensorMapEncodeTiled failed" );
	g.mapA2 = g.mapA;
	g.M = M; g.N = N; g.K = K;
	g.ep.M = M; g.ep.N = N; g.ep.ld = N; g.ep.out_f32 = dD.p;
	cudaEvent_t e0, e1;
	WSP_CUDA( cudaEventCreate( &e0 ) );
	WSP_CUDA( cudaEventCreate( &e1 ) );
	WSP_CUDA( gemm::launch( g, gemm::EPI_F32, gemm::A_PLAIN, bn, prop.multiProcessorCount, 0 ) );
	WSP_CUDA( cudaDeviceSynchronize() );
	if( iters > 0 )
	{
		WSP_CUDA( cudaEventRecord( e0 ) );
		for( int i = 0; i < iters; i++ ) WSP_CUDA( gemm::launch( g, gemm::EPI_F32, gemm::A_PLAIN, bn, prop.multiProcessorCount, 0 ) );
		WSP_CUDA( cudaEventRecord( e1 ) );
		WSP_CUDA( cudaDeviceSynchronize() );
		float t = 0;
		cudaEventElapsedTime( &t, e0, e1 );
		if( ms ) *ms = t / iters;
	}
	g_launchCount.fetch_add( (uint64_t)( 1 + ( iters > 0 ? iters : 0 ) ) );
	cudaEventDestroy( e0 ); cudaEventDestroy( e1 );
	WSP_CUDA( cudaMemcpy( D, dD.p, (size_t)M * N * 4, cudaMemcpyDeviceToHost ) );
	return WSP_OK;
}

__global__ void transpose_v_kernel( const __half* v, __half* vt, int T, int Tp )
{
	// v [BH][T][64] -> vt [BH][64][Tp]
	const int bh = blockIdx.y;
	const int t = blockIdx.x * blockDim.x + threadIdx.x;
	if( t >= T ) return;
	for( int e = 0; e < 64; e++ ) vt[ ( (size_t)bh * 64 + e ) * Tp + t ] = v[ ( (size_t)bh * T + t ) * 64 + e ];
}

wsp_status wsp_test_attention( int32_t device, int32_t BH, int32_t T, const uint16_t* Q, const uint16_t* K, const uint16_t* V, float* out, int32_t iters, float* ms )
{
	if( !Q || !K || !V || !out ) return fail( WSP_E_POINTER, "Q/K/V/out" );
	if( BH < 1 || T < 1 ) return fail( WSP_E_INVALIDARG, "shape" );
	WSP_CHECK( requireSm100( device ) );
	const int Tp = ( ( T + 127 ) / 128 ) * 128;
	const size_t n = (size_t)BH * T * 64;
	DevTmp<__half> dQ, dK, dV, dVt, dO;
	DevTmp<float> dOf;
	WSP_CUDA( dQ.alloc( n ) ); WSP_CUDA( dK.alloc( n ) ); WSP_CUDA( dV.alloc( n ) );
	WSP_CUDA( dVt.alloc( (size_t)BH * 64 * Tp, true ) );
	WSP_CUDA( dO.alloc( n, true ) ); WSP_CUDA( dOf.alloc( n ) );
	WSP_CUDA( cudaMemcpy( dQ.p, Q, n * 2, cudaMemcpyHostToDevice ) );
	WSP_CUDA( cudaMemcpy( dK.p, K, n * 2, cudaMemcpyHostToDevice ) );
	WSP_CUDA( cudaMemcpy( dV.p, V, n * 2, cudaMemcpyHostToDevice ) );
	transpose_v_kernel<<<dim3( ( T + 127 ) / 128, BH ), 128>>>( dV.p, dVt.p, T, Tp );
	CUtensorMap mq, mk, mv;
	if( !gemm::makeMap2D( &mq, dQ.p, 64, (uint64_t)BH * T, 128, 128 ) || !gemm::makeMap2D( &mk, dK.p, 64, (uint64_t)BH * T, 128, 128 ) ||
		!gemm::makeMap2D( &mv, dVt.p, Tp, (uint64_t)BH * 64, (uint64_t)Tp * 2, 64 ) )
		return fail( WSP_E_CUDA, "cuTensorMapEncodeTiled failed" );
	attn::EncParams p;
	// treat every (b,h) as its own "chunk" with one head: out layout [BH][T][64]
	p.T = T; p.H = 1; p.nBH = BH; p.d = 64; p.out = dO.p;
	p.scale_log2 = (float)( 0.125 * 1.4426950408889634 );
	WSP_CUDA( attn::launchEnc( mq, mk, mv, p, 0 ) );
	WSP_CUDA( cudaDeviceSynchronize() );
	if( iters > 0 )
	{
		cudaEvent_t e0, e1;
		WSP_CUDA( cudaEventCreate( &e0 ) ); WSP_CUDA( cudaEventCreate( &e1 ) );
		WSP_CUDA( cudaEventRecord( e0 ) );
		for( int i = 0; i < iters; i++ ) WSP_CUDA( attn::launchEnc( mq, mk, mv, p, 0 ) );
		WSP_CUDA( cudaEventRecord( e1 ) );
		WSP_CUDA( cudaDeviceSynchronize() );
		float t = 0;
		cudaEventElapsedTime( &t, e0, e1 );
		if( ms ) *ms = t / iters;
		cudaEventDestroy( e0 ); cudaEventDestroy( e1 );
	}
	g_launchCount.fetch_add( (uint64_t)( 2 + ( iters > 0 ? iters : 0 ) ) );
	half_to_float_kernel<<<(unsigned)( ( n + 255 ) / 256 ), 256>>>( dO.p, dOf.p, n );
	WSP_CUDA( cudaMemcpy( out, dOf.p, n * 4, cudaMemcpyDeviceToHost ) );
	return WSP_OK;
}

wsp_status wsp_test_skinny( int32_t device, int32_t nOut, int32_t K, int32_t cols, const uint16_t* W, const uint16_t* X, float* out, int32_t iters, float* ms )
{
	if( !W || !X || !out ) return fail( WSP_E_POINTER, "W/X/out" );
	if( nOut < 1 || K < 32 || K % 32 != 0 || cols < 1 ) return fail( WSP_E_INVALIDARG, "shape (K multiple of 32)" );
	WSP_CHECK( requireSm100( device ) );
	DevTmp<__half> dW, dX;
	DevTmp<float> dO;
	WSP_CUDA( dW.alloc( (size_t)nOut * K ) );
	WSP_CUDA( dX.alloc( (size_t)cols * K ) );
	WSP_CUDA( dO.alloc( (size_t)cols * nOut, true ) );
	WSP_CUDA( cudaMemcpy( dW.p, W, (size_t)nOut * K * 2, cudaMemcpyHostToDevice ) );
	WSP_CUDA( cudaMemcpy( dX.p, X, (size_t)cols * K * 2, cudaMemcpyHostToDevice ) );
	kern::SkinnyArgs a;
	a.W = dW.p; a.nOut = nOut; a.K = K; a.xF16 = dX.p; a.xStride = K; a.nCols = cols; a.epi = kern::SK_LOGITS; a.outF32 = dO.p; a.ld = nOut;
	WSP_CUDA( kern::skinnyGemm( a, 0 ) );
	WSP_CUDA( cudaDeviceSynchronize() );
	if( iters > 0 )
	{
		cudaEvent_t e0, e1;
		WSP_CUDA( cudaEventCreate( &e0 ) ); WSP_CUDA( cudaEventCreate( &e1 ) );
		WSP_CUDA( cudaEventRecord( e0 ) );
		for( int i = 0; i < iters; i++ ) WSP_CUDA( kern::skinnyGemm( a, 0 ) );
		WSP_CUDA( cudaEventRecord( e1 ) );
		WSP_CUDA( cudaDeviceSynchronize() );
		float t = 0;
		cudaEventElapsedTime( &t, e0, e1 );
		if( ms ) *ms = t / iters;
		cudaEventDestroy( e0 ); cudaEventDestroy( e1 );
	}
	g_launchCount.fetch_add( (uint64_t)( 1 + ( iters > 0 ? iters : 0 ) ) );
	WSP_CUDA( cudaMemcpy( out, dO.p, (size_t)cols * nOut * 4, cudaMemcpyDeviceToHost ) );
	return WSP_OK;
}

wsp_status wsp_test_layernorm( int32_t device, int32_t rows, int32_t d, const float* x, const float* gamma, const float* beta, uint16_t* out )
{
	if( !x || !gamma || !beta || !out ) return fail( WSP_E_POINTER, "x/gamma/beta/out" );
	WSP_CHECK( requireSm100( device ) );
	DevTmp<float> dx, dg, db;
	DevTmp<__half> dout;
	WSP_CUDA( dx.alloc( (size_t)rows * d ) ); WSP_CUDA( dg.alloc( d ) ); WSP_CUDA( db.alloc( d ) ); WSP_CUDA( dout.alloc( (size_t)rows * d ) );
	WSP_CUDA( cudaMemcpy( dx.p, x, (size_t)rows * d * 4, cudaMemcpyHostToDevice ) );
	WSP_CUDA( cudaMemcpy( dg.p, gamma, (size_t)d * 4, cudaMemcpyHostToDevice ) );
	WSP_CUDA( cudaMemcpy( db.p, beta, (size_t)d * 4, cudaMemcpyHostToDevice ) );
	WSP_CUDA( kern::layerNormF16( dx.p, dg.p, db.p, dout.p, rows, d, 0 ) );
	WSP_CUDA( cudaDeviceSynchronize() );
	g_launchCount.fetch_add( 1 );
	WSP_CUDA( cudaMemcpy( out, dout.p, (size_t)rows * d * 2, cudaMemcpyDeviceToHost ) );
	return WSP_OK;
}

// sampler alone: rows of hand-made logits -> softmax + the Whisper sampling rules (whisper_sample_best / _timestamp, whisper.cpp:1875-1964)
wsp_status wsp_test_sample( int32_t device, int32_t rows, int32_t n_vocab, const float* logits, const int32_t special4[ 4 ], int32_t force_timestamp,
	int32_t is_initial, float* probs, wsp_token_data* out )
{
	if( !logits || !special4 || !out ) return fail( WSP_E_POINTER, "logits/special/out" );
	if( rows < 1 || rows > 4096 || n_vocab < 8 ) return fail( WSP_E_INVALIDARG, "rows / n_vocab" );
	WSP_CHECK( requireSm100( device ) );
	static_assert( sizeof( wsp_token_data ) == sizeof( kern::TokenData ), "token data layout" );
	DevTmp<float> dl, dp;
	DevTmp<int> dflags, dscratch;
	DevTmp<kern::TokenData> dout;
	WSP_CUDA( dl.alloc( (size_t)rows * n_vocab ) ); WSP_CUDA( dp.alloc( (size_t)rows * n_vocab ) ); WSP_CUDA( dflags.alloc( 2 ) ); WSP_CUDA( dout.alloc( rows ) );
	WSP_CUDA( cudaMemcpy( dl.p, logits, (size_t)rows * n_vocab * 4, cudaMemcpyHostToDevice ) );
	const int fl[ 2 ] = { force_timestamp ? 1 : 0, is_initial ? 1 : 0 };
	WSP_CUDA( cudaMemcpy( dflags.p, fl, sizeof( fl ), cudaMemcpyHostToDevice ) );
	kern::SampleArgs sa;
	sa.logits = dl.p; sa.probs = dp.p; sa.B = rows; sa.nVocab = n_vocab;
	sa.tokenBeg = special4[ 0 ]; sa.tokenSot = special4[ 1 ]; sa.tokenSolm = special4[ 2 ]; sa.tokenNot = special4[ 3 ];
	sa.dForceTs = dflags.p; sa.out = dout.p; sa.N = 1;
	WSP_CUDA( dscratch.alloc( (size_t)rows * ( (size_t)n_vocab + 1024 ) ) );
	sa.tieScratch = dscratch.p;
	WSP_CUDA( kern::sampleGreedy( sa, 0 ) );
	WSP_CUDA( cudaDeviceSynchronize() );
	g_launchCount.fetch_add( 2 );
	WSP_CUDA( cudaMemcpy( out, dout.p, (size_t)rows * sizeof( wsp_token_data ), cudaMemcpyDeviceToHost ) );
	if( probs ) WSP_CUDA( cudaMemcpy( probs, dp.p, (size_t)rows * n_vocab * 4, cudaMemcpyDeviceToHost ) );
	return WSP_OK;
}

} // extern "C"
