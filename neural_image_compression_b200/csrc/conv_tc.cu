// tcgen05 / TMEM / TMA arm of the conv engine (NIC_PREC_BF16): implicit-GEMM convolution on the 5th-gen
// tensor cores of sm_100a, bf16 operands, fp32 accumulation in tensor memory.
//
// Formulation (conv_common.cuh): out[pixels, c_out] = sum over taps, c_in of shifted-input . W_tap.
//
// conv_tc_kernel - one persistent CTA per SM, 11 warps:
//   warp 0   A producer   TMA (cp.async.bulk.tensor.4d) loads of input PATCHES: for an output tile of 16 x 16 pixels (two
//                         M = 128 blocks of 16 rows x 8 pixels side by side) the (16 + halo) x (16 + halo) input pixels of
//                         one 64-channel chunk land ONCE in shared memory (128-byte swizzle, one 128 B row per pixel);
//                         stride-2 convs load the four even/odd "planes" of the input with TMA element strides of 2.
//                         Conv zero padding is the TMA out-of-bounds fill.
//   warp 1   B producer   TMA loads of the [c_out tile x 64] weight slab of each (tap, chunk) into a 4-8 deep ring (both
//                         blocks of the tile share it); layers with c_out <= 16 keep ALL their slabs resident instead.
//   warp 2   MMA issuer   the warp walks the loop uniformly (operands in uniform registers), one elected lane issues
//                         tcgen05.mma (M = 128, N = c_out tile, K = 16) for every tap straight from the patch: the A
//                         descriptor of tap (dy, dx) starts at patch pixel (dy, dx) and walks 16 groups of 8 consecutive
//                         pixels with a stride of one patch row - no im2col copy, every input byte is read from L2 once
//                         per chunk instead of once per tap (basis: tools/tc_probe.cu T2/T2b, profiles/r1_tc_probe.txt).
//   warps 3-10 epilogue   tcgen05.ld the accumulator (double-buffered in TMEM: 4 x 128 columns, so the next tile's MMAs
//                         overlap), add bias, LeakyReLU, or GDN / IGDN: x stays in registers, its squares go to shared
//                         memory as a bf16 K-major tile, a second tcgen05.mma against the resident gamma OVERWRITES the
//                         accumulator in place and the epilogue applies x * rsqrt(beta + .) (or sqrt) - the GDN of
//                         Components.py:11-15, 40-44 never touches HBM.  bf16 NHWC outputs are staged in shared memory
//                         and leave through TMA tensor stores (element strides 2 interleave transposed-conv phases).
// Special forms: ConvTranspose2d = stride^2 phase convs of a stride-1 kernel; ConvTranspose2d(128 -> 3) = ONE 3x3 conv to
// 4 x 3 sub-pixel channels (N = 16); 1x1 convs walk a flat pixel list.
//
// conv_first_tc_kernel - Conv2d(3, 128, 5, s2) + GDN from the NCHW fp32 image (K = 75: im2col built by producer warps).
//
// Activations are NHWC bf16 between layers (c_in a multiple of 64).
#include <cuda.h>
#include <stdlib.h>

#include "conv_common.cuh"
#include "tc_host.cuh"
#include "tc_primitives.cuh"

namespace nic {

using namespace tc;

void set_trace_buffer(void* p);
// conv_simt.cu
int conv_fwd_fp32(const nic_conv_desc*, const void*, const void*, const float*, const void*, const float*, void*, void*, size_t, cudaStream_t);
int gdn_fwd_fp32(const float* x, int n, int c, int h, int w, int layout, int inverse, const float* gamma, const float* beta, float* y, cudaStream_t st);
int gdn_fwd_fp32_split(const float* x, int n, int c, int h, int w, int inverse, const float* gamma, const float* beta, void* y, cudaStream_t st);
int conv_fwd_fp32_ex(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias, void* y, int out_bf16_nhwc,
                     cudaStream_t st);

// x3_tc.cu
int pack_gdn_x3(int32_t c, float beta_min, const float* beta_raw, const float* gamma_raw, float* beta_eff, void* gamma_packed, cudaStream_t st);
int gdn_fwd_tc_x3(const void* x, int pair_in, long npix, int c, int inverse, const void* gamma_packed, const float* beta_eff, void* y, cudaStream_t st);
size_t packed_first_x3_elems(int cout);
int pack_first_x3(const float* w_ref, void* w_packed, int cout, cudaStream_t st);
int conv_first_x3(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias, float* y, cudaStream_t st);
int conv_first_gdn_x3(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias, const void* gamma_packed,
                      const float* beta_eff, void* y, cudaStream_t st);

// last_tc.cu
bool last_scatter_applies(const nic_conv_desc* d);
size_t packed_last_scatter_elems(int cin);
int pack_last_scatter(const float* w_ref, void* w_packed, int cin, cudaStream_t st);
int conv_last_scatter_x3(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias, void* y, cudaStream_t st);

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

void* g_trace_buffer = nullptr;   // set through nic_debug_set_trace (timing experiments; not part of the product ABI surface)

int* status_word() {       // one device int per DEVICE: the kernels' "a bounded wait expired" flag
  static int* d[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  if (!d[dev]) { if (cudaMalloc(&d[dev], sizeof(int)) != cudaSuccess) return nullptr; cudaMemset(d[dev], 0, sizeof(int)); }
  return d[dev];
}

int encode_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {inner * 2};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled(2d %llu x %llu, box %u x %u) failed: %d", (unsigned long long)inner,
                                     (unsigned long long)rows, box_inner, box_rows, (int)r);
  return NIC_OK;
}

// 2-D row-major tensor of 2-byte (bf16) or 4-byte (f32) elements, 128-byte swizzled boxes (box_inner * elem_bytes = 128)
int encode_2d_ex(CUtensorMap* m, const void* base, int elem_bytes, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {inner * elem_bytes};
  cuuint32_t box[2] = {box_inner, box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims,
                   strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled(2d %llu x %llu, box %u x %u, %d B) failed: %d", (unsigned long long)inner,
                                     (unsigned long long)rows, box_inner, box_rows, elem_bytes, (int)r);
  return NIC_OK;
}

// NCHW f32 image [n][c][h][w] viewed as a 3-D tensor (w, h, n * c): boxes of box_w x box_h x c floats, no swizzle, zero fill
// outside the image (the conv padding of the first layer)
int encode_image_patch(CUtensorMap* m, const void* base, int n, int c, int h, int w, int box_w, int box_h) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n * c};
  cuuint64_t strides[2] = {(cuuint64_t)w * 4, (cuuint64_t)w * h * 4};
  cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)c};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled(image %dx%dx%dx%d, box %dx%d) failed: %d", n, c, h, w, box_w, box_h, (int)r);
  return NIC_OK;
}

int encode_nhwc(CUtensorMap* m, const void* base, int n, int h, int w, int c, int box_w, int box_h, int stride, int elem_bytes) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t eb = elem_bytes;
  cuuint64_t dims[4] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)c * eb, (cuuint64_t)w * c * eb, (cuuint64_t)h * w * c * eb};
  cuuint32_t box[4] = {(cuuint32_t)(128 / elem_bytes), (cuuint32_t)(box_w * stride), (cuuint32_t)(box_h * stride), 1};   // 128-byte rows
  cuuint32_t es[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  CUresult r = enc(m, elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled(nhwc %dx%dx%dx%d, box %dx%d stride %d) failed: %d", n, h, w, c, box_w,
                                     box_h, stride, (int)r);
  return NIC_OK;
}

// 2-D row-major bf16 tensor, boxes of 32 elements (64-byte rows, SWIZZLE_64B) x box_rows
int encode_2d_c32(CUtensorMap* m, const void* base, uint64_t inner, uint64_t rows, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {inner * 2};
  cuuint32_t box[2] = {32, box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled(2d %llu x %llu, 32-column box x %u) failed: %d", (unsigned long long)inner,
                                     (unsigned long long)rows, box_rows, (int)r);
  return NIC_OK;
}

// NHWC bf16 tensor, boxes of 32 channels (64-byte rows, SWIZZLE_64B: 16-byte chunk ^= (row >> 1) & 3) x box_w x box_h pixels,
// every stride-th pixel in w and h (the output phases of a transposed conv)
int encode_nhwc_c32(CUtensorMap* m, const void* base, int n, int h, int w, int c, int box_w, int box_h, int stride) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[4] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2};
  cuuint32_t box[4] = {32, (cuuint32_t)(box_w * stride), (cuuint32_t)(box_h * stride), 1};
  cuuint32_t es[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(NIC_E_CUDA, "cuTensorMapEncodeTiled(nhwc %dx%dx%dx%d, 32-channel box %dx%d) failed: %d", n, h, w, c, box_w, box_h, (int)r);
  return NIC_OK;
}


namespace {

constexpr int kTileH = 16, kTileW = 8;          // output pixels per M = 128 block: 16 groups of 8
constexpr int kMaxSlots = 4;
constexpr int kMaxBSlots = 8;
constexpr int kEpiWarps = 8;
constexpr int kMmaWarps = 2;                    // one MMA-issuing warp per M = 128 block of the tile (see the MMA issuer below)
constexpr int kFirstEpiWarp = 2 + kMmaWarps;
constexpr int kThreads = (kFirstEpiWarp + kEpiWarps) * 32;
constexpr int kMaxDynSmem = 232448 - 8192;    // 227 KB opt-in limit minus this kernel's static shared memory
constexpr int kMaxCout = 1792;                // bias table staged in shared memory (M = 192, K = 3: 1728 channels)

struct TcTap { int8_t plane, roff, coff, slab; };
struct TcPhase {
  int8_t py, px, nplanes, pad0;
  int8_t plane_ph[4], plane_pw[4], plane_dymin[4], plane_dxmin[4];
  int8_t plane_tap_begin[5];                   // taps of plane p: [plane_tap_begin[p], plane_tap_begin[p+1]) into taps[]
};

struct TcParams {
  TcPhase phases[kMaxPhases];
  TcTap taps[kMaxTaps];
  int nphases, in_stride, out_stride;
  int n, hin, win, cin, cout, hout, wout;
  int hp, wp;                                  // per-phase output grid
  int mt;                                      // M = 128 blocks per tile (1 or 2): the blocks share every weight slab
  int blk_roff[2], blk_coff[2];                // position of block b inside the tile (pixels)
  int tile_h, tile_w;                          // output pixels per tile
  int tiles_x, tiles_y, n_ntiles, total_tiles;
  int b_slot_bytes;                            // stride of the weight ring: 16 KB (a 128-row slab), 8 KB in pair mode (64 rows per CTA)
  int pair;                                    // conv_tc_kernel<true>: clusters of two CTAs, cta_group::2 MMAs
  int chunk_perm;                              // bf16x3: K chunks c-slice by c-slice (kchunk in the kernel)
  int tail_first, tail_n;                      // last wave in half tiles: first virtual slot, number of tiles split (0 = off)
  int nt_inner;                                // N tile innermost in the tile order (decode_tile)
  int pos_per_wave, spatial_tiles;             // phase-interleaved tile order (decode_tile); pos_per_wave = 0: phase-major
  int nchunks;                                 // K chunks of 64 (cin / 64; 3 cin / 64 in the bf16x3 arm)
  int a_chunk_mod;                             // input channel chunk of K chunk c is c % a_chunk_mod (bf16x3: [hi | lo | hi again])
  const int* lo_flag;                          // bf16x3, optional device flag: 0 = the lo half of the input pair tensor is all zero
                                               // (integer-valued symbols, Models.py:63-64) -> the lo . W_hi chunks are skipped
  int split_out;                               // bf16-pair output: hi to the channel window of the first half of the tensor,
  int split_lo_off;                            //   lo to the same window shifted by split_lo_off channels (the second half)
  int ph_rows, pw_cols;                        // patch rows / cols (pixels)
  int slot_bytes, nsa, nsb;
  int swap;                                    // operand roles swapped: weights are the M = 128 operand, the 256 pixels of the tile
                                               // (two vertically stacked blocks) the N = 256 operand; accumulator [c_out lanes][pixel
                                               // columns] - 6 KB of shared-memory operand reads per 128x128x16 instead of 8 KB
  int b_resident;                              // all weight slabs of the layer stay in shared memory (small c_out)
  int nslabs;                                  // taps over all phases
  int nb, cout_pad;                            // N of the MMA (c_out tile), padded c_out of the packed weights
  int epilogue;
  int out_dtype;                               // NIC_DT_*
  long ys_n, ys_c, ys_h, ys_w;                 // output strides (elements), channel offset already applied to y
  int flat_hw;                                 // > 0: 1x1 conv over a flattened pixel list; pixel p -> image p / flat_hw
  int stage2;                                  // bf16-pair output with TWO staging tiles (hi tile, lo tile): no store is waited for
                                               // right after it was issued (layers whose mainloop is as short as their epilogue)
  int epi_slices;                              // bf16-pair output, normal orientation: per-warp staging slices and stores
                                               // (epilogue_block_slices) instead of the CTA-wide rounds of epilogue_block
  int tma_out;                                 // NHWC output leaves through shared memory + TMA tensor stores: 1 = bf16 (two
                                               // [128 px][64 ch] panels), 2 = f32 (four [128 px][32 ch] panels)
  int out_c_offset;                            // channel window start inside the output tensor (TMA coordinates)
  int shuffle_cout;                            // > 0: sub-pixel (2x2) output: column n = (py * 2 + px) * shuffle_cout + c goes to
                                               //      pixel (2 oy + py, 2 ox + px), channel c of an fp32 tensor (ConvTranspose2d to RGB)
  int bias_mod;                                // bias index = column % bias_mod (shuffle) ; 0 = plain
  int dbg;                                     // NIC_TC_DEBUG bits (timing experiments only): 1 skip gamma MMA, 2 skip tensor store, 4 skip direct stores, 8 skip the epilogue
  long long* dbg_times;                        // NIC_TC_TRACE: [cta][16 tiles][16] clock64 stamps of the pipeline roles (null = off)
  const float* bias;
  const float* beta;
  void* y;
  int* status;
  // shared-memory carve-up (byte offsets from the 1024-aligned base)
  int off_a, off_b, off_gamma, off_sq, smem_bytes;
};

struct __align__(8) TcBarriers {
  uint64_t a_full[kMaxSlots], a_empty[kMaxSlots], b_full[kMaxBSlots], b_empty[kMaxBSlots];
  uint64_t acc_full[2], acc_empty[2], gdn_full, gamma_full, bres_full;
  uint32_t tmem_base;
  volatile int abort_flag;
};

__device__ __forceinline__ bool wait_or_abort(uint64_t* bar, uint32_t parity, TcBarriers* sb, int* status) {
  for (uint32_t i = 0; i < (1u << 22); ++i) {
    if (mbar_try_wait(bar, parity)) return true;
    if ((i & 255u) == 255u && sb->abort_flag) return false;
  }
  sb->abort_flag = 1;
  atomicExch(status, 1);
  return false;
}

__device__ __forceinline__ void trace(const TcParams& p, uint32_t tile_iter, int slot) {
  if (p.dbg_times && tile_iter < 16) {
    p.dbg_times[(static_cast<long>(blockIdx.x) * 32 + tile_iter) * 16 + slot] = clock64();
    if (slot == 0) {          // wall-clock ns beside the cycle stamp: their ratio is the SM clock the kernel actually ran at
      unsigned long long ns;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
      p.dbg_times[(static_cast<long>(blockIdx.x) * 32 + tile_iter) * 16 + 15] = static_cast<long long>(ns);
    }
  }
}

// a value (not a clock) into the same trace record: the phase of the tile, for tools/trace_layer.py's per-phase summary
__device__ __forceinline__ void trace_value(const TcParams& p, uint32_t tile_iter, int slot, long long value) {
  if (p.dbg_times && tile_iter < 16) p.dbg_times[(static_cast<long>(blockIdx.x) * 32 + tile_iter) * 16 + slot] = value;
}

// Tile order.  Default: x, y, image, phase, N tile (phase-major: consecutive tiles cost the same, the static round robin over
// the CTAs is balanced).  Transposed convs whose input does not fit L2 use a phase-interleaved order instead (pos_per_wave != 0):
// consecutive slots are the phases (x N tiles) of ONE spatial tile, so the input patch a phase reads is in L2 from its sibling
// phases (phase-major re-read the whole input from DRAM once per phase: g_s layer 3, 809 MB for a 201 MB input), and the phase of
// a slot is rotated by its position so that every CTA still cycles through the cheap and the expensive phases.
// Returns false for the unused slots of the last wave of the pair form (always a CTA's last iteration).
__device__ __forceinline__ bool decode_tile(const TcParams& p, int tile, int& ntile, int& phase, int& img, int& ty, int& tx) {
  if (p.pair && (p.pos_per_wave || p.n_ntiles > 1)) {
    // CTA pairs: cluster slot u = tile / 2 is variant u % V (V = phases x N tiles) of the pair of adjacent spatial tiles u / V - the
    // two CTAs of a cluster share phase and N tile (the weights), consecutive clusters cover the variants of one input region;
    // in the interleaved order the phase is rotated by the position so that a cluster keeps cycling through the phases
    const int V = p.nphases * p.n_ntiles;
    const int u = tile >> 1, pp = u / V, v = u - pp * V;
    int s = 2 * pp + (tile & 1);
    if (s >= p.spatial_tiles) return false;
    ntile = v % p.n_ntiles;
    phase = (v / p.n_ntiles + (p.pos_per_wave ? pp : 0)) % p.nphases;
    tx = s % p.tiles_x; s /= p.tiles_x;
    ty = s % p.tiles_y; img = s / p.tiles_y;
    return true;
  }
  if (p.pos_per_wave) {
    // one-CTA form: slot u is variant u % V (V = phases x N tiles) of spatial tile u / V, the phase rotated by the position so that
    // a CTA (u = c + wave x grid) keeps cycling through the phases; consecutive CTAs work on the V variants of one input region
    const int V = p.nphases * p.n_ntiles;
    int s = tile / V;
    const int v = tile - s * V;
    ntile = v % p.n_ntiles;
    phase = (v / p.n_ntiles + s) % p.nphases;
    tx = s % p.tiles_x; s /= p.tiles_x;
    ty = s % p.tiles_y; img = s / p.tiles_y;
    return true;
  }
  if (p.tail_n && tile >= p.tail_first) {   // last wave in half tiles (tail_block): slot k -> its tile
    const int k = tile - p.tail_first;
    tile = p.tail_first + (p.pair ? ((k >> 2) << 1) + (k & 1) : k >> 1);
  }
  if (p.nt_inner) {                       // N tile innermost: the CTAs of one wave share their input tiles, not their weights
    ntile = tile % p.n_ntiles; tile /= p.n_ntiles;
    tx = tile % p.tiles_x; tile /= p.tiles_x;
    ty = tile % p.tiles_y; tile /= p.tiles_y;
    img = tile % p.n; phase = tile / p.n;
    return true;
  }
  tx = tile % p.tiles_x; tile /= p.tiles_x;
  ty = tile % p.tiles_y; tile /= p.tiles_y;
  img = tile % p.n; tile /= p.n;
  phase = tile % p.nphases; tile /= p.nphases;
  ntile = tile;
  return true;
}

// Last wave in half tiles: when the tiles left over after the full waves would occupy fewer than half of the CTAs (g_a layer 2:
// 1536 tiles = 10 waves of 148 + 56), each of them is done as two one-block slots on two CTAs (pair form: on two clusters) - the
// layer ends after 10.5 tile times instead of 11.  Returns the block a slot computes, or -1 for a whole tile.
__device__ __forceinline__ int tail_block(const TcParams& p, int tile) {
  if (!p.tail_n || tile < p.tail_first) return -1;
  const int k = tile - p.tail_first;
  return p.pair ? (k >> 1) & 1 : k & 1;
}

// number of M blocks of the tile that contain at least one real output pixel
__device__ __forceinline__ int live_blocks(const TcParams& p, int ty, int tx) {
  int nblk = 0;
  for (int b = 0; b < p.mt; ++b)
    if (ty * p.tile_h + p.blk_roff[b] < p.hp && tx * p.tile_w + p.blk_coff[b] < p.wp) nblk = b + 1;
  return nblk;
}

__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

// one 32-channel group of one pixel to global memory
__device__ __forceinline__ void store_group(const TcParams& p, long obase, int c0, const float* v) {
  if (p.ys_c == 1 && c0 + 32 <= p.cout) {
    if (p.out_dtype == NIC_DT_BF16) {
      uint4* dst = reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(p.y) + obase + c0);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        dst[j] = make_uint4(pack_bf16x2(v[j * 8], v[j * 8 + 1]), pack_bf16x2(v[j * 8 + 2], v[j * 8 + 3]),
                            pack_bf16x2(v[j * 8 + 4], v[j * 8 + 5]), pack_bf16x2(v[j * 8 + 6], v[j * 8 + 7]));
    } else {
      float4* dst = reinterpret_cast<float4*>(static_cast<float*>(p.y) + obase + c0);
#pragma unroll
      for (int j = 0; j < 8; ++j) dst[j] = make_float4(v[j * 4], v[j * 4 + 1], v[j * 4 + 2], v[j * 4 + 3]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const int c = c0 + j;
      if (c < p.cout) {
        if (p.out_dtype == NIC_DT_BF16) static_cast<__nv_bfloat16*>(p.y)[obase + c * p.ys_c] = __float2bfloat16_rn(v[j]);
        else static_cast<float*>(p.y)[obase + c * p.ys_c] = v[j];
      }
    }
  }
}

// columns n = (py * 2 + px) * SC + c of one input pixel -> the 2 x 2 output pixels it owns, SC channels, fp32
template <int SC>
__device__ __forceinline__ void store_subpixel(const TcParams& p, float* yb, const float* v) {
#pragma unroll
  for (int c = 0; c < SC; ++c)
#pragma unroll
    for (int yy = 0; yy < 2; ++yy) {
      float* dst = yb + c * p.ys_c + yy * p.ys_h;
      const float a = v[(yy * 2) * SC + c], b = v[(yy * 2 + 1) * SC + c];
      if (p.ys_w == 1 && (reinterpret_cast<uintptr_t>(dst) & 7) == 0) *reinterpret_cast<float2*>(dst) = make_float2(a, b);
      else { dst[0] = a; dst[p.ys_w] = b; }
    }
}

__device__ __forceinline__ float rsqrt_approx(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Epilogue of one M = 128 accumulator block: bias, LeakyReLU or the fused GDN / IGDN, then the store (TMA tensor store of a
// bf16 NHWC tile staged in shared memory, or direct stores).  NW = 4 or 8 epilogue warps; thread <-> accumulator row <->
// pixel; with 8 warps the second warpgroup (hs = 1) takes channels 64..127 of the same rows, i.e. the other 64-channel half
// of the squares / staging tile.  Returns false when a bounded wait expired.
// KEEPX = true: x stays in registers and the gamma contraction overwrites the accumulator in place (no extra TMEM);
// KEEPX = false: the contraction goes to `gdn_tmem` and x is read from the accumulator a second time (fewer registers).
template <int NW, bool KEEPX = true>
__device__ __forceinline__ bool epilogue_block(const TcParams& p, TcBarriers* sb, const float* s_bias, const float* s_beta, uint8_t* sq,
                                               const uint8_t* gamma_smem, const CUtensorMap* map_o_ptr, uint32_t acc_tmem, int q, int lane,
                                               int hs, bool leader, int img, int oy0, int ox0, int py, int px, int cbase, uint32_t& gdn_count,
                                               uint32_t trace_tile = 0xffffffffu, int trace_base = 8, int bar_id = 1,
                                               uint64_t* gdn_bar = nullptr, uint32_t gdn_tmem = 0) {
  if (!gdn_bar) gdn_bar = &sb->gdn_full;
  if (KEEPX) gdn_tmem = acc_tmem;
  const uint32_t gdn_addr = gdn_tmem + (static_cast<uint32_t>(q * 32) << 16);
  constexpr int NG = (NW == 8) ? 2 : 4;                     // 32-channel groups per thread in the 128-wide paths
  const bool gdn = p.epilogue == NIC_EPI_GDN || p.epilogue == NIC_EPI_IGDN;
  const bool igdn = p.epilogue == NIC_EPI_IGDN;
  const int ncg = (p.nb + 31) / 32;
  const int cg0 = (NW == 8) ? hs * 2 : 0;                   // first channel group of this thread
  const int row = q * 32 + lane, g = row >> 3, c8 = row & 7;
  const uint32_t acc_addr = acc_tmem + (static_cast<uint32_t>(q * 32) << 16);
  const int oy = oy0 + g, ox = ox0 + c8;
  const int out_y = oy * p.out_stride + py, out_x = ox * p.out_stride + px;
  const bool valid = oy < p.hp && ox < p.wp && out_y < p.hout && out_x < p.wout;
  long obase;
  if (p.flat_hw > 0) {
    const long pix = static_cast<long>(oy) * kTileW + ox;
    obase = (pix / p.flat_hw) * p.ys_n + (pix % p.flat_hw) * p.ys_w;
  } else {
    obase = img * p.ys_n + static_cast<long>(out_y) * p.ys_h + static_cast<long>(out_x) * p.ys_w;
  }
  auto epi_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(NW * 32) : "memory"); };
  if (p.tma_out) {
    // the staging tile (= the squares tile) may still be read by the previous block's tensor store; with two staging tiles
    // the hi tile was handed to the store BEFORE the most recent one (the previous block's lo store)
    if (leader) { if (p.stage2) tma_store_wait_read_1(); else tma_store_wait_read(); }
    epi_sync();
  }
  uint8_t* stg = sq;                                        // staging tile of the current pass
  if (leader) trace(p, trace_tile, trace_base + 0);
  float xr[KEEPX ? NG * 32 : 32];
  if (gdn) {
    // x (+ bias) stays in registers; its squares go to shared memory as the bf16 K-major A operand of the
    // gamma contraction, whose result OVERWRITES this accumulator (no extra TMEM); then y = x * rsqrt(beta + .)
    if (KEEPX) {      // all of this thread's accumulator columns in flight at once, one wait
#pragma unroll
      for (int i = 0; i < NG; ++i) tmem_ld_32x32(acc_addr + (cg0 + i) * 32, xr + i * 32);
      tmem_ld_wait();
    }
#pragma unroll
    for (int i = 0; i < NG; ++i) {
      const int cg = cg0 + i;
      if (!KEEPX) {
        tmem_ld_32x32(acc_addr + cg * 32, xr);
        tmem_ld_wait();
      }
      uint8_t* half = sq + (cg >> 1) * (128 * 128) + row * 128;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t w[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int l = (KEEPX ? i * 32 : 0) + j * 8 + e * 2, c0 = cg * 32 + j * 8 + e * 2;
          const float a = xr[l] + s_bias[c0], bb = xr[l + 1] + s_bias[c0 + 1];
          xr[l] = a; xr[l + 1] = bb;
          w[e] = pack_bf16x2(a * a, bb * bb);
        }
        const int chunk = ((cg & 1) * 4 + j) ^ (row & 7);
        *reinterpret_cast<uint4*>(half + chunk * 16) = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
    fence_proxy_async_smem();
    tcgen05_fence_before();
    if (leader) trace(p, trace_tile, trace_base + 1);
    epi_sync();
    if (leader) trace(p, trace_tile, trace_base + 2);
    if (leader && !(p.dbg & 1)) {
      if (gdn_count == 0) wait_or_abort(&sb->gamma_full, 0, sb, p.status);
      tcgen05_fence_after();
      const uint32_t idg = umma_idesc_bf16(128, 128);
      const uint32_t hi = umma_desc_hi(1024);
      const uint32_t sq_lo = umma_desc_lo(smem_u32(sq)), g_lo = umma_desc_lo(smem_u32(gamma_smem));
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const uint32_t off = ((k >> 2) * (128 * 128) + (k & 3) * 32) >> 4;
        umma_bf16_lohi(gdn_tmem, sq_lo + off, hi, g_lo + off, hi, idg, k);
      }
      umma_commit(gdn_bar);
    }
    if (!(p.dbg & 1)) {
      if (!__all_sync(0xffffffffu, wait_or_abort(gdn_bar, gdn_count & 1, sb, p.status))) return false;
    }
    ++gdn_count;
    tcgen05_fence_after();
    if (leader) trace(p, trace_tile, trace_base + 3);
  }
  const int nvalid_c = p.cout - cbase;                      // channels of this N tile that exist
  auto emit_group = [&](int cg, const float* v) {             // one pixel x 32 channels: to the staging tile or to HBM
    if (p.tma_out == 2) {
      uint8_t* panel = sq + cg * (128 * 128) + row * 128;       // f32: one 128-byte row per pixel and 32-channel group
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *reinterpret_cast<float4*>(panel + ((j ^ (row & 7)) << 4)) = make_float4(v[j * 4], v[j * 4 + 1], v[j * 4 + 2], v[j * 4 + 3]);
    } else if (p.tma_out) {
      uint8_t* half = stg + (cg >> 1) * (128 * 128) + row * 128;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int chunk = ((cg & 1) * 4 + j) ^ (row & 7);
        *reinterpret_cast<uint4*>(half + chunk * 16) =
            make_uint4(pack_bf16x2(v[j * 8], v[j * 8 + 1]), pack_bf16x2(v[j * 8 + 2], v[j * 8 + 3]),
                       pack_bf16x2(v[j * 8 + 4], v[j * 8 + 5]), pack_bf16x2(v[j * 8 + 6], v[j * 8 + 7]));
      }
    } else if (valid && !(p.dbg & 4)) {
      if (p.shuffle_cout > 0) {
        // sub-pixel scatter: this thread's input pixel (oy, ox) owns output pixels (2 oy + {0,1}, 2 ox + {0,1})
        float* yb = static_cast<float*>(p.y) + img * p.ys_n + static_cast<long>(2 * oy) * p.ys_h + static_cast<long>(2 * ox) * p.ys_w;
        switch (p.shuffle_cout) {
          case 1: store_subpixel<1>(p, yb, v); break;
          case 2: store_subpixel<2>(p, yb, v); break;
          case 3: store_subpixel<3>(p, yb, v); break;
          default: store_subpixel<4>(p, yb, v); break;
        }
      } else {
        store_group(p, obase, cbase + cg * 32, v);
      }
    }
  };
  if (gdn) {
    if (KEEPX && NG == 2) {
      // both 32-column groups of the contraction in flight at once
      float v0[32], v1[32];
      tmem_ld_32x32(gdn_addr + cg0 * 32, v0);
      tmem_ld_32x32(gdn_addr + (cg0 + 1) * 32, v1);
      tmem_ld_wait();
      if (igdn) {
#pragma unroll
        for (int j = 0; j < 32; ++j) { v0[j] = xr[j] * sqrt_approx(v0[j] + s_beta[cg0 * 32 + j]); v1[j] = xr[32 + j] * sqrt_approx(v1[j] + s_beta[cg0 * 32 + 32 + j]); }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) { v0[j] = xr[j] * rsqrt_approx(v0[j] + s_beta[cg0 * 32 + j]); v1[j] = xr[32 + j] * rsqrt_approx(v1[j] + s_beta[cg0 * 32 + 32 + j]); }
      }
      emit_group(cg0, v0);
      emit_group(cg0 + 1, v1);
    } else {
#pragma unroll
      for (int i = 0; i < NG; ++i) {
        const int cg = cg0 + i;
        float v[32];
        tmem_ld_32x32(gdn_addr + cg * 32, v);
        if (!KEEPX) {
          tmem_ld_32x32(acc_addr + cg * 32, xr);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) xr[j] += s_bias[cg * 32 + j];
        } else {
          tmem_ld_wait();
        }
        const float* xp = xr + (KEEPX ? i * 32 : 0);
        if (igdn) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = xp[j] * sqrt_approx(v[j] + s_beta[cg * 32 + j]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = xp[j] * rsqrt_approx(v[j] + s_beta[cg * 32 + j]);
        }
        emit_group(cg, v);
      }
    }
  } else {
    // channel groups of this warpgroup: with 8 warps the second one takes the upper half of the groups
    const int per = (NW == 8) ? (ncg + 1) / 2 : ncg;
    const int first = (NW == 8) ? hs * per : 0;
    const int last = (first + per < ncg) ? first + per : ncg;
    const int npass = p.split_out ? 2 : 1;         // bf16-pair output: one staging + store round for hi, one for lo
    for (int pass = 0; pass < npass; ++pass) {
      if (pass == 1) {
        // hand the staging tile from the hi round to the lo round
        fence_proxy_async_smem();
        epi_sync();
        if (leader) {
          const int wc = ox0 * p.out_stride + px, hc = oy0 * p.out_stride + py;
          for (int h = 0; h < 2; ++h)
            if (h * 64 < nvalid_c) tma_store_4d(map_o_ptr, sq + h * (128 * 128), p.out_c_offset + cbase + h * 64, wc, hc, img);
          tma_store_commit();
          // one tile: wait for this store; two tiles: the lo tile was handed to the store before this one (previous block)
          if (p.stage2) tma_store_wait_read_1(); else tma_store_wait_read();
        }
        if (p.stage2) stg = sq + 2 * 128 * 128;
        epi_sync();
      }
      for (int cg = first; cg < last; ++cg) {
        float v[32];
        tmem_ld_32x32(acc_addr + cg * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int c = cbase + cg * 32 + j;
          float x = v[j] + (c < p.cout ? s_bias[c] : 0.f);
          if (p.epilogue == NIC_EPI_LRELU) x = x > 0.f ? x : 0.01f * x;
          v[j] = x;
        }
        if (pass == 1) {        // lo = x - bf16(x), through packed conversions (single-value F2F is a 16 / clk / SM instruction)
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const uint32_t h = pack_bf16x2(v[j], v[j + 1]);
            v[j] -= __uint_as_float(h << 16);
            v[j + 1] -= __uint_as_float(h & 0xffff0000u);
          }
        }
        emit_group(cg, v);
      }
    }
  }
  if (leader) trace(p, trace_tile, trace_base + 4);
  if (p.tma_out) {
    fence_proxy_async_smem();
    epi_sync();
    if (leader) trace(p, trace_tile, trace_base + 5);
    if (leader && !(p.dbg & 2)) {
      const int wc = ox0 * p.out_stride + px, hc = oy0 * p.out_stride + py;
      const int lo_off = p.split_out ? p.split_lo_off : 0;
      if (p.tma_out == 2) {
        for (int h = 0; h < 4; ++h)
          if (h * 32 < nvalid_c) tma_store_4d(map_o_ptr, sq + h * (128 * 128), p.out_c_offset + cbase + h * 32, wc, hc, img);
      } else {
        for (int h = 0; h < 2; ++h)
          if (h * 64 < nvalid_c) tma_store_4d(map_o_ptr, stg + h * (128 * 128), p.out_c_offset + lo_off + cbase + h * 64, wc, hc, img);
      }
      tma_store_commit();
    }
  }
  return true;
}

// bf16-pair output of one M = 128 block, normal orientation, bias / LeakyReLU (TcParams::epi_slices).  epilogue_block stages
// hi and lo in turn through the one CTA-wide 32 KB tile and waits for each store right after issuing it, inside CTA-wide
// barriers - on layers whose mainloop is short (g_s layer 3: ~300 MMAs per tile) that epilogue is longer than the mainloop.
// Here each of the 8 warps owns 4 KB of that tile: two 2 KB slices of 32 pixels (4 rows x 8) x 32 channels in the 64-byte
// swizzle layout, each stored by the warp's own TMA box.  The warp reads its two 32-column groups of the accumulator once,
// forms hi and lo together in registers, and sends hi / lo / hi / lo through the two slices in rotation, one bulk group per
// store: a slice is rewritten only after the store two groups back (its previous use) has read it, never the one just issued.
// No barrier between warps.  The caller's `release` runs right after the block's TMEM reads when `last` is set, so the MMAs of
// the next tile but one may start while the stores are still draining.
template <typename Release>
__device__ __forceinline__ void epilogue_block_slices(const TcParams& p, const float* s_bias, uint8_t* sq, const CUtensorMap* map_o_ptr,
                                                      uint32_t acc_tmem, int q, int lane, int wi, int img, int oy0, int ox0, int py, int px,
                                                      int cbase, bool last, Release&& release, uint32_t trace_tile) {
  const bool leader = wi == 0 && lane == 0;
  if (leader) trace(p, trace_tile, 8 + 0);
  const int cg0 = (wi >> 2) * 2;                                 // warpgroup hs takes channel groups 2 hs, 2 hs + 1
  const bool live = cbase + cg0 * 32 < p.cout;                   // c_out % 64 == 0: both groups exist or neither
  uint32_t hi[32], lo[32];                                       // 64 channels of this thread's pixel, packed in pairs
  if (live) {
    const uint32_t addr = acc_tmem + (static_cast<uint32_t>(q * 32) << 16) + cg0 * 32;
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      float v[32];
      tmem_ld_32x32(addr + g * 32, v);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; j += 2) {
        const int c = cbase + (cg0 + g) * 32 + j;
        float a = v[j] + s_bias[c], b = v[j + 1] + s_bias[c + 1];
        if (p.epilogue == NIC_EPI_LRELU) { a = a > 0.f ? a : 0.01f * a; b = b > 0.f ? b : 0.01f * b; }
        const uint32_t h = pack_bf16x2(a, b);
        hi[g * 16 + (j >> 1)] = h;
        lo[g * 16 + (j >> 1)] = pack_bf16x2(a - __uint_as_float(h << 16), b - __uint_as_float(h & 0xffff0000u));   // lo = x - bf16(x)
      }
    }
  }
  if (last) release();
  if (leader) trace(p, trace_tile, 8 + 4);
  if (!live) return;
  uint8_t* slices = sq + wi * 4096;
  uint8_t* mine = slices + lane * 64;                            // box row = lane: pixel (q * 4 + lane / 8, lane % 8) of the block
  const uint32_t swz = static_cast<uint32_t>(lane >> 1) & 3u;
  const int wc = ox0 * p.out_stride + px, hc = (oy0 + q * 4) * p.out_stride + py;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int g = k >> 1, half = k & 1;                          // hi of group 0, lo of group 0, hi of group 1, lo of group 1
    if (lane == 0) tma_store_wait_read_1();
    __syncwarp();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint32_t w[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) w[e] = half ? lo[g * 16 + j * 4 + e] : hi[g * 16 + j * 4 + e];
      *reinterpret_cast<uint4*>(mine + half * 2048 + ((static_cast<uint32_t>(j) ^ swz) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0 && !(p.dbg & 2)) {
      tma_store_4d(map_o_ptr, slices + half * 2048, p.out_c_offset + (half ? p.split_lo_off : 0) + cbase + (cg0 + g) * 32, wc, hc, img);
      tma_store_commit();
    }
  }
  if (leader) trace(p, trace_tile, 8 + 5);
}

// Epilogue of one tile in the swapped orientation (TcParams::swap): TMEM lane = output channel, column = pixel (block h of the
// tile owns columns [128 h, 128 h + 128)).  Bias / LeakyReLU per lane, then the tile is TRANSPOSED into the same [pixel][64 ch]
// 128-byte-swizzled staging panels the TMA stores of the normal orientation use: lane c writes bf16 (pixel p, channel c) with
// 2-byte stores - a warp covers 32 consecutive channels of one pixel, i.e. four 16-byte chunks of one 128-byte row, conflict
// free.  bf16 or bf16-pair NHWC outputs only (one staging + store round for hi, one for lo).
__device__ __forceinline__ bool epilogue_tile_swapped(const TcParams& p, const float* s_bias, uint8_t* sq, const CUtensorMap* map_o_ptr,
                                                      uint32_t acc_tmem, int q, int lane, int hs, bool leader, int img, int ty, int tx,
                                                      int py, int px, int cbase, int nblk) {
  const int c = q * 32 + lane;                                   // channel of this thread inside the N tile
  const uint32_t lane_addr = acc_tmem + (static_cast<uint32_t>(q * 32) << 16);
  const float bias = (cbase + c < p.cout) ? s_bias[cbase + c] : 0.f;
  const int nvalid_c = p.cout - cbase;
  auto epi_sync = [&]() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory"); };
  uint8_t* col = sq + (c >> 6) * (128 * 128) + (c & 7) * 2;      // panel of this channel + its byte inside a 16-byte chunk
  const uint32_t cchunk = static_cast<uint32_t>((c & 63) >> 3);
  const int npass = p.split_out ? 2 : 1;
  if (p.split_out && p.stage2) {
    // bf16-pair output through TWO staging tiles (hi tile, lo tile): every accumulator column is read ONCE, hi and lo are formed
    // together in registers BEFORE the wait for the previous block's stores (so that wait overlaps the TMEM loads and the
    // arithmetic), and one round of four TMA stores per block replaces two rounds of two - half the barriers, half the TMEM traffic
    for (int h = 0; h < nblk; ++h) {
      const int oy0 = ty * p.tile_h + p.blk_roff[h], ox0 = tx * p.tile_w + p.blk_coff[h];
      const int wc = ox0 * p.out_stride + px, hc = oy0 * p.out_stride + py;
      uint32_t whi[32], wlo[32];                                     // 64 pixel columns of this lane's channel, packed in pairs
#pragma unroll
      for (int g2 = 0; g2 < 2; ++g2) {
        float v[32];
        tmem_ld_32x32(lane_addr + h * 128 + hs * 64 + g2 * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          float a = v[j] + bias, b = v[j + 1] + bias;
          if (p.epilogue == NIC_EPI_LRELU) { a = a > 0.f ? a : 0.01f * a; b = b > 0.f ? b : 0.01f * b; }
          const uint32_t w = pack_bf16x2(a, b);
          whi[g2 * 16 + (j >> 1)] = w;
          wlo[g2 * 16 + (j >> 1)] = pack_bf16x2(a - __uint_as_float(w << 16), b - __uint_as_float(w & 0xffff0000u));
        }
      }
      if (leader) tma_store_wait_read();                             // the previous block's stores have read both tiles
      epi_sync();
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int ra = hs * 64 + 2 * i, rb = ra + 1;                 // pixel rows of the pair inside the block
        uint8_t* pa = col + ra * 128 + ((cchunk ^ (ra & 7)) << 4);
        uint8_t* pb = col + rb * 128 + ((cchunk ^ (rb & 7)) << 4);
        *reinterpret_cast<uint16_t*>(pa) = static_cast<uint16_t>(whi[i] & 0xffffu);
        *reinterpret_cast<uint16_t*>(pb) = static_cast<uint16_t>(whi[i] >> 16);
        *reinterpret_cast<uint16_t*>(pa + 2 * 128 * 128) = static_cast<uint16_t>(wlo[i] & 0xffffu);
        *reinterpret_cast<uint16_t*>(pb + 2 * 128 * 128) = static_cast<uint16_t>(wlo[i] >> 16);
      }
      fence_proxy_async_smem();
      epi_sync();
      if (leader && !(p.dbg & 2)) {
        const int off = p.out_c_offset + cbase;
        for (int k = 0; k < 2; ++k)
          if (k * 64 < nvalid_c) {
            tma_store_4d(map_o_ptr, sq + k * (128 * 128), off + k * 64, wc, hc, img);
            tma_store_4d(map_o_ptr, sq + (2 + k) * (128 * 128), off + p.split_lo_off + k * 64, wc, hc, img);
          }
        tma_store_commit();
      }
    }
    return true;
  }
  for (int h = 0; h < nblk; ++h) {
    const int oy0 = ty * p.tile_h + p.blk_roff[h], ox0 = tx * p.tile_w + p.blk_coff[h];
    const int wc = ox0 * p.out_stride + px, hc = oy0 * p.out_stride + py;
    for (int pass = 0; pass < npass; ++pass) {
      if (leader) tma_store_wait_read();                         // the staging tile may still be read by the previous store
      epi_sync();
#pragma unroll
      for (int g2 = 0; g2 < 2; ++g2) {
        float v[32];
        tmem_ld_32x32(lane_addr + h * 128 + hs * 64 + g2 * 32, v);
        tmem_ld_wait();
        const int r0 = hs * 64 + g2 * 32;                        // pixel row of v[0] inside the block (16 rows x 8 pixels)
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          float a = v[j] + bias, b = v[j + 1] + bias;
          if (p.epilogue == NIC_EPI_LRELU) { a = a > 0.f ? a : 0.01f * a; b = b > 0.f ? b : 0.01f * b; }
          uint32_t w = pack_bf16x2(a, b);
          if (pass == 1) w = pack_bf16x2(a - __uint_as_float(w << 16), b - __uint_as_float(w & 0xffff0000u));
          const int ra = r0 + j, rb = ra + 1;
          *reinterpret_cast<uint16_t*>(col + ra * 128 + ((cchunk ^ (ra & 7)) << 4)) = static_cast<uint16_t>(w & 0xffffu);
          *reinterpret_cast<uint16_t*>(col + rb * 128 + ((cchunk ^ (rb & 7)) << 4)) = static_cast<uint16_t>(w >> 16);
        }
      }
      fence_proxy_async_smem();
      epi_sync();
      if (leader && !(p.dbg & 2)) {
        const int off = p.out_c_offset + cbase + (pass == 1 ? p.split_lo_off : 0);
        for (int k = 0; k < 2; ++k)
          if (k * 64 < nvalid_c) tma_store_4d(map_o_ptr, sq + k * (128 * 128), off + k * 64, wc, hc, img);
        tma_store_commit();
      }
    }
  }
  return true;
}

// PAIR: the kernel runs as clusters of two CTAs (cta_group::2, see tc_primitives.cuh): CTA r of a cluster works on tile 2 j + r
// (same phase, same N tile), loads its own input patches and HALF of every weight slab (rows [64 r, 64 r + 64) of the N = 128
// slab); the leader's two issuing warps issue M = 256 MMAs over both CTAs' blocks and multicast the ring / accumulator commits;
// both CTAs' loads signal the leader's "full" barriers, both CTAs' epilogues release the leader's accumulator barriers.  Per MMA
// an SM then reads 4 KB of pixels + 2 KB of weights (96 B/clk) and fills half the weight bytes: the N = 128 mainloop stops being
// bound by shared-memory bandwidth.  Normal orientation, weight ring, one or two N tiles.
template <bool PAIR>
__global__ void __launch_bounds__(kThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
               const __grid_constant__ CUtensorMap map_g, const __grid_constant__ CUtensorMap map_o, const __grid_constant__ TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned, still a shared-space pointer
  __shared__ TcBarriers sb;
  __shared__ float s_bias[kMaxCout];
  __shared__ float s_beta[128];
  __shared__ int s_tap_brow[kMaxTaps];           // weight row of the tap's slab (TMA coordinate of the B producer)
  __shared__ uint32_t s_tap_aoff[kMaxTaps];      // descriptor offset (16-byte units) of the tap's first pixel inside the patch
  pdl_launch_dependents();
  if (threadIdx.x < kMaxTaps) {
    s_tap_brow[threadIdx.x] = p.taps[threadIdx.x].slab;
    s_tap_aoff[threadIdx.x] = static_cast<uint32_t>((p.taps[threadIdx.x].roff * p.pw_cols + p.taps[threadIdx.x].coff) * 128) >> 4;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool gdn = p.epilogue == NIC_EPI_GDN || p.epilogue == NIC_EPI_IGDN;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  if (threadIdx.x == 0) {
    for (int i = 0; i < kMaxSlots; ++i) { mbar_init(&sb.a_full[i], 1); mbar_init(&sb.a_empty[i], kMmaWarps); }
    for (int i = 0; i < kMaxBSlots; ++i) { mbar_init(&sb.b_full[i], 1); mbar_init(&sb.b_empty[i], kMmaWarps); }
    for (int i = 0; i < 2; ++i) { mbar_init(&sb.acc_full[i], kMmaWarps); mbar_init(&sb.acc_empty[i], PAIR ? 2 * kEpiWarps : kEpiWarps); }
    mbar_init(&sb.gdn_full, 1); mbar_init(&sb.gamma_full, 1); mbar_init(&sb.bres_full, 1);
    sb.abort_flag = 0;
    fence_barrier_init();
  }
  if (warp == 2) {
    if (PAIR) { tmem_alloc_pair(&sb.tmem_base, 512); tmem_relinquish_pair(); }
    else { tmem_alloc(&sb.tmem_base, 512); tmem_relinquish(); }
  }
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&map_a); tma_prefetch_desc(&map_w); if (gdn) tma_prefetch_desc(&map_g); if (p.tma_out) tma_prefetch_desc(&map_o); }
  // everything above is independent of the preceding kernel; from here on global memory it may have written is read
  pdl_wait();
  for (int i = threadIdx.x; i < p.cout; i += kThreads) s_bias[i] = p.bias[p.bias_mod ? i % p.bias_mod : i];
  if (p.beta) for (int i = threadIdx.x; i < 128; i += kThreads) s_beta[i] = p.beta[i];
  // K chunks this launch walks: all of [hi | lo | hi] x [W_hi | W_hi | W_lo], or - when the producer of the input flagged its lo
  // half as all zero - without the middle third (every role derives the same list from the same device word)
  int nchunks_eff = p.nchunks, skip_from = 1 << 30, skip_add = 0;
  if (p.lo_flag && __ldg(p.lo_flag) == 0) { skip_add = p.a_chunk_mod / 2; skip_from = skip_add; nchunks_eff = p.nchunks - skip_add; }
  // bf16x3 with a weight ring: the K chunks are walked c-slice by c-slice - (A_hi c, W_hi c), (A_hi c, W_lo c), (A_lo c, W_hi c) -
  // instead of in K-concatenation order, so that the second fetch of an A_hi patch follows the first within a sixth of the tile
  // (it used to come four sixths later and a quarter of those re-reads had left L2: g_a layer 2 read 1048 MB for an 805 MB input)
  const int nc = p.a_chunk_mod / 2, per = (skip_add ? 2 : 3);
  const bool perm = p.chunk_perm != 0;
  auto kchunk = [&](int chunk) {
    if (perm) { const int c = chunk / per, r = chunk - c * per; return r == 0 ? c : (r == 1 ? 2 * nc + c : nc + c); }
    return chunk + (chunk >= skip_from ? skip_add : 0);
  };

  tcgen05_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync();                      // the peer's barriers are initialised before anything arrives on them
  tcgen05_fence_after();
  const uint32_t tmem = sb.tmem_base;

  const int first_tile = blockIdx.x, tile_step = gridDim.x;

  if (warp == 0) {
    // ===================== A producer =====================
    if (lane == 0) {
      uint32_t it = 0;
      bool ok = true;
      const uint32_t bytes = p.ph_rows * p.pw_cols * 128;
      for (int tile = first_tile; tile < p.total_tiles && ok; tile += tile_step) {
        int ntile, phase, img, ty, tx;
        if (!decode_tile(p, tile, ntile, phase, img, ty, tx)) break;
        const TcPhase& ph = p.phases[phase];
        for (int chunk = 0; chunk < nchunks_eff && ok; ++chunk) {
          const int kc = kchunk(chunk);
          for (int pl = 0; pl < ph.nplanes; ++pl, ++it) {
            const int s = it % p.nsa;
            if (!wait_or_abort(&sb.a_empty[s], ((it / p.nsa) & 1) ^ 1, &sb, p.status)) { ok = false; break; }
            if (chunk == 0 && pl == 0) trace(p, (tile - first_tile) / tile_step, 5);
            if (chunk == nchunks_eff - 1 && pl == ph.nplanes - 1) trace(p, (tile - first_tile) / tile_step, 6);
            const int w0 = p.in_stride * (tx * p.tile_w + ph.plane_dxmin[pl]) + ph.plane_pw[pl];
            const int h0 = p.in_stride * (ty * p.tile_h + ph.plane_dymin[pl]) + ph.plane_ph[pl];
            if (PAIR) {       // both CTAs' patches complete the LEADER's barrier
              if (rank == 0) mbar_expect_tx(&sb.a_full[s], 2 * bytes);
              tma_load_4d_pair(smem + p.off_a + s * p.slot_bytes, &map_a, mapa_u32(smem_u32(&sb.a_full[s]), 0), (kc % p.a_chunk_mod) * 64, w0, h0, img);
            } else {
              mbar_expect_tx(&sb.a_full[s], bytes);
              tma_load_4d(smem + p.off_a + s * p.slot_bytes, &map_a, &sb.a_full[s], (kc % p.a_chunk_mod) * 64, w0, h0, img);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== B producer =====================
    if (lane == 0) {
      if (gdn) {   // gamma [c][c] bf16, K-major: two 64-column halves, resident for the whole kernel
        mbar_expect_tx(&sb.gamma_full, 2 * 128 * 128);
        tma_load_2d(smem + p.off_gamma, &map_g, &sb.gamma_full, 0, 0);
        tma_load_2d(smem + p.off_gamma + 128 * 128, &map_g, &sb.gamma_full, 64, 0);
      }
      const uint32_t bytes = p.nb * 128;
      if (p.b_resident) {
        // every (slab, chunk) tile of the layer once: [slab][chunk] tiles of nb x 64
        mbar_expect_tx(&sb.bres_full, bytes * p.nslabs * p.nchunks);
        for (int t = 0; t < p.nslabs; ++t)
          for (int chunk = 0; chunk < p.nchunks; ++chunk)
            tma_load_2d(smem + p.off_b + (t * p.nchunks + chunk) * bytes, &map_w, &sb.bres_full, chunk * 64, t * p.cout_pad);
      } else {
        uint32_t it = 0;
        bool ok = true;
        for (int tile = first_tile; tile < p.total_tiles && ok; tile += tile_step) {
          int ntile, phase, img, ty, tx;
          if (!decode_tile(p, tile, ntile, phase, img, ty, tx)) break;
          const TcPhase& ph = p.phases[phase];
          const int t0 = ph.plane_tap_begin[0], t1 = ph.plane_tap_begin[ph.nplanes];
          for (int chunk = 0; chunk < nchunks_eff && ok; ++chunk) {
            const int kc = kchunk(chunk);
            for (int t = t0; t < t1; ++t, ++it) {
              const int s = it % p.nsb;
              if (!wait_or_abort(&sb.b_empty[s], ((it / p.nsb) & 1) ^ 1, &sb, p.status)) { ok = false; break; }
              if (PAIR) {     // this CTA's half of the slab (the tensor map's box is nb / 2 rows)
                if (rank == 0) mbar_expect_tx(&sb.b_full[s], bytes);
                tma_load_2d_pair(smem + p.off_b + s * p.b_slot_bytes, &map_w, mapa_u32(smem_u32(&sb.b_full[s]), 0), kc * 64,
                                 s_tap_brow[t] * p.cout_pad + ntile * p.nb + static_cast<int>(rank) * (p.nb / 2));
              } else {
                mbar_expect_tx(&sb.b_full[s], bytes);
                tma_load_2d(smem + p.off_b + s * p.b_slot_bytes, &map_w, &sb.b_full[s], kc * 64, s_tap_brow[t] * p.cout_pad + ntile * p.nb);
              }
            }
          }
        }
      }
    }
  } else if (warp < kFirstEpiWarp) {
    // ===================== MMA issuers =====================
    // Warp 2 + b issues the MMAs of block b of every tile: the address arithmetic, barrier polls and uniform-register moves
    // between two taps cost one warp ~300-400 clk, about what the 8 MMAs of a two-block tap occupy the tensor pipe at
    // N = 128 and twice that at N = 16 - two issuers keep the pipe's queue full.  Both walk the same rings; the ring and
    // accumulator barriers count one tcgen05.commit per issuer.
    // The whole warp walks the loop (so every address below is warp-uniform); only the tcgen05 instructions themselves are
    // issued by one elected lane.
    {
      const int mw = warp - 2;
      const uint32_t idesc = umma_idesc_bf16(128, p.nb);
      const uint32_t a_base = smem_u32(smem + p.off_a), b_base = smem_u32(smem + p.off_b);
      const uint32_t a_hi = umma_desc_hi(p.pw_cols * 128), b_hi = umma_desc_hi(1024);
      const uint32_t bbytes = p.nb * 128;
      const int nsa = p.nsa, nsb = p.nsb, nchunks = nchunks_eff, b_res = p.b_resident;
      const bool swp = p.swap != 0;
      const uint32_t blk_off = (mw && !swp) ? static_cast<uint32_t>((p.blk_roff[1] * p.pw_cols + p.blk_coff[1]) * 128) >> 4 : 0u;
      const uint32_t idesc_use = PAIR ? umma_idesc_bf16(256, p.nb) : (swp ? umma_idesc_bf16(128, 256) : idesc);
      const uint32_t f_hi = swp ? b_hi : a_hi, g_hi = swp ? a_hi : b_hi;
      const uint32_t a_base_lo = umma_desc_lo(a_base), b_base_lo = umma_desc_lo(b_base);
      const uint32_t slot16 = static_cast<uint32_t>(p.slot_bytes) >> 4, bb16 = bbytes >> 4, bslot16 = static_cast<uint32_t>(p.b_slot_bytes) >> 4;
      // Resident weights (N = 16 layers): ONE thread per issuer walks the loop - no barrier polls inside a plane, so dropping the
      // per-tap elect / reconvergence / warp barrier matters (per-tap overhead, not the tensor pipe, bounds these layers).
      // Weight ring (everything else): the warp-uniform loop below is faster (mbarrier polls by the whole warp wake sooner).
      if (b_res && lane == 0) {
        uint32_t tcount = 0;
        uint32_t sa = 0, pa = 0, sbi = 0, pb = 0;      // ring slot + phase parity of the A and B rings
        bool ok = true;
        if (b_res) { ok = wait_or_abort(&sb.bres_full, 0, &sb, p.status); tcgen05_fence_after(); }
        // 3x3 stride-1 layers (the sub-pixel form of the 128 -> 3 transposed conv): the nine tap offsets live in registers and
        // the tap loop is unrolled - 36 back-to-back MMAs per chunk with no shared-memory loads or loop control between them
        uint32_t ao[9], bo[9];
        const bool nine = p.nphases == 1 && p.phases[0].nplanes == 1 && p.nslabs == 9;
#pragma unroll
        for (int i = 0; i < 9; ++i) { ao[i] = nine ? s_tap_aoff[i] : 0u; bo[i] = nine ? s_tap_brow[i] * nchunks * bb16 : 0u; }
        for (int tile = first_tile; tile < p.total_tiles && ok; tile += tile_step, ++tcount) {
          int ntile, phase, img, ty, tx;
          if (!decode_tile(p, tile, ntile, phase, img, ty, tx)) break;
          const TcPhase& ph = p.phases[phase];
          const int nblk = live_blocks(p, ty, tx);
          const int nplanes = ph.nplanes;
          const uint32_t buf = tcount & 1;
          if (!wait_or_abort(&sb.acc_empty[buf], ((tcount >> 1) & 1) ^ 1, &sb, p.status)) break;
          if (mw == 0) trace(p, tcount, 0);
          tcgen05_fence_after();
          const uint32_t d_tmem = tmem + buf * 256 + mw * 128;
          const bool live = mw < nblk;
          uint32_t accumulate = 0;
          for (int chunk = 0; chunk < nchunks && ok; ++chunk) {
            for (int pl = 0; pl < nplanes && ok; ++pl) {
              if (!mbar_try_wait(&sb.a_full[sa], pa) && !wait_or_abort(&sb.a_full[sa], pa, &sb, p.status)) { ok = false; break; }
              if (chunk == 0 && pl == 0 && mw == 0) trace(p, tcount, 1);
              tcgen05_fence_after();
              const uint32_t a_slot_lo = a_base_lo + sa * slot16 + blk_off;
              const int t_begin = ph.plane_tap_begin[pl], t_end = ph.plane_tap_begin[pl + 1];
              if (nine) {
                if (live) {
                  const uint32_t bc = b_base_lo + chunk * bb16;
#pragma unroll
                  for (int i = 0; i < 9; ++i) {
                    const uint32_t b_lo = bc + bo[i], a_lo0 = a_slot_lo + ao[i];
                    umma_bf16_lohi(d_tmem, a_lo0, a_hi, b_lo, b_hi, idesc, i == 0 ? accumulate : 1u);
                    umma_bf16_lohi(d_tmem, a_lo0 + 2, a_hi, b_lo + 2, b_hi, idesc, 1);
                    umma_bf16_lohi(d_tmem, a_lo0 + 4, a_hi, b_lo + 4, b_hi, idesc, 1);
                    umma_bf16_lohi(d_tmem, a_lo0 + 6, a_hi, b_lo + 6, b_hi, idesc, 1);
                  }
                  accumulate = 1;
                }
              } else if (b_res) {
                if (live) {
                  for (int t = t_begin; t < t_end; ++t) {
                    const uint32_t b_lo = b_base_lo + (s_tap_brow[t] * nchunks + chunk) * bb16;
                    const uint32_t a_lo0 = a_slot_lo + s_tap_aoff[t];
                    umma_bf16_lohi(d_tmem, a_lo0, a_hi, b_lo, b_hi, idesc, accumulate);
                    umma_bf16_lohi(d_tmem, a_lo0 + 2, a_hi, b_lo + 2, b_hi, idesc, 1);
                    umma_bf16_lohi(d_tmem, a_lo0 + 4, a_hi, b_lo + 4, b_hi, idesc, 1);
                    umma_bf16_lohi(d_tmem, a_lo0 + 6, a_hi, b_lo + 6, b_hi, idesc, 1);
                    accumulate = 1;
                  }
                }
              } else {
                for (int t = t_begin; t < t_end; ++t) {
                  if (!mbar_try_wait(&sb.b_full[sbi], pb) && !wait_or_abort(&sb.b_full[sbi], pb, &sb, p.status)) { ok = false; break; }
                  tcgen05_fence_after();
                  if (live) {
                    const uint32_t b_lo = b_base_lo + sbi * bslot16;
                    const uint32_t a_lo0 = a_slot_lo + s_tap_aoff[t];
                    umma_bf16_lohi(d_tmem, a_lo0, a_hi, b_lo, b_hi, idesc, accumulate);
                    umma_bf16_lohi(d_tmem, a_lo0 + 2, a_hi, b_lo + 2, b_hi, idesc, 1);
                    umma_bf16_lohi(d_tmem, a_lo0 + 4, a_hi, b_lo + 4, b_hi, idesc, 1);
                    umma_bf16_lohi(d_tmem, a_lo0 + 6, a_hi, b_lo + 6, b_hi, idesc, 1);
                    accumulate = 1;
                  }
                  umma_commit(&sb.b_empty[sbi]);
                  if (++sbi == static_cast<uint32_t>(nsb)) { sbi = 0; pb ^= 1; }
                }
              }
              umma_commit(&sb.a_empty[sa]);
              if (++sa == static_cast<uint32_t>(nsa)) { sa = 0; pa ^= 1; }
            }
          }
          if (mw == 0) trace(p, tcount, 2);
          umma_commit(&sb.acc_full[buf]);
        }
      }
      if (!b_res && !(PAIR && rank != 0)) {       // (pair: the leader CTA issues for both)
        auto MMA = [&](uint32_t d, uint32_t f, uint32_t fh, uint32_t g, uint32_t gh, uint32_t id, uint32_t acc) {
          if constexpr (PAIR) umma_bf16_lohi_pair(d, f, fh, g, gh, id, acc); else umma_bf16_lohi(d, f, fh, g, gh, id, acc);
        };
        auto COMMIT = [&](uint64_t* bar) { if constexpr (PAIR) umma_commit_pair(bar); else umma_commit(bar); };
        uint32_t tcount = 0;
        uint32_t sa = 0, pa = 0, sbi = 0, pb = 0;      // ring slot + phase parity of the A and B rings
        bool ok = true;
        if (b_res) { ok = wait_or_abort(&sb.bres_full, 0, &sb, p.status); tcgen05_fence_after(); }
        for (int tile = first_tile; tile < p.total_tiles && ok; tile += tile_step, ++tcount) {
          int ntile, phase, img, ty, tx;
          if (!decode_tile(p, tile, ntile, phase, img, ty, tx)) break;
          const TcPhase& ph = p.phases[phase];
          int nblk = live_blocks(p, ty, tx);
          if (PAIR) {       // the M = 256 MMA covers block b of both tiles of the pair
            int n2, ph2, img2, ty2, tx2;
            if (decode_tile(p, tile + 1, n2, ph2, img2, ty2, tx2)) { const int nb2 = live_blocks(p, ty2, tx2); nblk = nb2 > nblk ? nb2 : nblk; }
          }
          const int nplanes = ph.nplanes;
          const uint32_t buf = tcount & 1;
          if (!wait_or_abort(&sb.acc_empty[buf], ((tcount >> 1) & 1) ^ 1, &sb, p.status)) break;
          if (lane == 0 && mw == 0) { trace(p, tcount, 0); trace_value(p, tcount, 7, phase); }
          tcgen05_fence_after();
          // swapped orientation: issuer 0 alone issues N = 256 MMAs (weights first, the pixels of both blocks second) into the
          // whole 256-column buffer; issuer 1 walks the rings and only commits
          const uint32_t d_tmem = tmem + buf * 256 + (swp ? 0 : mw * 128);
          const int only = tail_block(p, tile);
          const bool live = swp ? mw == 0 : (mw < nblk && (only < 0 || mw == only));
          uint32_t accumulate = 0;
          if (nplanes == 1 && ph.plane_tap_begin[1] - ph.plane_tap_begin[0] == 1) {
            // one tap per K chunk (1x1 convs): the per-chunk bookkeeping of the generic loop below (one ring wait, one elect / warp
            // barrier and two commits for 4 MMAs) costs more than the MMAs - two chunks per iteration: 8 MMAs per wait / elect round
            const uint32_t aoff = s_tap_aoff[ph.plane_tap_begin[0]] + blk_off;
            for (int chunk = 0; chunk < nchunks && ok; chunk += 2) {
              const bool two = chunk + 1 < nchunks;
              if (!mbar_try_wait(&sb.a_full[sa], pa) && !wait_or_abort(&sb.a_full[sa], pa, &sb, p.status)) { ok = false; break; }
              if (chunk == 0 && lane == 0 && mw == 0) trace(p, tcount, 1);
              const uint32_t sa0 = sa;
              if (++sa == static_cast<uint32_t>(nsa)) { sa = 0; pa ^= 1; }
              uint32_t sa1 = sa0;
              if (two) {
                if (!mbar_try_wait(&sb.a_full[sa], pa) && !wait_or_abort(&sb.a_full[sa], pa, &sb, p.status)) { ok = false; break; }
                sa1 = sa;
                if (++sa == static_cast<uint32_t>(nsa)) { sa = 0; pa ^= 1; }
              }
              if (!mbar_try_wait(&sb.b_full[sbi], pb) && !wait_or_abort(&sb.b_full[sbi], pb, &sb, p.status)) { ok = false; break; }
              const uint32_t s0 = sbi;
              if (++sbi == static_cast<uint32_t>(nsb)) { sbi = 0; pb ^= 1; }
              uint32_t s1 = s0;
              if (two) {
                if (!mbar_try_wait(&sb.b_full[sbi], pb) && !wait_or_abort(&sb.b_full[sbi], pb, &sb, p.status)) { ok = false; break; }
                s1 = sbi;
                if (++sbi == static_cast<uint32_t>(nsb)) { sbi = 0; pb ^= 1; }
              }
              tcgen05_fence_after();
              const uint32_t a_lo0 = a_base_lo + sa0 * slot16 + aoff, a_lo1 = a_base_lo + sa1 * slot16 + aoff;
              const uint32_t b_lo0 = b_base_lo + s0 * bslot16, b_lo1 = b_base_lo + s1 * bslot16;
              const uint32_t f0 = swp ? b_lo0 : a_lo0, g0 = swp ? a_lo0 : b_lo0, f1 = swp ? b_lo1 : a_lo1, g1 = swp ? a_lo1 : b_lo1;
              if (elect_one()) {
                if (live) {
                  MMA(d_tmem, f0, f_hi, g0, g_hi, idesc_use, accumulate);
                  MMA(d_tmem, f0 + 2, f_hi, g0 + 2, g_hi, idesc_use, 1);
                  MMA(d_tmem, f0 + 4, f_hi, g0 + 4, g_hi, idesc_use, 1);
                  MMA(d_tmem, f0 + 6, f_hi, g0 + 6, g_hi, idesc_use, 1);
                }
                COMMIT(&sb.b_empty[s0]);
                COMMIT(&sb.a_empty[sa0]);
                if (two) {
                  if (live) {
                    MMA(d_tmem, f1, f_hi, g1, g_hi, idesc_use, 1);
                    MMA(d_tmem, f1 + 2, f_hi, g1 + 2, g_hi, idesc_use, 1);
                    MMA(d_tmem, f1 + 4, f_hi, g1 + 4, g_hi, idesc_use, 1);
                    MMA(d_tmem, f1 + 6, f_hi, g1 + 6, g_hi, idesc_use, 1);
                  }
                  COMMIT(&sb.b_empty[s1]);
                  COMMIT(&sb.a_empty[sa1]);
                }
              }
              __syncwarp();
              accumulate = 1;
            }
          } else
          for (int chunk = 0; chunk < nchunks && ok; ++chunk) {
            for (int pl = 0; pl < nplanes && ok; ++pl) {
              if (!mbar_try_wait(&sb.a_full[sa], pa) && !wait_or_abort(&sb.a_full[sa], pa, &sb, p.status)) { ok = false; break; }
              if (chunk == 0 && pl == 0 && lane == 0 && mw == 0) trace(p, tcount, 1);
              tcgen05_fence_after();
              const uint32_t a_slot_lo = umma_desc_lo(a_base + sa * p.slot_bytes);
              const int t_end = ph.plane_tap_begin[pl + 1];
              // two taps per iteration: one elect / reconvergence / warp barrier per 8 MMAs of this issuer
              for (int t = ph.plane_tap_begin[pl]; t < t_end; t += 2) {
                const bool two = t + 1 < t_end;
                if (!mbar_try_wait(&sb.b_full[sbi], pb) && !wait_or_abort(&sb.b_full[sbi], pb, &sb, p.status)) { ok = false; break; }
                const uint32_t s0 = sbi;
                if (++sbi == static_cast<uint32_t>(nsb)) { sbi = 0; pb ^= 1; }
                uint32_t s1 = s0;
                if (two) {
                  if (!mbar_try_wait(&sb.b_full[sbi], pb) && !wait_or_abort(&sb.b_full[sbi], pb, &sb, p.status)) { ok = false; break; }
                  s1 = sbi;
                  if (++sbi == static_cast<uint32_t>(nsb)) { sbi = 0; pb ^= 1; }
                }
                tcgen05_fence_after();
                const uint32_t b_lo0 = b_base_lo + s0 * bslot16, b_lo1 = b_base_lo + s1 * bslot16;
                const uint32_t a_lo0 = a_slot_lo + s_tap_aoff[t] + blk_off, a_lo1 = a_slot_lo + s_tap_aoff[two ? t + 1 : t] + blk_off;
                // first / second operand of the MMA: (pixels, weights), or (weights, pixels) in the swapped orientation
                const uint32_t f0 = swp ? b_lo0 : a_lo0, g0 = swp ? a_lo0 : b_lo0, f1 = swp ? b_lo1 : a_lo1, g1 = swp ? a_lo1 : b_lo1;
                if (elect_one()) {
                  if (live) {
                    MMA(d_tmem, f0, f_hi, g0, g_hi, idesc_use, accumulate);
                    MMA(d_tmem, f0 + 2, f_hi, g0 + 2, g_hi, idesc_use, 1);
                    MMA(d_tmem, f0 + 4, f_hi, g0 + 4, g_hi, idesc_use, 1);
                    MMA(d_tmem, f0 + 6, f_hi, g0 + 6, g_hi, idesc_use, 1);
                  }
                  COMMIT(&sb.b_empty[s0]);
                  if (two) {
                    if (live) {
                      MMA(d_tmem, f1, f_hi, g1, g_hi, idesc_use, 1);
                      MMA(d_tmem, f1 + 2, f_hi, g1 + 2, g_hi, idesc_use, 1);
                      MMA(d_tmem, f1 + 4, f_hi, g1 + 4, g_hi, idesc_use, 1);
                      MMA(d_tmem, f1 + 6, f_hi, g1 + 6, g_hi, idesc_use, 1);
                    }
                    COMMIT(&sb.b_empty[s1]);
                  }
                }
                __syncwarp();
                accumulate = 1;
              }
              if (elect_one()) COMMIT(&sb.a_empty[sa]);
              __syncwarp();
              if (++sa == static_cast<uint32_t>(nsa)) { sa = 0; pa ^= 1; }
            }
          }
          if (lane == 0 && mw == 0) trace(p, tcount, 2);
          if (elect_one()) COMMIT(&sb.acc_full[buf]);
          __syncwarp();
        }
      }
      __syncwarp();
    }
  } else if (p.epi_slices) {
    // ===================== epilogue (8 warps): bf16-pair output through per-warp slices =====================
    // (a loop of its own: inlined into the generic loop below, epilogue_block_slices pushes the fused-GDN path of epilogue_block
    // into register spills)
    const int q = warp & 3, wi = warp - kFirstEpiWarp;
    uint8_t* sq = smem + p.off_sq;
    uint32_t tcount = 0;
    for (int tile = first_tile; tile < p.total_tiles; tile += tile_step, ++tcount) {
      int ntile, phase, img, ty, tx;
      if (!decode_tile(p, tile, ntile, phase, img, ty, tx)) break;
      const TcPhase& ph = p.phases[phase];
      const int nblk = live_blocks(p, ty, tx);
      const uint32_t buf = tcount & 1;
      if (!__all_sync(0xffffffffu, wait_or_abort(&sb.acc_full[buf], (tcount >> 1) & 1, &sb, p.status))) break;
      tcgen05_fence_after();
      auto release = [&]() {
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR && rank != 0) mbar_arrive_cluster(mapa_u32(smem_u32(&sb.acc_empty[buf]), 0));   // the leader's issuers wait for both CTAs
          else mbar_arrive(&sb.acc_empty[buf]);
        }
      };
      int b0 = 0, b1 = (p.dbg & 8) ? 0 : nblk;                     // the blocks of this slot (tail_block: one of them)
      if (const int only = tail_block(p, tile); only >= 0) { b0 = only; b1 = only < b1 ? only + 1 : b0; }
      for (int b = b0; b < b1; ++b)      // the last block releases the accumulator right after its TMEM reads
        epilogue_block_slices(p, s_bias, sq, &map_o, tmem + buf * 256 + b * 128, q, lane, wi, img, ty * p.tile_h + p.blk_roff[b],
                              tx * p.tile_w + p.blk_coff[b], ph.py, ph.px, ntile * p.nb, b == b1 - 1, release, b == b0 ? tcount : 0xffffffffu);
      if (wi == 0 && lane == 0) trace(p, tcount, 4);
      if (b0 >= b1) release();
    }
    if (lane == 0) tma_store_wait_all();     // bulk groups belong to the thread that committed them: every warp has its own
  } else {
    // ===================== epilogue (8 warps) =====================
    const int q = warp & 3;                       // TMEM lane quadrant this warp may read
    uint8_t* sq = smem + p.off_sq;
    uint32_t tcount = 0, gdn_count = 0;
    bool ok = true;
    for (int tile = first_tile; tile < p.total_tiles && ok; tile += tile_step, ++tcount) {
      int ntile, phase, img, ty, tx;
      if (!decode_tile(p, tile, ntile, phase, img, ty, tx)) break;
      const TcPhase& ph = p.phases[phase];
      const int nblk = live_blocks(p, ty, tx);
      const uint32_t buf = tcount & 1;
      if (!__all_sync(0xffffffffu, wait_or_abort(&sb.acc_full[buf], (tcount >> 1) & 1, &sb, p.status))) break;
      tcgen05_fence_after();
      if (p.swap) {
        if (!(p.dbg & 8))
          ok = epilogue_tile_swapped(p, s_bias, sq, &map_o, tmem + buf * 256, q, lane, (warp - kFirstEpiWarp) >> 2,
                                     warp == kFirstEpiWarp && lane == 0, img, ty, tx, ph.py, ph.px, ntile * p.nb, nblk);
      } else
      for (int b = 0; b < nblk && ok && !(p.dbg & 8); ++b)
        if (const int only = tail_block(p, tile); only < 0 || b == only)
        ok = epilogue_block<kEpiWarps>(p, &sb, s_bias, s_beta, sq, smem + p.off_gamma, &map_o, tmem + buf * 256 + b * 128, q, lane,
                                       (warp - kFirstEpiWarp) >> 2, warp == kFirstEpiWarp && lane == 0, img, ty * p.tile_h + p.blk_roff[b],
                                       tx * p.tile_w + p.blk_coff[b], ph.py, ph.px, ntile * p.nb, gdn_count, b == 0 ? tcount : 0xffffffffu);
      if (warp == kFirstEpiWarp && lane == 0) trace(p, tcount, 4);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR && rank != 0) mbar_arrive_cluster(mapa_u32(smem_u32(&sb.acc_empty[buf]), 0));   // the leader's issuers wait for both CTAs
        else mbar_arrive(&sb.acc_empty[buf]);
      }
    }
    if (p.tma_out && warp == kFirstEpiWarp && lane == 0) tma_store_wait_all();
  }

  tcgen05_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync();                      // no CTA leaves while its peer may still read its shared memory or signal its barriers
  if (warp == 2) { if (PAIR) tmem_dealloc_pair(tmem, 512); else tmem_dealloc(tmem, 512); }
}

// ---------------------------------------------------------------------------------------------
// First layer of g_a: Conv2d(3, 128, 5, stride 2, pad 2) + GDN straight from the NCHW fp32 image (Components.py:10-11).
// K = 75 is too shallow for a TMA-fed pipeline, so four producer warps build the [128 pixel x 80] bf16 A operand of each
// block in shared memory (im2col of a 35 x 35 x 3 image patch, k = (kh * 5 + kw) * 3 + c, zero padded to 80), one thread
// issues 5 tcgen05.mma per block against the resident [128 x 80] weights, and the shared epilogue applies the fused GDN and
// stores the bf16 NHWC tile with TMA.  13 warps: 0-3 producers, 4 MMA issuer / weight loader, 5-12 epilogue (two groups).
// ---------------------------------------------------------------------------------------------
constexpr int kFirstThreads = 160 + 8 * 32;
constexpr int kPatchW = 20, kPatchH = 35, kPatchCols = 19, kPatchPlane = kPatchH * kPatchW;   // fp32 patch rows padded to 20 floats

struct FirstParams {
  const float* x;                 // [n, 3, hin, win] fp32
  int n, hin, win, tiles_x, tiles_y, total_tiles;
  int off_a, off_w, off_gamma, off_sq, off_patch;
};

struct __align__(8) FirstBarriers {
  uint64_t a_full[2], a_empty[2], w_full, gdn_full2;
  TcBarriers common;              // acc_full / acc_empty / gdn_full / gamma_full + tmem_base + abort flag (epilogue_block uses these)
};

// Tile = one M = 128 block (16 rows x 8 output pixels).  Everything is double-buffered by tile parity g = it & 1: A operand
// stage g, accumulator columns [g*128, +128), gamma-contraction columns [256 + g*128, +128), and epilogue GROUP g (4 warps
// with their own squares / staging tile, named barrier and gamma barrier) - so the two epilogue groups work on consecutive
// tiles concurrently while the producers expand the next patch.
__global__ void __launch_bounds__(kFirstThreads, 1)
conv_first_tc_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_g,
                     const __grid_constant__ CUtensorMap map_o, const __grid_constant__ TcParams p, const __grid_constant__ FirstParams f) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // 1024-aligned, still a shared-space pointer
  __shared__ FirstBarriers fb;
  __shared__ float s_bias[128];
  __shared__ float s_beta[128];
  TcBarriers& sb = fb.common;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
  if (tid < 128) { s_bias[tid] = p.bias[tid]; s_beta[tid] = p.beta[tid]; }
  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&fb.a_full[i], 128); mbar_init(&fb.a_empty[i], 1);
      mbar_init(&sb.acc_full[i], 1); mbar_init(&sb.acc_empty[i], 4);
    }
    mbar_init(&fb.w_full, 1); mbar_init(&fb.gdn_full2, 1);
    mbar_init(&sb.gdn_full, 1); mbar_init(&sb.gamma_full, 1);
    sb.abort_flag = 0;
    fence_barrier_init();
  }
  if (warp == 4) { tmem_alloc(&sb.tmem_base, 512); tmem_relinquish(); }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = sb.tmem_base;
  const int first_tile = blockIdx.x, tile_step = gridDim.x;
  float* patch = reinterpret_cast<float*>(smem + f.off_patch);

  auto tile_coords = [&](int tile, int& img, int& ty, int& tx) {
    tx = tile % f.tiles_x; tile /= f.tiles_x; ty = tile % f.tiles_y; img = tile / f.tiles_y;
  };

  if (warp < 4) {
    // ===================== producers: image patch -> bf16 im2col A operand =====================
    // The fp32 patch (3 x 35 x 19) of tile i+1 streams into the other half of a double buffer with cp.async (zero fill =
    // conv padding) while tile i is expanded; warp w copies patch rows w, w+4, ...
    auto fetch_patch = [&](int tile, int bufi) {
      int img, ty, tx;
      tile_coords(tile, img, ty, tx);
      const int y0 = 2 * (ty * 16) - 2, x0 = 2 * (tx * 8) - 2;
      const int gx = x0 + lane;
      const bool col_ok = lane < kPatchCols && gx >= 0 && gx < f.win;
      const float* base = f.x + static_cast<long>(img) * 3 * f.hin * f.win + (col_ok ? gx : 0);
      const uint32_t dst0 = smem_u32(patch + bufi * (3 * kPatchPlane)) + lane * 4;
      if (lane < kPatchCols) {
        // warp w copies rows w, w + 4, ... of each colour plane; fully unrolled so the 27 copies are independent
#pragma unroll
        for (int c = 0; c < 3; ++c) {
#pragma unroll
          for (int j = 0; j < 9; ++j) {
            const int yy = warp + 4 * j;
            if (yy < kPatchH) {
              const int gy = y0 + yy;
              const bool ok = col_ok && gy >= 0 && gy < f.hin;
              const float* src = base + (static_cast<long>(c) * f.hin + (ok ? gy : 0)) * f.win;
              asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst0 + (c * kPatchPlane + yy * kPatchW) * 4), "l"(src),
                           "r"(ok ? 4 : 0)
                           : "memory");
            }
          }
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (first_tile < f.total_tiles) fetch_patch(first_tile, 0);
    uint32_t it = 0;
    const int r = tid, g = r >> 3, c8 = r & 7;
    for (int tile = first_tile; tile < f.total_tiles; tile += tile_step, ++it) {
      const uint32_t st = it & 1;
      if (tid == 0) trace(p, it, 0);
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      asm volatile("bar.sync 3, 128;" ::: "memory");         // patch(it) visible to all producers; patch(it-1) no longer read
      if (tid == 0) trace(p, it, 1);
      if (tile + tile_step < f.total_tiles) fetch_patch(tile + tile_step, st ^ 1);
      if (tid == 0) trace(p, it, 2);
      if (!__all_sync(0xffffffffu, wait_or_abort(&fb.a_empty[st], ((it >> 1) & 1) ^ 1, &sb, p.status))) break;
      if (tid == 0) trace(p, it, 3);
      const float* src = patch + st * (3 * kPatchPlane) + (2 * g) * kPatchW + 2 * c8;
      uint8_t* dst = smem + f.off_a + st * (2 * 128 * 128) + r * 128;
#pragma unroll
      for (int ch = 0; ch < 10; ++ch) {
        uint32_t w[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          float v2[2];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int k = ch * 8 + e * 2 + h;
            if (k < 75) { const int tap = k / 3, c = k % 3; v2[h] = src[c * kPatchPlane + (tap / 5) * kPatchW + (tap % 5)]; }
            else v2[h] = 0.f;
          }
          w[e] = pack_bf16x2(v2[0], v2[1]);
        }
        *reinterpret_cast<uint4*>(dst + (ch >> 3) * (128 * 128) + (((ch & 7) ^ (r & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
      }
      fence_proxy_async_smem();
      mbar_arrive(&fb.a_full[st]);
      if (tid == 0) trace(p, it, 4);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else if (warp == 4) {
    // ===================== weight loader + MMA issuer =====================
    if (lane == 0) {
      tma_prefetch_desc(&map_w); tma_prefetch_desc(&map_g); tma_prefetch_desc(&map_o);
      mbar_expect_tx(&fb.w_full, 2 * 128 * 128);
      tma_load_2d(smem + f.off_w, &map_w, &fb.w_full, 0, 0);
      tma_load_2d(smem + f.off_w + 128 * 128, &map_w, &fb.w_full, 64, 0);
      mbar_expect_tx(&sb.gamma_full, 2 * 128 * 128);
      tma_load_2d(smem + f.off_gamma, &map_g, &sb.gamma_full, 0, 0);
      tma_load_2d(smem + f.off_gamma + 128 * 128, &map_g, &sb.gamma_full, 64, 0);
      const uint32_t idesc = umma_idesc_bf16(128, 128);
      const uint32_t hi = umma_desc_hi(1024);
      const uint32_t a_lo = umma_desc_lo(smem_u32(smem + f.off_a)), w_lo = umma_desc_lo(smem_u32(smem + f.off_w));
      bool ok = wait_or_abort(&fb.w_full, 0, &sb, p.status);
      uint32_t it = 0;
      for (int tile = first_tile; tile < f.total_tiles && ok; tile += tile_step, ++it) {
        const uint32_t g = it & 1, par = (it >> 1) & 1;
        if (!wait_or_abort(&sb.acc_empty[g], par ^ 1, &sb, p.status)) break;
        trace(p, it, 5);
        if (!wait_or_abort(&fb.a_full[g], par, &sb, p.status)) break;
        trace(p, it, 6);
        tcgen05_fence_after();
        const uint32_t d = tmem + g * 128;
        const uint32_t ab = a_lo + g * ((2 * 128 * 128) >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16_lohi(d, ab + 2 * k, hi, w_lo + 2 * k, hi, idesc, k);
        umma_bf16_lohi(d, ab + ((128 * 128) >> 4), hi, w_lo + ((128 * 128) >> 4), hi, idesc, 1);      // k = 64..79
        umma_commit(&fb.a_empty[g]);
        umma_commit(&sb.acc_full[g]);
      }
    }
  } else {
    // ===================== epilogue (warps 5..12): group g = (warp - 5) / 4 takes the tiles of parity g =====================
    const int q = warp & 3;
    const int grp = (warp - 5) >> 2;
    uint8_t* sq = smem + f.off_sq + grp * (2 * 128 * 128);
    uint64_t* gbar = grp ? &fb.gdn_full2 : &sb.gdn_full;
    const bool leader = ((warp - 5) & 3) == 0 && lane == 0;
    uint32_t it = 0, gdn_count = 0;
    bool ok = true;
    for (int tile = first_tile; tile < f.total_tiles && ok; tile += tile_step, ++it) {
      if ((it & 1) != static_cast<uint32_t>(grp)) continue;
      int img, ty, tx;
      tile_coords(tile, img, ty, tx);
      if (!__all_sync(0xffffffffu, wait_or_abort(&sb.acc_full[grp], (it >> 1) & 1, &sb, p.status))) break;
      if (leader) trace(p, it, 7);
      tcgen05_fence_after();
      ok = epilogue_block<4, false>(p, &sb, s_bias, s_beta, sq, smem + f.off_gamma, &map_o, tmem + grp * 128, q, lane, 0, leader,
                                    img, ty * 16, tx * 8, 0, 0, 0, gdn_count, it, 8, 1 + grp, gbar, tmem + 256 + grp * 128);
      if (leader) trace(p, it, 14);
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&sb.acc_empty[grp]);
    }
    if (leader) tma_store_wait_all();
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// Builds phases / planes / taps of the kernel from the generic tap table.
int build_tc_geometry(const nic_conv_desc* d, const TapTable& tt, TcParams* p) {
  p->nphases = tt.nphases; p->in_stride = tt.in_stride; p->out_stride = tt.out_stride;
  int q = 0, ph_rows = 0, pw_cols = 0;
  const int s = tt.in_stride;
  for (int ph = 0; ph < tt.nphases; ++ph) {
    TcPhase& P = p->phases[ph];
    P.py = tt.py[ph]; P.px = tt.px[ph]; P.nplanes = 0;
    for (int a = 0; a < s; ++a)
      for (int b = 0; b < s; ++b) {
        int dymin = 127, dymax = -127, dxmin = 127, dxmax = -127, cnt = 0;
        for (int t = tt.phase_begin[ph]; t < tt.phase_begin[ph + 1]; ++t) {
          // input offset (dy, dx) in full-resolution pixels -> plane (dy mod s, dx mod s), plane offset floor(dy / s)
          const int pa = ((tt.dy[t] % s) + s) % s, pb = ((tt.dx[t] % s) + s) % s;
          if (pa != a || pb != b) continue;
          const int ry = (tt.dy[t] - pa) / s, rx = (tt.dx[t] - pb) / s;
          dymin = ry < dymin ? ry : dymin; dymax = ry > dymax ? ry : dymax;
          dxmin = rx < dxmin ? rx : dxmin; dxmax = rx > dxmax ? rx : dxmax;
          ++cnt;
        }
        if (!cnt) continue;
        const int pl = P.nplanes++;
        P.plane_ph[pl] = a; P.plane_pw[pl] = b; P.plane_dymin[pl] = dymin; P.plane_dxmin[pl] = dxmin;
        P.plane_tap_begin[pl] = q;
        for (int t = tt.phase_begin[ph]; t < tt.phase_begin[ph + 1]; ++t) {
          const int pa = ((tt.dy[t] % s) + s) % s, pb = ((tt.dx[t] % s) + s) % s;
          if (pa != a || pb != b) continue;
          const int ry = (tt.dy[t] - pa) / s, rx = (tt.dx[t] - pb) / s;
          p->taps[q].plane = pl; p->taps[q].roff = ry - dymin; p->taps[q].coff = rx - dxmin; p->taps[q].slab = t; ++q;
        }
        P.plane_tap_begin[pl + 1] = q;
        const int rows = kTileH + (dymax - dymin), cols = kTileW + (dxmax - dxmin);
        ph_rows = rows > ph_rows ? rows : ph_rows; pw_cols = cols > pw_cols ? cols : pw_cols;
      }
  }
  p->ph_rows = ph_rows; p->pw_cols = pw_cols;
  return NIC_OK;
}

__global__ void pack_weight_bf16_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int cin, int cout, int cout_pad,
                                        int kh, int kw, int transposed, TapTable tt) {
  const long total = static_cast<long>(tt.ntaps) * cout_pad * cin;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int ci = static_cast<int>(i % cin);
    const int co = static_cast<int>((i / cin) % cout_pad);
    const int t = static_cast<int>(i / (static_cast<long>(cin) * cout_pad));
    float v = 0.f;
    if (co < cout) {
      const int a = tt.kh[t], b = tt.kw[t];
      const long src = transposed ? ((static_cast<long>(ci) * cout + co) * kh + a) * kw + b
                                  : ((static_cast<long>(co) * cin + ci) * kh + a) * kw + b;
      v = w[src];
    }
    out[i] = __float2bfloat16_rn(v);
  }
}

// sub-pixel form of ConvTranspose2d(c_in, c_out, 5, stride 2, pad 2, output_padding 1), reference weight [c_in, c_out, 5, 5]:
//   out[2 oy + py, 2 ox + px, c] = sum_{(dy, dx) in 3x3} in[oy + dy, ox + dx, :] . W'[(dy + 1) * 3 + (dx + 1)][(py * 2 + px) * c_out + c][:]
// where W' holds w[:, c, kh, kw] of the tap of phase (py, px) that reads offset (dy, dx) and 0 where the phase has no such tap.
__global__ void pack_weight_subpixel_bf16_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int cin, int cout, TapTable tt) {
  const long total = 9L * 16 * cin;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int ci = static_cast<int>(i % cin);
    const int n = static_cast<int>((i / cin) % 16);
    const int slab = static_cast<int>(i / (16L * cin));
    const int dy = slab / 3 - 1, dx = slab % 3 - 1;
    float v = 0.f;
    if (n < 4 * cout) {
      const int phase = n / cout, c = n % cout;          // tap-table phases are ordered (py, px) = (0,0) (0,1) (1,0) (1,1)
      for (int t = tt.phase_begin[phase]; t < tt.phase_begin[phase + 1]; ++t)
        if (tt.dy[t] == dy && tt.dx[t] == dx) v = w[((static_cast<long>(ci) * cout + c) * 5 + tt.kh[t]) * 5 + tt.kw[t]];
    }
    out[i] = __float2bfloat16_rn(v);
  }
}

// the same in the bf16x3 arm: [9][16][3 c_in] = [W_hi | W_hi | W_lo]
__global__ void pack_weight_subpixel_x3_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int cin, int cout, TapTable tt) {
  const long total = 9L * 16 * 3 * cin;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int k = static_cast<int>(i % (3 * cin));
    const int n = static_cast<int>((i / (3 * cin)) % 16);
    const int slab = static_cast<int>(i / (16L * 3 * cin));
    const int ci = k % cin, part = k / cin;
    const int dy = slab / 3 - 1, dx = slab % 3 - 1;
    float v = 0.f;
    if (n < 4 * cout) {
      const int phase = n / cout, c = n % cout;
      for (int t = tt.phase_begin[phase]; t < tt.phase_begin[phase + 1]; ++t)
        if (tt.dy[t] == dy && tt.dx[t] == dx) v = w[((static_cast<long>(ci) * cout + c) * 5 + tt.kh[t]) * 5 + tt.kw[t]];
    }
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    out[i] = (part < 2) ? hi : __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

// first layer: reference [128, 3, 5, 5] -> [128][128] bf16, k = (kh * 5 + kw) * 3 + c, zero for k >= 75
__global__ void pack_first_bf16_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 128 * 128; i += gridDim.x * blockDim.x) {
    const int co = i / 128, k = i % 128;
    float v = 0.f;
    if (k < 75) { const int tap = k / 3, c = k % 3; v = w[((co * 3 + c) * 5 + tap / 5) * 5 + tap % 5]; }
    out[i] = __float2bfloat16_rn(v);
  }
}

int check_first_layer(const nic_conv_desc* d) {
  // bf16x3 also serves the bare conv (bias epilogue, f32 NHWC output): the training step keeps the pre-GDN tensor, and the
  // data gradient of the last g_s layer is this same conv over the image-shaped gradient; that form is also built for 192
  // output channels (the reference's default capacity, Models.py:17, and ScalableImageCoding(192, 128))
  const bool bare_x3 = d->precision == NIC_PREC_BF16X3 && d->epilogue == NIC_EPI_BIAS;
  const bool cout_ok = d->c_out == 128 || (d->precision == NIC_PREC_BF16X3 && d->c_out == 192);
  if (d->c_in != 3 || !cout_ok || d->kh != 5 || d->kw != 5 || d->stride != 2 || d->pad != 2 || d->transposed || d->mask_a ||
      (d->epilogue != NIC_EPI_GDN && !bare_x3))
    return fail(NIC_E_UNSUPPORTED, "conv bf16: the only c_in < 64 layer built is Conv2d(3, 128 | 192, 5, stride 2, pad 2) (+ GDN for 128) (g_a layer 1)");
  return NIC_OK;
}

// bf16x3: [tap][c_out padded][3 c_in] = [W_hi | W_hi | W_lo], W_hi = bf16(W), W_lo = bf16(W - W_hi)
__global__ void pack_weight_x3_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int cin, int cout, int cout_pad,
                                      int kh, int kw, int transposed, TapTable tt) {
  const long total = static_cast<long>(tt.ntaps) * cout_pad * 3 * cin;
  for (long i = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += static_cast<long>(gridDim.x) * blockDim.x) {
    const int k = static_cast<int>(i % (3 * cin));
    const int co = static_cast<int>((i / (3 * cin)) % cout_pad);
    const int t = static_cast<int>(i / (static_cast<long>(3) * cin * cout_pad));
    const int ci = k % cin, part = k / cin;
    float v = 0.f;
    if (co < cout) {
      const int a = tt.kh[t], b = tt.kw[t];
      const long src = transposed ? ((static_cast<long>(ci) * cout + co) * kh + a) * kw + b
                                  : ((static_cast<long>(co) * cin + ci) * kh + a) * kw + b;
      v = w[src];
    }
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    out[i] = (part < 2) ? hi : __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

__global__ void pack_gdn_bf16_kernel(int c, float beta_bound, float gamma_bound, float pedestal, const float* __restrict__ beta,
                                     const float* __restrict__ gamma, float* __restrict__ beta_eff, __nv_bfloat16* __restrict__ gamma_out) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < c * c; i += gridDim.x * blockDim.x) {
    const float g = fmaxf(gamma[i], gamma_bound);
    gamma_out[i] = __float2bfloat16_rn(g * g - pedestal);          // [i (out)][j (in)]: K-major B operand
    if (i < c) { const float b = fmaxf(beta[i], beta_bound); beta_eff[i] = b * b - pedestal; }
  }
}

inline int nb_for(int cout) { return cout <= 16 ? 16 : 128; }
// stride-2 transposed conv with <= 4 output channels (g_s last layer, 128 -> 3): run as ONE 3x3 stride-1 conv to 4 * c_out
// "sub-pixel" channels instead of four phase convs with N = 16 each (an N = 16 MMA costs 39 clk, tools/tc_probe T6)
inline bool subpixel_form(const nic_conv_desc* d) {
  return d->transposed && d->stride == 2 && d->kh == 5 && d->kw == 5 && d->pad == 2 && d->output_padding == 1 && 4 * d->c_out <= 16 && d->c_in >= 64;
}
inline nic_conv_desc subpixel_desc(const nic_conv_desc* d) {
  nic_conv_desc e = *d;
  e.transposed = 0; e.output_padding = 0; e.kh = e.kw = 3; e.stride = 1; e.pad = 1;
  e.c_out = 4 * d->c_out; e.h_out = d->h_in; e.w_out = d->w_in; e.out_c_total = 0; e.out_c_offset = 0;
  return e;
}
inline bool small_cin(const nic_conv_desc* d) { return d->c_in < 64; }

}  // namespace

void set_trace_buffer(void* p) { g_trace_buffer = p; }

int read_and_clear_status() {
  int* d = status_word();
  if (!d) return 0;
  int h = 0;
  if (cudaDeviceSynchronize() != cudaSuccess) return 1;
  if (cudaMemcpy(&h, d, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
  if (h) cudaMemset(d, 0, sizeof(int));
  return h ? 1 : 0;
}

// Packed layout (bf16 elements):
//   c_in >= 64 : [tap][c_out padded to a multiple of nb][c_in]
//   c_in  = 3  : [c_out = 128][k padded to 128], k = (kh * kw_size + kw) * 3 + c   (first layer, conv_first_tc_kernel)
size_t packed_weight_elems_tc(const nic_conv_desc* d, const TapTable& tt) {
  if (d->precision == NIC_PREC_BF16X3) {
    if (small_cin(d)) return packed_first_x3_elems(d->c_out == 192 ? 192 : 128);
    if (last_scatter_applies(d)) return packed_last_scatter_elems(d->c_in);
    if (subpixel_form(d)) return static_cast<size_t>(9) * 16 * 3 * d->c_in;
    const int nbx = nb_for(d->c_out);
    const int cp = (d->c_out + nbx - 1) / nbx * nbx;          // the kernel's c_out padding: N tiles of 128, or one of 16
    return static_cast<size_t>(tt.ntaps) * cp * 3 * d->c_in;
  }
  if (small_cin(d)) return static_cast<size_t>(128) * 128;
  if (subpixel_form(d)) return static_cast<size_t>(9) * 16 * d->c_in;
  const int nb = nb_for(d->c_out);
  const int cout_pad = (d->c_out + nb - 1) / nb * nb;
  return static_cast<size_t>(tt.ntaps) * cout_pad * d->c_in;
}

__global__ void pack_weight_f32_kernel(const float*, float*, int, int, int, int, int, TapTable);

int pack_weight_tc(const nic_conv_desc* d, const TapTable& tt, const float* w_ref, void* w_packed, cudaStream_t st) {
  if (d->precision == NIC_PREC_BF16X3) {
    if (small_cin(d)) {
      if (int rc = check_first_layer(d)) return rc;
      return pack_first_x3(w_ref, w_packed, d->c_out, st);
    }
    if (d->c_in % 64) return fail(NIC_E_UNSUPPORTED, "conv bf16x3: c_in=%d must be a multiple of 64 (or 3 for the first layer)", d->c_in);
    if (last_scatter_applies(d)) return pack_last_scatter(w_ref, w_packed, d->c_in, st);
    if (subpixel_form(d)) {
      const long total = 9L * 16 * 3 * d->c_in;
      pack_weight_subpixel_x3_kernel<<<static_cast<int>((total + 255) / 256), 256, 0, st>>>(w_ref, static_cast<__nv_bfloat16*>(w_packed), d->c_in,
                                                                                         d->c_out, tt);
      return check_launch("pack_weight_subpixel_x3_kernel");
    }
    const int nbx = nb_for(d->c_out);
    const int cp = (d->c_out + nbx - 1) / nbx * nbx;
    const long total = static_cast<long>(tt.ntaps) * cp * 3 * d->c_in;
    const int blocks = static_cast<int>((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    pack_weight_x3_kernel<<<blocks, 256, 0, st>>>(w_ref, static_cast<__nv_bfloat16*>(w_packed), d->c_in, d->c_out, cp, d->kh, d->kw,
                                                  d->transposed, tt);
    return check_launch("pack_weight_x3_kernel");
  }
  if (d->precision != NIC_PREC_BF16) return fail(NIC_E_UNSUPPORTED, "pack_conv_weight: precision %d", d->precision);
  if (small_cin(d)) {
    if (int rc = check_first_layer(d)) return rc;
    pack_first_bf16_kernel<<<64, 256, 0, st>>>(w_ref, static_cast<__nv_bfloat16*>(w_packed));
    return check_launch("pack_first_bf16_kernel");
  }
  if (subpixel_form(d)) {
    if (d->c_in % 64) return fail(NIC_E_UNSUPPORTED, "conv bf16: c_in=%d must be a multiple of 64", d->c_in);
    const long total = 9L * 16 * d->c_in;
    pack_weight_subpixel_bf16_kernel<<<static_cast<int>((total + 255) / 256), 256, 0, st>>>(w_ref, static_cast<__nv_bfloat16*>(w_packed), d->c_in,
                                                                                         d->c_out, tt);
    return check_launch("pack_weight_subpixel_bf16_kernel");
  }
  if (d->c_in % 64) return fail(NIC_E_UNSUPPORTED, "conv bf16: c_in=%d must be a multiple of 64 (or < 64 for the first layer)", d->c_in);
  const int nb = nb_for(d->c_out);
  const int cout_pad = (d->c_out + nb - 1) / nb * nb;
  const long total = static_cast<long>(tt.ntaps) * cout_pad * d->c_in;
  const int blocks = static_cast<int>((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  pack_weight_bf16_kernel<<<blocks, 256, 0, st>>>(w_ref, static_cast<__nv_bfloat16*>(w_packed), d->c_in, d->c_out, cout_pad, d->kh, d->kw,
                                                  d->transposed, tt);
  return check_launch("pack_weight_bf16_kernel");
}

int pack_gdn_tc(int32_t c, float beta_min, const float* beta_raw, const float* gamma_raw, float* beta_eff, void* gamma_packed,
                int32_t precision, cudaStream_t st) {
  if (precision == NIC_PREC_BF16X3) return pack_gdn_x3(c, beta_min, beta_raw, gamma_raw, beta_eff, gamma_packed, st);
  if (precision != NIC_PREC_BF16) return fail(NIC_E_UNSUPPORTED, "pack_gdn: precision %d", precision);
  const float pedestal = static_cast<float>(3.814697265625e-06 * 3.814697265625e-06);
  const float beta_bound = static_cast<float>(sqrt(static_cast<double>(beta_min) + static_cast<double>(pedestal)));
  const float gamma_bound = static_cast<float>(sqrt(static_cast<double>(pedestal)));
  pack_gdn_bf16_kernel<<<(c * c + 255) / 256, 256, 0, st>>>(c, beta_bound, gamma_bound, pedestal, beta_raw, gamma_raw, beta_eff,
                                                            static_cast<__nv_bfloat16*>(gamma_packed));
  return check_launch("pack_gdn_bf16_kernel");
}

size_t conv_workspace_bytes_tc(const nic_conv_desc* d) {
  const bool gdn = d->epilogue == NIC_EPI_GDN || d->epilogue == NIC_EPI_IGDN;
  if (d->precision == NIC_PREC_BF16X3 && gdn) return static_cast<size_t>(d->n) * d->h_out * d->w_out * d->c_out * sizeof(float);
  return 0;
}

// `shuffle`: non-null when `d` is the 3x3 stride-1 sub-pixel form of a stride-2 transposed conv (see conv_fwd_tc); it is the
// ORIGINAL descriptor, whose output tensor the epilogue scatters into.
static int launch_tc(const nic_conv_desc* d, const TapTable& tt, const void* x, const void* w_packed, const float* bias, const void* gdn_gamma,
                     const float* gdn_beta, void* y, cudaStream_t st, const nic_conv_desc* shuffle = nullptr, const int* lo_flag = nullptr) {
  TcParams p{};
  if (int rc = build_tc_geometry(d, tt, &p)) return rc;
  const bool gdn = d->epilogue == NIC_EPI_GDN || d->epilogue == NIC_EPI_IGDN;
  const bool x3 = d->precision == NIC_PREC_BF16X3;
  if (d->in_layout != NIC_LAYOUT_NHWC || d->in_dtype != (x3 ? NIC_DT_BF16X2 : NIC_DT_BF16))
    return fail(NIC_E_UNSUPPORTED, "conv %s: input must be NHWC %s", x3 ? "bf16x3" : "bf16", x3 ? "bf16 pairs" : "bf16");
  if (x3 && gdn) return fail(NIC_E_UNSUPPORTED, "conv bf16x3: the conv kernel has bias / LeakyReLU epilogues only (GDN follows as gdn_x3_kernel)");
  if (d->c_in % 64) return fail(NIC_E_UNSUPPORTED, "conv bf16: c_in=%d must be a multiple of 64", d->c_in);
  if (d->c_out > kMaxCout) return fail(NIC_E_UNSUPPORTED, "conv bf16: c_out=%d exceeds the %d-entry bias table of the kernel", d->c_out, kMaxCout);
  if (gdn && (d->c_out != 128 || !gdn_gamma || !gdn_beta)) return fail(NIC_E_UNSUPPORTED, "conv bf16: the fused GDN epilogue needs c_out = 128 and packed gamma/beta");
  if ((reinterpret_cast<uintptr_t>(x) & 127) || (reinterpret_cast<uintptr_t>(w_packed) & 127)) return fail(NIC_E_BADALIGN, "conv bf16: tensors must be 128-byte aligned for TMA");
  p.n = d->n; p.hin = d->h_in; p.win = d->w_in; p.cin = d->c_in; p.cout = d->c_out; p.hout = d->h_out; p.wout = d->w_out;
  p.nb = nb_for(d->c_out);
  p.cout_pad = (d->c_out + p.nb - 1) / p.nb * p.nb;
  p.n_ntiles = p.cout_pad / p.nb;
  p.nchunks = (x3 ? 3 : 1) * d->c_in / 64;
  p.a_chunk_mod = (x3 ? 2 : 1) * d->c_in / 64;
  p.lo_flag = x3 ? lo_flag : nullptr;
  p.split_out = d->out_dtype == NIC_DT_BF16X2;
  if (p.split_out && (!x3 || d->out_layout != NIC_LAYOUT_NHWC || d->c_out % 64 || d->out_c_total % 64 || d->out_c_offset % 64))
    return fail(NIC_E_UNSUPPORTED, "conv: bf16-pair output needs the bf16x3 arm, NHWC, channel counts / offsets multiples of 64");
  p.epilogue = d->epilogue; p.out_dtype = p.split_out ? NIC_DT_BF16 : d->out_dtype;
  const int chalf = d->out_c_total ? d->out_c_total : d->c_out;
  p.split_lo_off = chalf;
  const int ctot = p.split_out ? 2 * chalf : chalf;
  if (d->out_layout == NIC_LAYOUT_NCHW) { p.ys_n = static_cast<long>(ctot) * d->h_out * d->w_out; p.ys_c = static_cast<long>(d->h_out) * d->w_out; p.ys_h = d->w_out; p.ys_w = 1; }
  else { p.ys_n = static_cast<long>(d->h_out) * d->w_out * ctot; p.ys_h = static_cast<long>(d->w_out) * ctot; p.ys_w = ctot; p.ys_c = 1; }
  const size_t esz = d->out_dtype == NIC_DT_F32 ? 4 : 2;
  p.y = static_cast<uint8_t*>(y) + static_cast<size_t>(d->out_c_offset) * p.ys_c * esz;
  if (!shuffle && p.ys_c == 1 && ((reinterpret_cast<uintptr_t>(p.y) & 15) || (ctot * esz) % 16)) return fail(NIC_E_BADALIGN, "conv bf16: NHWC output rows must be 16-byte aligned");
  p.bias = bias; p.beta = gdn_beta;
  if (shuffle) {
    if (shuffle->out_dtype != NIC_DT_F32) return fail(NIC_E_UNSUPPORTED, "conv bf16: the sub-pixel output path writes fp32");
    const int sct = shuffle->out_c_total ? shuffle->out_c_total : shuffle->c_out;
    p.shuffle_cout = shuffle->c_out; p.bias_mod = shuffle->c_out;
    if (shuffle->out_layout == NIC_LAYOUT_NCHW) { p.ys_n = static_cast<long>(sct) * shuffle->h_out * shuffle->w_out; p.ys_c = static_cast<long>(shuffle->h_out) * shuffle->w_out; p.ys_h = shuffle->w_out; p.ys_w = 1; }
    else { p.ys_n = static_cast<long>(shuffle->h_out) * shuffle->w_out * sct; p.ys_h = static_cast<long>(shuffle->w_out) * sct; p.ys_w = sct; p.ys_c = 1; }
    p.y = static_cast<uint8_t*>(y) + static_cast<size_t>(shuffle->out_c_offset) * p.ys_c * 4;
  }
  p.status = status_word();
  if (!p.status) return fail(NIC_E_CUDA, "conv bf16: cannot allocate the status word");
  { const char* e = getenv("NIC_TC_DEBUG"); p.dbg = e ? atoi(e) : 0; }
  p.dbg_times = reinterpret_cast<long long*>(g_trace_buffer);

  // geometry of the pixel grid the tiles walk
  int gn = d->n, gh = d->h_in, gw = d->w_in;
  const bool pointwise = d->kh == 1 && d->kw == 1 && d->stride == 1 && !d->transposed;
  const long npix = static_cast<long>(d->n) * d->h_in * d->w_in;
  const bool flat = pointwise && npix % kTileW == 0;
  if (flat) {                                    // 1x1: a flat list of pixels, 8 per row -> every block is 128 consecutive pixels
    gn = 1; gh = static_cast<int>(npix / kTileW); gw = kTileW;
    p.flat_hw = d->h_in * d->w_in;
    p.n = 1; p.hin = gh; p.win = gw; p.hout = gh; p.wout = gw;
  }
  p.hp = (p.hout + tt.out_stride - 1) / tt.out_stride;
  p.wp = (p.wout + tt.out_stride - 1) / tt.out_stride;
  // Swapped orientation (weights = the M operand, the 256 pixels of a two-block tile = the N operand of ONE N = 256 MMA) for the
  // layers it is built for: bias / LeakyReLU epilogue, bf16 or bf16-pair NHWC output through TMA, c_out tiles of 128, weights
  // streamed.  It needs the two blocks stacked vertically (one uniform group stride through the patch), like the flat 1x1 case.
  const char* swap_env = getenv("NIC_TC_SWAP");
  const bool out_bf16_tma = !shuffle && d->out_layout == NIC_LAYOUT_NHWC && p.out_dtype == NIC_DT_BF16 && p.nb == 128 && d->c_out % 64 == 0 &&
                            ctot % 8 == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0;
  // Measured (bf16x3, 16 images): transposed convs gain 6-8 % (g_s layer 3: 1.105 -> 1.04 ms); stride-2 convs LOSE ~8 % (an
  // N = 256 MMA over their four 34 x 10 plane patches runs at ~160 clk, not 128) and the small stride-1 layers lose a few us to
  // the heavier transposing epilogue - so the default is transposed convs only; NIC_TC_SWAP=1 forces it wherever it is built,
  // NIC_TC_SWAP=0 disables it.
  const bool swap_ok = !gdn && out_bf16_tma && (d->epilogue == NIC_EPI_BIAS || d->epilogue == NIC_EPI_LRELU);
  // (round 2, after the two-chunk issue loop: the stride-1 layers now gain too - entropy-parameter 1x1s 90 -> 74 / 97 -> 88 us, h_a
  // layer 1 38.6 -> 32.8, h_s layer 3 81 -> 74, context conv 72 -> 67 us; the stride-2 g_a layer 4 still loses, 65 -> 69 us)
  bool swap = swap_ok && (swap_env ? atoi(swap_env) != 0 : (tt.nphases > 1 || tt.in_stride == 1));
  // CTA pairs (conv_tc_kernel<true>): normal orientation, side-by-side two-block tiles, one N tile of 128, an even number of tiles
  // per phase (the two CTAs of a cluster take tiles 2 j and 2 j + 1 of the same phase) and at least two waves of them
  bool pair = false;
  {
    const char* pair_env = getenv("NIC_TC_PAIR");
    const int tx2 = (p.wp + 2 * kTileW - 1) / (2 * kTileW), ty2 = (p.hp + kTileH - 1) / kTileH;
    const long per_phase = static_cast<long>(tx2) * ty2 * p.n;
    // measured (bf16x3, 16 images, same box, results bit-identical): g_a layer 2 743.8 -> 709.3 us, layer 3 212.1 -> 201.6, g_s layer 3
    // 1040.7 -> 1018.7 (against the swapped one-CTA form); g_s layer 2 (1536 tiles in four phases) 271.0 -> 278.4: stays unpaired
    // bf16x3 only by default: the single-pass bf16 arm LOSES with it (whole step 1.79 -> 1.89 ms); never together with the fused GDN
    // epilogue, whose own MMAs and commits are cta_group::1 (a kernel should not mix the two forms)
    const bool worth = x3 && (tt.nphases == 1 || per_phase * tt.nphases >= 16 * kNumSMs);
    pair = (pair_env ? atoi(pair_env) != 0 : worth) && !gdn && !flat && p.nb == 128 && p.n_ntiles <= 2 && p.wp > kTileW && per_phase % 2 == 0 &&
           per_phase * tt.nphases >= 2 * kNumSMs && !getenv("NIC_TC_MT");
    if (pair) swap = false;
  }
  p.pair = pair ? 1 : 0;
  const bool stacked = flat || swap;
  // two M = 128 blocks per tile share every weight slab (halves the L2 -> shared-memory weight traffic, which is
  // what bounds M = 128 tiles: profiles/README.md); side by side for images, stacked for the flat 1x1 case
  p.mt = (stacked ? p.hp > kTileH : p.wp > kTileW) ? 2 : 1;
  {
    // small layers: one block per tile when two-block tiles would leave SMs idle (fewer than two tiles per SM)
    const long tiles2 = static_cast<long>((p.wp + (stacked ? kTileW : 2 * kTileW) - 1) / (stacked ? kTileW : 2 * kTileW)) *
                        ((p.hp + (stacked ? 2 * kTileH : kTileH) - 1) / (stacked ? 2 * kTileH : kTileH)) * p.n * tt.nphases * p.n_ntiles;
    // measured (bf16x3, 16 images, tools/layer_bench.py): with ONE block per tile only one of the two MMA issuers works and its
    // per-tap bookkeeping bounds the tile, so two-block tiles win down to ~half a wave of tiles (h_a layer 1, 96 tiles: 46.9 ->
    // 39.5 us; g_a layer 4, 96 tiles: 98.8 -> 67.9 us; context conv, 192 tiles: 80.8 -> 71.6 us) and lose below (h_a layer 2,
    // 24 tiles: 54.9 -> 67.0 us)
    if (tiles2 < kNumSMs / 2) p.mt = 1;
    if (const char* e = getenv("NIC_TC_MT")) { const int f = atoi(e); if (f == 1) p.mt = 1; else if (f == 2 && (stacked ? p.hp > kTileH : p.wp > kTileW)) p.mt = 2; }   // timing experiments
  }
  if (p.mt == 1) swap = false;                   // one-block tiles: N = 128 either way, keep the normal orientation
  p.swap = swap ? 1 : 0;
  p.blk_roff[0] = p.blk_coff[0] = 0;
  p.blk_roff[1] = stacked ? kTileH : 0; p.blk_coff[1] = stacked ? 0 : kTileW;
  p.tile_h = stacked ? kTileH * p.mt : kTileH; p.tile_w = stacked ? kTileW : kTileW * p.mt;
  p.ph_rows += p.tile_h - kTileH; p.pw_cols += p.tile_w - kTileW;      // build_tc_geometry sized the patch for one block
  p.tiles_x = (p.wp + p.tile_w - 1) / p.tile_w;
  p.tiles_y = (p.hp + p.tile_h - 1) / p.tile_h;
  p.total_tiles = p.tiles_x * p.tiles_y * p.n * p.nphases * p.n_ntiles;
  p.pos_per_wave = 0; p.spatial_tiles = p.tiles_x * p.tiles_y * p.n;
  // layers with several N tiles (1x1 stack: 5 / 5 / 9, h_s, context: 2): N tile innermost, so that a wave's CTAs read one input
  // tile from L2 together instead of sweeping the whole input once per N tile (cold: 2.2x / 3.8x the input from DRAM on the last two
  // 1x1 layers); measured warm: h_s layer 2 53.1 -> 49.6, 1x1 stack 75.0 / 88.5 / 133.6 -> 72.6 / 84.1 / 128.6 us, others unchanged
  p.nt_inner = p.n_ntiles > 1 ? 1 : 0;
  if (const char* e = getenv("NIC_TC_NT_INNER")) p.nt_inner = (atoi(e) != 0 && p.n_ntiles > 1) ? 1 : 0;
  {
    static const bool interleave = !(getenv("NIC_TC_PHASE_ORDER") && atoi(getenv("NIC_TC_PHASE_ORDER")) == 0);
    // measured (bf16x3, 16 images): g_s layer 3 (6144 tiles) 1109 -> 1031 us; layer 2 (1536 tiles, input L2-resident either way)
    // 272.7 -> 273.7, layer 1 (384 tiles) 85.5 -> 88.8 - so only where the input cannot stay in L2 across the phase passes
    // (... i.e. the input does not fit L2: the single-pass bf16 arm's 100 MB input does, and loses 25 us of 1.85 ms to the order)
    const double in_bytes = static_cast<double>(d->n) * d->h_in * d->w_in * d->c_in * (x3 ? 4 : 2);
    if (interleave && in_bytes > 112e6 && p.nphases > 1 && p.total_tiles >= 16 * kNumSMs) {
      p.pos_per_wave = 1;                      // (a flag: both interleaved orders are computed from the slot index)
    }
  }
  p.tail_first = 0; p.tail_n = 0;
  {
    static const bool tail = !(getenv("NIC_TC_TAIL") && atoi(getenv("NIC_TC_TAIL")) == 0);
    const int rem = p.total_tiles % kNumSMs;
    if (tail && !p.swap && p.mt == 2 && p.n_ntiles == 1 && p.nphases == 1 && !p.pos_per_wave && !p.nt_inner && p.nb == 128 &&
        p.total_tiles > 4 * kNumSMs && rem > 0 && 2 * rem <= kNumSMs && rem % 2 == 0) {
      p.tail_first = p.total_tiles - rem; p.tail_n = rem;
      p.total_tiles = p.tail_first + 2 * rem;
    }
  }
  p.nslabs = tt.ntaps;

  // shared memory: A slots | B ring (or resident weights) | gamma | squares
  p.slot_bytes = (p.ph_rows * p.pw_cols * 128 + 1023) / 1024 * 1024;
  p.out_c_offset = d->out_c_offset;
  p.tma_out = (!shuffle && d->out_layout == NIC_LAYOUT_NHWC && p.out_dtype == NIC_DT_BF16 && p.nb == 128 && d->c_out % 64 == 0 &&
               ctot % 8 == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0) ? 1 : 0;
  // f32 NHWC outputs (the conv -> GDN scratch of the bf16x3 arm, y / z before the hand-off): 16-byte scattered stores from the
  // epilogue put it ON the critical path (g_s layer 3, bf16x3: 1.17 ms, 0.91 ms with the stores removed) - stage + TMA store
  if (!p.tma_out && !shuffle && !gdn && d->out_layout == NIC_LAYOUT_NHWC && p.out_dtype == NIC_DT_F32 && p.nb == 128 && d->c_out % 32 == 0 &&
      ctot % 4 == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 && !getenv("NIC_TC_NO_F32_TMA"))
    p.tma_out = 2;      // (y and z, the f32 tensors the latent hand-off reads: small layers, the ring depth does not matter there)
  // bf16-pair outputs in the normal orientation leave through per-warp staging slices (epilogue_block_slices): bit-identical,
  // and the epilogue no longer serialises on its own stores.  NIC_TC_EPI_SLICES=0 keeps the CTA-wide rounds as a cross-check.
  {
    const char* e = getenv("NIC_TC_EPI_SLICES");
    p.epi_slices = (p.split_out && p.tma_out == 1 && !gdn && !p.swap && !(e && atoi(e) == 0)) ? 1 : 0;
  }
  // gamma (32 KB, GDN only) + one tile (32 KB; 64 KB for f32 outputs) that holds the squares for the gamma contraction and
  // then stages the output
  // bf16-pair outputs of layers with a short mainloop (<= 96 tap-chunks per tile: the 1x1 stack, the 3x3 layers, the masked
  // context conv): a second staging tile, so that the hi and lo stores of a block never wait for each other (each
  // cp.async.bulk.wait_group.read right after its store costs 3-5k clk behind the TMA loads in flight - as long as such a
  // layer's whole mainloop)
  const int tapchunks = (tt.ntaps / tt.nphases) * p.nchunks;
  // normal orientation: measured, no gain (the smaller rings cost as much: ep2 96.5 -> 109.8 us) - opt-in only (NIC_TC_STAGE2=1).
  // Swapped orientation: the transposing epilogue then reads every accumulator column once and stores once per block
  // (epilogue_tile_swapped).  Measured (bf16x3, 16 images): it pays on the small multi-tap layers (h_s layers 1, 2: 30.1 -> 26.4,
  // 56.3 -> 52.6 us; h_a layer 1: 34.0 -> 29.3; h_s layer 3: 74.3 -> 70.9) and not on the 1x1 stack (88.7 -> 95.6 us) or the big
  // transposed convs (g_s layer 3: 1069 -> 1081 us incl. its IGDN: the two ring slots it costs weigh as much) - so: swapped,
  // 2 .. 96 tap-chunks per tile, and only if two A slots and four ring slots still fit.  NIC_TC_STAGE2=0 / 1 forces it off / on.
  const char* st2 = getenv("NIC_TC_STAGE2");
  const bool st2_fits = 2 * p.slot_bytes + 4 * 128 * 128 + 4 * 128 * 128 + 1024 <= kMaxDynSmem;
  const bool st2_auto = p.swap && tapchunks <= 96 && tt.ntaps > tt.nphases;
  p.stage2 = (p.split_out && p.tma_out == 1 && !gdn && !p.epi_slices && st2_fits &&
              (st2 ? (atoi(st2) != 0 && (p.swap || tapchunks <= 96)) : st2_auto)) ? 1 : 0;
  const int stage_bytes = p.tma_out == 2 ? 4 * 128 * 128 : ((gdn || p.tma_out) ? (p.stage2 ? 4 : 2) * 128 * 128 : 0);
  const int gdn_bytes = (gdn ? 2 * 128 * 128 : 0) + stage_bytes;
  const int bres_bytes = tt.ntaps * p.nchunks * p.nb * 128;
  p.b_resident = (p.n_ntiles == 1 && p.nb <= 16 && bres_bytes + 2 * p.slot_bytes + gdn_bytes + 1024 <= kMaxDynSmem) ? 1 : 0;
  {
    static const bool perm = !(getenv("NIC_TC_CHUNK_PERM") && atoi(getenv("NIC_TC_CHUNK_PERM")) == 0);
    // For every size, although it only pays when the input cannot stay in L2 (the 8 x 256 x 256 training step, whose inputs do, is
    // 30 us of 3.8 ms faster without it): the chunk order is the fp32 accumulation order, and a pixel's value must not depend on the
    // size of the image or batch around it (tests/test_gpu_scalable.py compares a crop with the full image symbol for symbol)
    p.chunk_perm = (perm && x3 && !p.b_resident) ? 1 : 0;
  }
  p.b_slot_bytes = p.pair ? 64 * 128 : 128 * 128;
  if (p.b_resident) p.lo_flag = nullptr;          // resident weights are indexed by chunk position: always the full list
  int b_bytes;
  if (p.b_resident) {
    b_bytes = (bres_bytes + 1023) / 1024 * 1024; p.nsb = 1;
    p.nsa = 4;
    while (p.nsa > 2 && p.nsa * p.slot_bytes + b_bytes + gdn_bytes + 1024 > kMaxDynSmem) --p.nsa;
  } else {
    const int bslot = p.pair ? 64 * 128 : 128 * 128;
    // prefer a deep weight ring (TMA latency ~1 us vs ~0.13 us of MMA per slab and block), then A slots
    p.nsa = 2; p.nsb = 4;
    if (2 * p.slot_bytes + 4 * bslot + gdn_bytes + 1024 > kMaxDynSmem) {
      if (p.stage2) return fail(NIC_E_UNSUPPORTED, "conv bf16x3: internal: staging tiles do not fit");   // cannot happen: slots of these layers are <= 42 KB
      return fail(NIC_E_UNSUPPORTED, "conv bf16: patch of %d x %d pixels does not fit shared memory", p.ph_rows, p.pw_cols);
    }
    const bool one_tap = tt.ntaps == tt.nphases;       // 1x1: an A slot is consumed per weight slab - balance the rings in slots, not bytes
    if (one_tap) {
      p.nsa = 2; p.nsb = 2;
      for (;;) {
        if (p.nsa <= p.nsb && p.nsa < kMaxSlots && (p.nsa + 1) * p.slot_bytes + p.nsb * bslot + gdn_bytes + 1024 <= kMaxDynSmem) ++p.nsa;
        else if (p.nsb < kMaxBSlots && p.nsa * p.slot_bytes + (p.nsb + 1) * bslot + gdn_bytes + 1024 <= kMaxDynSmem) ++p.nsb;
        else break;
      }
    } else
    for (;;) {
      if (p.nsb < kMaxBSlots && p.nsa * p.slot_bytes + (p.nsb + 1) * bslot + gdn_bytes + 1024 <= kMaxDynSmem && p.nsb < 2 * p.nsa + 2) ++p.nsb;
      else if (p.nsa < kMaxSlots && (p.nsa + 1) * p.slot_bytes + p.nsb * bslot + gdn_bytes + 1024 <= kMaxDynSmem) ++p.nsa;
      else if (p.nsb < kMaxBSlots && p.nsa * p.slot_bytes + (p.nsb + 1) * bslot + gdn_bytes + 1024 <= kMaxDynSmem) ++p.nsb;
      else break;
    }
    {   // timing experiments: NIC_TC_NSA / NIC_TC_NSB force the ring depths (checked against the shared-memory budget)
      const char* ea = getenv("NIC_TC_NSA"); const char* eb = getenv("NIC_TC_NSB");
      const int fa = ea ? atoi(ea) : 0, fb = eb ? atoi(eb) : 0;
      if (fa || fb) {
        const int na = fa ? fa : p.nsa, nb2 = fb ? fb : p.nsb;
        if (na >= 2 && na <= kMaxSlots && nb2 >= 2 && nb2 <= kMaxBSlots && na * p.slot_bytes + nb2 * bslot + gdn_bytes + 1024 <= kMaxDynSmem) { p.nsa = na; p.nsb = nb2; }
      }
    }
    b_bytes = p.nsb * bslot;
  }
  p.off_a = 0; p.off_b = p.nsa * p.slot_bytes; p.off_gamma = p.off_b + b_bytes; p.off_sq = p.off_gamma + (gdn ? 2 * 128 * 128 : 0);
  p.smem_bytes = p.off_sq + stage_bytes + 1024;

  CUtensorMap map_a, map_w, map_g, map_o;
  if (p.split_out && !p.tma_out) return fail(NIC_E_BADALIGN, "conv bf16x3: bf16-pair output must be 16-byte aligned");
  if (int rc = encode_nhwc(&map_a, x, gn, gh, gw, (x3 ? 2 : 1) * d->c_in, p.pw_cols, p.ph_rows, tt.in_stride, 2)) return rc;
  if (int rc = encode_2d(&map_w, w_packed, static_cast<uint64_t>(x3 ? 3 : 1) * d->c_in, static_cast<uint64_t>(tt.ntaps) * p.cout_pad, 64,
                         p.pair ? p.nb / 2 : p.nb)) return rc;
  if (gdn) { if (int rc = encode_2d(&map_g, gdn_gamma, 128, 128, 64, 128)) return rc; }
  else map_g = map_w;
  if (p.tma_out) {
    // the output tensor (all ctot channels), walked with the output stride of the phase decomposition
    const int on = flat ? 1 : d->n, oh = flat ? gh : d->h_out, ow = flat ? gw : d->w_out;
    if (p.epi_slices) {       // one warp's slice: 32 channels x 8 x 4 pixels
      if (int rc = encode_nhwc_c32(&map_o, y, on, oh, ow, ctot, kTileW, 4, tt.out_stride)) return rc;
    } else if (int rc = encode_nhwc(&map_o, y, on, oh, ow, ctot, kTileW, kTileH, tt.out_stride, p.tma_out == 2 ? 4 : 2)) return rc;
  } else map_o = map_w;

  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(conv_tc_kernel<false>), kMaxDynSmem)) return rc;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(conv_tc_kernel<true>), kMaxDynSmem)) return rc;
  const int grid = p.total_tiles < kNumSMs ? p.total_tiles : kNumSMs;
  if (p.pair) {
    if (p.mt != 2 || p.swap || p.b_resident || grid % 2) return fail(NIC_E_UNSUPPORTED, "conv tc: CTA-pair launch with an unsupported tiling");
    if (int rc = check_cuda(launch_pdl_cluster(conv_tc_kernel<true>, grid, kThreads, p.smem_bytes, st, 2, map_a, map_w, map_g, map_o, p), "conv_tc_kernel launch")) return rc;
  } else if (int rc = check_cuda(launch_pdl(conv_tc_kernel<false>, grid, kThreads, p.smem_bytes, st, map_a, map_w, map_g, map_o, p), "conv_tc_kernel launch")) return rc;
  return check_launch("conv_tc_kernel");
}

static int launch_first(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias, const void* gdn_gamma,
                        const float* gdn_beta, void* y, cudaStream_t st) {
  if (int rc = check_first_layer(d)) return rc;
  if (d->in_layout != NIC_LAYOUT_NCHW || d->in_dtype != NIC_DT_F32) return fail(NIC_E_UNSUPPORTED, "conv bf16 (first layer): input must be the NCHW fp32 image");
  if (d->out_layout != NIC_LAYOUT_NHWC || d->out_dtype != NIC_DT_BF16 || d->out_c_total > 128) return fail(NIC_E_UNSUPPORTED, "conv bf16 (first layer): output must be NHWC bf16");
  if (!gdn_gamma || !gdn_beta) return fail(NIC_E_BADSHAPE, "conv bf16 (first layer): packed gamma / beta missing");
  if ((reinterpret_cast<uintptr_t>(y) & 127) || (reinterpret_cast<uintptr_t>(w_packed) & 127)) return fail(NIC_E_BADALIGN, "conv bf16: tensors must be 128-byte aligned for TMA");
  TcParams p{};
  p.epilogue = NIC_EPI_GDN; p.out_dtype = NIC_DT_BF16; p.nb = 128; p.cout = 128; p.tma_out = 1; p.out_stride = 1;
  p.n = d->n; p.hout = d->h_out; p.wout = d->w_out; p.hp = d->h_out; p.wp = d->w_out;
  p.bias = bias; p.beta = gdn_beta; p.y = y;
  p.ys_n = static_cast<long>(d->h_out) * d->w_out * 128; p.ys_h = static_cast<long>(d->w_out) * 128; p.ys_w = 128; p.ys_c = 1;
  p.status = status_word();
  if (!p.status) return fail(NIC_E_CUDA, "conv bf16: cannot allocate the status word");
  { const char* e = getenv("NIC_TC_DEBUG"); p.dbg = e ? atoi(e) : 0; }
  p.dbg_times = reinterpret_cast<long long*>(g_trace_buffer);
  FirstParams f{};
  f.x = static_cast<const float*>(x); f.n = d->n; f.hin = d->h_in; f.win = d->w_in;
  f.tiles_x = (d->w_out + 7) / 8; f.tiles_y = (d->h_out + 15) / 16; f.total_tiles = f.tiles_x * f.tiles_y * d->n;
  f.off_a = 0; f.off_w = 4 * 128 * 128; f.off_gamma = f.off_w + 2 * 128 * 128; f.off_sq = f.off_gamma + 2 * 128 * 128;
  f.off_patch = f.off_sq + 4 * 128 * 128;      // two squares / staging tiles (one per epilogue group)
  const int smem_bytes = f.off_patch + 2 * 3 * kPatchPlane * 4 + 1024 + 64;
  CUtensorMap map_w, map_g, map_o;
  if (int rc = encode_2d(&map_w, w_packed, 128, 128, 64, 128)) return rc;
  if (int rc = encode_2d(&map_g, gdn_gamma, 128, 128, 64, 128)) return rc;
  if (int rc = encode_nhwc(&map_o, y, d->n, d->h_out, d->w_out, 128, kTileW, kTileH, 1, 2)) return rc;
  if (int rc = ensure_dyn_smem(reinterpret_cast<const void*>(conv_first_tc_kernel), 232448 - 2048)) return rc;
  const int grid = f.total_tiles < kNumSMs ? f.total_tiles : kNumSMs;
  conv_first_tc_kernel<<<grid, kFirstThreads, smem_bytes, st>>>(map_w, map_g, map_o, p, f);
  return check_launch("conv_first_tc_kernel");
}

int conv_fwd_tc(const nic_conv_desc* d, const void* x, const void* w_packed, const float* bias, const void* gdn_gamma, const float* gdn_beta,
                void* y, void* workspace, size_t workspace_bytes, cudaStream_t st, const int* lo_flag) {
  TapTable tt;
  if (int rc = build_tap_table(d, &tt)) return rc;
  if (d->precision == NIC_PREC_BF16X3) {
    const bool gdn = d->epilogue == NIC_EPI_GDN || d->epilogue == NIC_EPI_IGDN;
    if (last_scatter_applies(d)) return conv_last_scatter_x3(d, x, w_packed, bias, y, st);
    if (subpixel_form(d)) {
      if (d->epilogue != NIC_EPI_BIAS) return fail(NIC_E_UNSUPPORTED, "conv bf16x3: the sub-pixel path has a bias-only epilogue");
      const nic_conv_desc e = subpixel_desc(d);
      TapTable te;
      if (int rc = build_tap_table(&e, &te)) return rc;
      return launch_tc(&e, te, x, w_packed, bias, nullptr, nullptr, y, st, d);
    }
    if (!gdn) {
      if (small_cin(d)) {            // Conv2d(3, 128, 5, s2, p2) + bias from the NCHW f32 image into a plain NHWC f32 tensor
        if (int rc = check_first_layer(d)) return rc;
        if (d->out_layout != NIC_LAYOUT_NHWC || d->out_dtype != NIC_DT_F32 || d->out_c_total != 0)
          return fail(NIC_E_UNSUPPORTED, "conv bf16x3 (first layer, bias epilogue): output must be a plain NHWC f32 tensor");
        return conv_first_x3(d, x, w_packed, bias, static_cast<float*>(y), st);
      }
      return launch_tc(d, tt, x, w_packed, bias, nullptr, nullptr, y, st, nullptr, lo_flag);
    }
    // GDN / IGDN layer: conv + bias on the tensor cores into an fp32 NHWC scratch, then the hi/lo-split gamma contraction
    // (gdn_x3_kernel) writes the bf16-pair activation
    const size_t need = conv_workspace_bytes_tc(d);
    if (!workspace || workspace_bytes < need) return fail(NIC_E_WORKSPACE, "conv bf16x3 + GDN: workspace %zu < %zu bytes", workspace_bytes, need);
    if (!gdn_gamma || !gdn_beta) return fail(NIC_E_BADSHAPE, "conv: GDN epilogue without gamma/beta");
    if (d->out_dtype != NIC_DT_BF16X2 || d->out_layout != NIC_LAYOUT_NHWC || d->out_c_total != 0)
      return fail(NIC_E_UNSUPPORTED, "conv bf16x3 + GDN: output must be a plain NHWC bf16-pair tensor");
    int pair_in = 0;
    if (small_cin(d) && d->c_out == 128 && !getenv("NIC_X3_FIRST_TWO_KERNELS")) {       // fused conv + GDN (the env switch keeps the two-kernel form testable; 192 channels: two kernels)
      if (int rc = check_first_layer(d)) return rc;
      return conv_first_gdn_x3(d, x, w_packed, bias, gdn_gamma, gdn_beta, y, st);
    }
    if (small_cin(d)) {
      if (int rc = check_first_layer(d)) return rc;
      if (int rc = conv_first_x3(d, x, w_packed, bias, static_cast<float*>(workspace), st)) return rc;
    } else {
      // the conv hands its result to the GDN kernel as a bf16 hi/lo pair tensor (same 4 B / element as f32): that is the output
      // format conv_tc_kernel stores through its 32 KB staging tile + TMA, which leaves the weight ring 6 slots; f32 rows
      // would need 16-byte scattered stores (measured +0.22 ms on g_s layer 3) or a 64 KB staging tile (ring down to 4 slots)
      nic_conv_desc c1 = *d;
      c1.epilogue = NIC_EPI_BIAS; c1.out_dtype = NIC_DT_BF16X2; c1.out_layout = NIC_LAYOUT_NHWC; c1.out_c_total = 0; c1.out_c_offset = 0;
      if (int rc = launch_tc(&c1, tt, x, w_packed, bias, nullptr, nullptr, workspace, st, nullptr, lo_flag)) return rc;
      pair_in = 1;
    }
    return gdn_fwd_tc_x3(workspace, pair_in, static_cast<long>(d->n) * d->h_out * d->w_out, d->c_out,
                         d->epilogue == NIC_EPI_IGDN, gdn_gamma, gdn_beta, y, st);
  }
  if (d->precision != NIC_PREC_BF16) return fail(NIC_E_UNSUPPORTED, "conv: precision %d", d->precision);
  if (subpixel_form(d)) {
    if (d->epilogue != NIC_EPI_BIAS) return fail(NIC_E_UNSUPPORTED, "conv bf16: the sub-pixel path has a bias-only epilogue");
    const nic_conv_desc e = subpixel_desc(d);
    TapTable te;
    if (int rc = build_tap_table(&e, &te)) return rc;
    return launch_tc(&e, te, x, w_packed, bias, nullptr, nullptr, y, st, d);
  }
  if (!small_cin(d)) return launch_tc(d, tt, x, w_packed, bias, gdn_gamma, gdn_beta, y, st);

  return launch_first(d, x, w_packed, bias, gdn_gamma, gdn_beta, y, st);
}

}  // namespace nic

// Debug hook for tools/trace_layer.py (not declared in include/nic.h): a device buffer of 148 * 16 * 8 int64 that
// conv_tc_kernel fills with clock64 stamps of its pipeline roles; NULL switches tracing off.
extern "C" void nic_debug_set_trace(void* device_buffer) { nic::set_trace_buffer(device_buffer); }

extern "C" int nic_pipeline_status(void) { return nic::read_and_clear_status(); }
