// ab_gemm_tcgen05_kernel.cuh — device code of the tcgen05 GEMM (parameters, TMA producer /
// MMA issuer / epilogue warps, 1-CTA and 2-CTA bodies).  Included by ab_gemm_tcgen05.cu
// (ahead-of-time kernels with the plain alpha/beta epilogue) and, with AB_EPILOGUE
// defined, concatenated behind a generated `ab_ep_body` and compiled by NVRTC
// (codegen/gemm_epilogue.py): the Elemwise node that consumes a Gemm/Dot22 result is then
// applied to the accumulator registers before the only store.
#pragma once

// Thread layout.  Ahead-of-time kernels (plain alpha/beta epilogue, ~124 registers): warp 0 =
// TMA producer, warp 1 = MMA issuer, warps 2..9 = epilogue.  Fused-epilogue builds: the
// generated region (read-ahead buffers, 32 accumulator columns, transposes, pair sums) wants
// more than the 168 registers a 320-thread block gets -- ptxas then spills and re-reads
// SR_TID at every use of `lane` (profiles/r02_region2_single_body.txt: 7 % of the samples on
// the instruction behind an S2R) -- so those run 384 threads as three warpgroups: warps 0..3
// (producer, issuer, two idle) shrink to kRegsControl registers and the epilogue warps 4..11
// grow to kRegsEpilogue (setmaxnreg; 128 * 72 + 256 * 216 = 64 512 <= 65 536).
#ifdef AB_EPILOGUE
constexpr int kGemmThreads = kThreadsFused;
constexpr int kEpiWarp0 = 4;
#define AB_SETMAXNREG_CONTROL() asm volatile("setmaxnreg.dec.sync.aligned.u32 72;")
#define AB_SETMAXNREG_EPILOGUE() asm volatile("setmaxnreg.inc.sync.aligned.u32 216;")
#else
constexpr int kGemmThreads = kThreads;
constexpr int kEpiWarp0 = 2;
#define AB_SETMAXNREG_CONTROL()
#define AB_SETMAXNREG_EPILOGUE()
#endif
constexpr int kEpiThreads = 256;  // 8 epilogue warps

struct GemmParams {
  long long M, N, K;      // K in elements of the packed type
  float alpha, beta;
  float* C;
  long long c_rs, c_cs;
  const float* Cin;       // beta term source (== C for the in-place Gemm, another buffer otherwise)
  long long cin_rs, cin_cs;
  int block_n;            // 64 / 128 / 256
  int acc_stages;         // TMEM accumulator stages (2 -> epilogue overlaps the next segment)
  int seg_kblocks;        // k-blocks accumulated inside the tensor core before the epilogue
                          // folds the partial sum into its FP32 registers (see "segments")
  int group_m;            // tile rows per group of the grouped unit order (AB_UNIT_DECODE)
  int k_splits;           // split-K: work unit = (K range, tile)
  int kb_per_split;       // k-blocks per K range
  float* partial;         // [k_splits - 1][M][N] alpha * (A@B over K range s), s >= 1
  int stages;
  int nparts;             // 1, or 2 for the hi/lo split (3 MMAs per k-step)
  int k_elems_per_row;    // K elements per stage = per 128-byte K-major row: 32 (tf32) / 64 (bf16)
  int a_tile_bytes, b_tile_bytes;
  int a_mn, b_mn;         // operand is MN-major
  int a_mn3d, b_mn3d;     // ... and its tensor map is 3-D {128 B of MN, K rows, MN chunks}: the
                          // whole tile arrives with ONE bulk copy instead of one per chunk
                          // (measured: every extra cp.async.bulk.tensor per k-block costs the
                          // 2-CTA mainloop ~0.1 ms of a 2.2 TFLOP product)
  int a_chunks, b_chunks; // MN-major: 128-byte MN chunks per tile (tile_rows * elem_size / 128)
  int chunk_bytes;        // MN-major: k_elems_per_row rows * 128 B
  int mn_per_chunk;       // MN-major: elements per chunk (128 / elem_size)
  int a_kstep, b_kstep;   // descriptor advance per MMA K-step: 32 B (K-major) or umma_k rows * 128 B
  uint32_t idesc;
  // fused consumer (AB_EPILOGUE builds only; zero otherwise): out = ab_ep_body(v, e0..e3)
  // with v = alpha*acc + beta*Cin and e_k = ep_ptr[k][row * ep_rs[k] + col * ep_cs[k]]
  // (stride 0 = broadcast); `shadow` receives the bf16 copy of out as a [M, shadow_pitch]
  // K-major operand plane for the GEMM that consumes it next
  const float* ep_ptr[4];
  long long ep_rs[4], ep_cs[4];
  // the epilogue program yields AB_EP_NOUT values per element.  Value 0 goes to C (when C is
  // not null), value k >= 1 to out_ptr[k] ([M, out_rs[k]] rows, unit column stride; null =
  // not materialised); shadow[k] (optional) receives the bf16 copy of value k as a
  // [M, shadow_pitch[k]] K-major operand plane for the GEMM that consumes it next.
  float* out_ptr[3];
  long long out_rs[3];
  void* shadow[3];
  long long shadow_pitch[3];
  // shadow_t (optional, value AB_EP_TPLANE only): the TRANSPOSED bf16 copy, an [N, shadow_t_pitch]
  // plane whose rows are the columns of the value -- the K-major operand of a product that
  // contracts over the ROWS of the value (h.T @ dout, X.T @ dpre: both operands of a weight
  // gradient).  Read as an MN-major operand instead, the natural plane costs the tensor pipe
  // 10-28 % of its cycles (profiles/r02_dw_layouts_ncu.txt).
  void* shadow_t;
  long long shadow_t_pitch;
  // reductions of one value each, accumulated in float64 like the reference's CAReduce
  // (tensor/elemwise.py:1371-1385): colsum_ws[rb][col] = sum over the 32 rows of row block
  // rb of value AB_EP_COLSUM; fullsum_ws[rb][cb] = sum of value AB_EP_FULLSUM over row block
  // rb and column block cb (half a tile).  A second, deterministic pass adds the partials.
  double* colsum_ws;
  double* fullsum_ws;
  long long fullsum_cols;
  // L2 eviction priority of the operands' tiles (make_l2_policy): a weight matrix that every
  // tile row re-reads is kept (evict_last) against the stream of the large operand and of the
  // epilogue's reads and writes (those use .cs accesses).  Without it the 32 MB W of cfg3 was
  // fetched from DRAM ~50 times per product (dram__bytes_read 2.3-5.1 GB per launch against
  // 0.5-1.5 GB of operands, profiles/r02_bench_step_ncu_v2.txt).
  int a_l2, b_l2;
};

// one operand tile -> shared memory.  K-major: a single box {128 B of K, tile rows};
// MN-major: one box {128 B of MN, BLOCK_K rows} per chunk.
// Loop-invariant description of one operand's tile loads.  The producer and the MMA issuer
// copy what they need from GemmParams into locals BEFORE their loops: the kernel parameter
// lives in constant memory, every mbarrier / TMA asm statement carries a "memory" clobber, and
// a field read through `p` inside the loop is re-loaded (LDCU + dependent UISETP) after each
// of them -- the single producer thread of the MN-major weight-gradient products spent ~540
// of the 770 cycles per k-block on that (profiles/r02_region2_fp64_stalls.txt, dW launches).
struct OperandLoad {
  int mn_major, chunks, mn3d, chunk_bytes, mn_per_chunk;
  uint64_t policy;
};
__device__ __forceinline__ OperandLoad operand_load_a(const GemmParams& p) {
  return OperandLoad{p.a_mn, p.a_chunks, p.a_mn3d, p.chunk_bytes, p.mn_per_chunk, make_l2_policy(p.a_l2)};
}
__device__ __forceinline__ OperandLoad operand_load_b(const GemmParams& p) {
  return OperandLoad{p.b_mn, p.b_chunks, p.b_mn3d, p.chunk_bytes, p.mn_per_chunk, make_l2_policy(p.b_l2)};
}
__device__ __forceinline__ void load_tile(uint8_t* dst, const CUtensorMap* map, uint64_t* bar,
                                          int kc, int mn0, const OperandLoad& o) {
  if (!o.mn_major) {
    tma_load_2d_hint(dst, map, bar, kc, mn0, o.policy);
  } else if (o.mn3d) {
    tma_load_3d(dst, map, bar, 0, kc, mn0 / o.mn_per_chunk);
  } else {
    for (int c = 0; c < o.chunks; ++c)
      tma_load_2d_hint(dst + c * o.chunk_bytes, map, bar, mn0 + c * o.mn_per_chunk, kc, o.policy);
  }
}

// ---------------------------------------------------------------------- segments
// The tensor core adds each MMA's products into the FP32 accumulator with truncation
// (round toward zero), a bias that grows linearly with the number of accumulation steps:
// measured on B200, an unsegmented 3xTF32 K = 4096 product is ~3e-5 from the FP64 result
// where a true-fp32 sgemm is ~4e-7 (tests/test_gpu_blas.py::test_gemm_long_k_accuracy).
// So the K loop is cut into segments of seg_kblocks k-blocks: each segment starts a fresh
// TMEM accumulator, and the epilogue warps add the finished segment into FP32 registers
// with round-to-nearest while the tensor core works on the next segment in the other
// TMEM stage.  For precision 0 a segment is 128 K elements (48 truncating steps); the
// tf32 / bf16 policies keep the whole K loop in one segment.
constexpr int kAccRegs = 128;  // accumulator columns per epilogue thread (BLOCK_N 256 / 2)

__device__ __forceinline__ void fold_segment(float (&acc)[kAccRegs], uint32_t t_acc, int nchunks,
                                             bool first) {
#pragma unroll
  for (int c = 0; c < kAccRegs / 32; ++c) {
    if (c < nchunks) {
      uint32_t r[32];
      tmem_ld_32x32b_x32(t_acc + (uint32_t)(c * 32), r);
      if (first) {
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[c * 32 + j] = __uint_as_float(r[j]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[c * 32 + j] += __uint_as_float(r[j]);
      }
    }
  }
}

// C[row, n0 + ...] = alpha * acc + beta * Cin for one thread's row and column range
// 8 consecutive floats: one 256-bit access (sm_100 LDG/STG.256) when 32-byte aligned, else
// two 128-bit ones (16-byte alignment is the caller's precondition)
// (PTX ISA 8.8 = CUDA 12.9; an older NVRTC, e.g. the 12.8 one bundled with PyTorch that wins
// the SONAME race in a Python process, only knows 128-bit vectors)
#if defined(__CUDACC_VER_MAJOR__) && (__CUDACC_VER_MAJOR__ * 100 + __CUDACC_VER_MINOR__ >= 1209)
#define AB_HAS_V8 1
#else
#define AB_HAS_V8 0
#endif
// STREAM: the access belongs to a fused epilogue region -- [M, N] operands read once and values
// written once, far larger than L2: evict-first, so that they do not push the products' small
// operand (a weight matrix, GemmParams::b_l2) out of L2.  The plain alpha/beta epilogue keeps
// the default policy (a small result is usually the next node's operand).
template <bool STREAM>
__device__ __forceinline__ void ld8(const float* q, float (&o)[8], bool wide) {
#if AB_HAS_V8
  if (wide) {
    if (STREAM)
      asm volatile("ld.global.L1::no_allocate.L2::evict_first.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                   : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3]), "=f"(o[4]), "=f"(o[5]), "=f"(o[6]), "=f"(o[7])
                   : "l"(q));
    else
      asm volatile("ld.global.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                   : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3]), "=f"(o[4]), "=f"(o[5]), "=f"(o[6]), "=f"(o[7])
                   : "l"(q));
  } else
#endif
  {
    const float4 a = STREAM ? __ldcs(reinterpret_cast<const float4*>(q)) : *reinterpret_cast<const float4*>(q);
    const float4 b = STREAM ? __ldcs(reinterpret_cast<const float4*>(q + 4)) : *reinterpret_cast<const float4*>(q + 4);
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
  }
}
template <bool STREAM>
__device__ __forceinline__ void st8(float* q, const float (&v)[8], bool wide) {
#if AB_HAS_V8
  if (wide) {
    if (STREAM)
      asm volatile("st.global.L2::evict_first.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(q), "f"(v[0]), "f"(v[1]),
                   "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                   : "memory");
    else
      asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(q), "f"(v[0]), "f"(v[1]), "f"(v[2]),
                   "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                   : "memory");
  } else
#endif
  {
    if (STREAM) {
      __stcs(reinterpret_cast<float4*>(q), make_float4(v[0], v[1], v[2], v[3]));
      __stcs(reinterpret_cast<float4*>(q + 4), make_float4(v[4], v[5], v[6], v[7]));
    } else {
      *reinterpret_cast<float4*>(q) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(q + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
}

#ifndef AB_EP_STAGED
#define AB_EP_STAGED 0
#endif
constexpr int kStageBytesPerWarp = 32 * 32 * 4;                     // one 32 x 32 float32 chunk
constexpr int kStageBytes = (kEpiThreads / 32) * kStageBytesPerWarp;  // behind the operand ring

struct EpilogueOut {
  const GemmParams& p;
  bool vec_ok, wide_out, wide_in;
  uint32_t stage;  // AB_EP_STAGED builds: shared-space address of this warp's 4 KB (see fused_reduce)
  __device__ explicit EpilogueOut(const GemmParams& p_, uint32_t stage_ = 0) : p(p_), stage(stage_) {
    vec_ok = (p.c_cs == 1) && ((p.c_rs & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0) &&
             (p.beta == 0.0f || ((p.cin_cs == 1) && ((p.cin_rs & 3) == 0) &&
                                 ((reinterpret_cast<uintptr_t>(p.Cin) & 15) == 0)));
    wide_out = ((p.c_rs & 7) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 31) == 0);
    wide_in = ((p.cin_rs & 7) == 0) && ((reinterpret_cast<uintptr_t>(p.Cin) & 31) == 0);
  }
  // split-K: alpha * acc of K range `split` (>= 1) into its [M, N] scratch plane
  __device__ __forceinline__ void store_partial(const float (&acc)[kAccRegs], long long row,
                                                long long n0, int nchunks, int split) const {
    if (row >= p.M) return;
    float* prow = p.partial + ((long long)(split - 1) * p.M + row) * p.N;
    const bool vec = (p.N & 3) == 0;
#pragma unroll
    for (int c = 0; c < kAccRegs / 32; ++c) {
      if (c < nchunks) {
        const long long col0 = n0 + c * 32;
        if (vec && col0 + 32 <= p.N) {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(prow + col0 + j) =
                make_float4(p.alpha * acc[c * 32 + j], p.alpha * acc[c * 32 + j + 1],
                            p.alpha * acc[c * 32 + j + 2], p.alpha * acc[c * 32 + j + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (col0 + j < p.N) prow[col0 + j] = p.alpha * acc[c * 32 + j];
        }
      }
    }
  }
  __device__ __forceinline__ void store(const float (&acc)[kAccRegs], long long row, long long n0,
                                        int nchunks) const {
    if (row >= p.M) return;
    float* crow = p.C + row * p.c_rs;
    const float* irow = p.Cin + row * p.cin_rs;
#pragma unroll
    for (int c = 0; c < kAccRegs / 32; ++c) {
      if (c < nchunks) {
        const long long col0 = n0 + c * 32;
        if (vec_ok && col0 + 32 <= p.N) {
          // 8 columns per step: one 256-bit access per 32-byte sector where the rows are
          // 32-byte aligned (each L2 sector is touched by one request instead of two)
#pragma unroll
          for (int j = 0; j < 32; j += 8) {
            float v[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) v[t] = p.alpha * acc[c * 32 + j + t];
            if (p.beta != 0.0f) {
              float o[8];
              ld8<false>(irow + col0 + j, o, wide_in);
#pragma unroll
              for (int t = 0; t < 8; ++t) v[t] += p.beta * o[t];
            }
            st8<false>(crow + col0 + j, v, wide_out);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const long long col = col0 + j;
            if (col < p.N) {
              float v = p.alpha * acc[c * 32 + j];
              if (p.beta != 0.0f) v += p.beta * irow[col * p.cin_cs];
              crow[col * p.c_cs] = v;
            }
          }
        }
      }
    }
  }
#ifdef AB_EPILOGUE
  // ---- fused consumer region (codegen/gemm_epilogue.py) -------------------------------
  // The generated AB_EP_EVAL(V, E, T, O) evaluates the region's scalar program on
  // v = alpha*acc + beta*Cin and the memory operands E[k][T], leaving its AB_EP_NOUT values
  // in O[0..][T].  Contract (gemm_run refuses the fused launch otherwise): N % 8 == 0, every
  // matrix that is read or written 8 columns at a time (C, Cin, extra outputs, operands with
  // unit column stride) has 16-byte aligned rows.
  //
  // The work is organised per 32-column chunk of one accumulator row (`fused_chunk`), so that
  // the body exists ONCE in the instruction stream: an epilogue unrolled over all 128
  // columns of a thread (tanh, IEEE division, float64 sums per element) is several hundred KB
  // of SASS, which every warp re-fetches from L2 for every tile (measured: the region with
  // two values and two reductions ran 1.5 ms slower than its five separate kernels).
  // v: the [1, 1] operands' values; rcp: ab_uniform_rcp of the statically [1, 1] ones, udiv:
  // all of those are exact reciprocals, so the divisions by them may multiply (AB_EP_UDIV
  // builds; codegen/gemm_epilogue.py)
  struct FusedScalars { float v[4]; float rcp[4]; bool is[4]; bool vec[4]; bool udiv; };
  // Sums of the region are kept as unevaluated float pairs (hi + lo, error-free TwoSum) while
  // they stay inside a thread or a warp, and become float64 where they leave it: the FP64
  // pipe of this part retires a warp-wide DADD every ~20 cycles, and one DADD + one F2F.F64
  // per element made the epilogue of the region with two reductions the critical path (ncu,
  // profiles/r02_region2_fp64_stalls.txt: 47 % of the epilogue warps' samples on DADD,
  // stall_math).  A pair carries ~48 bits: the float64 accumulator of the reference's
  // CAReduce (tensor/elemwise.py:1371-1385) to well below the float32 rounding of the result.
  struct FF { float hi, lo; };
  static __device__ __forceinline__ void ff_add(FF& a, float x) {
    const float t = __fadd_rn(a.hi, x);
    const float bp = __fsub_rn(t, a.hi);
    a.lo = __fadd_rn(a.lo, __fadd_rn(__fsub_rn(a.hi, __fsub_rn(t, bp)), __fsub_rn(x, bp)));
    a.hi = t;
  }
  static __device__ __forceinline__ void ff_add(FF& a, const FF& b) {
    const float lo = a.lo;
    a.lo = 0.0f;
    ff_add(a, b.hi);
    a.lo = __fadd_rn(a.lo, __fadd_rn(lo, b.lo));
  }
  // non-finite sums: hi already is the inf / nan the float64 sum would be (lo is nan then)
  static __device__ __forceinline__ double ff_double(const FF& a) {
    return (a.hi - a.hi == 0.0f) ? (double)a.hi + (double)a.lo : (double)a.hi;
  }
  __device__ __forceinline__ FusedScalars load_scalars() const {
    FusedScalars s;
    s.udiv = true;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      s.is[k] = k < AB_EP_NOPS && (is_scalar_op(k) || (p.ep_rs[k] == 0 && p.ep_cs[k] == 0));  // a [1,1] operand
      s.v[k] = s.is[k] ? p.ep_ptr[k][0] : 0.0f;
      s.rcp[k] = is_scalar_op(k) ? ab_uniform_rcp(s.v[k]) : 0.0f;
      if (is_scalar_op(k) && s.rcp[k] == 0.0f) s.udiv = false;
      s.vec[k] = k < AB_EP_NOPS && (is_row_op(k) || (!is_scalar_op(k) && p.ep_rs[k] == 0 && p.ep_cs[k] == 1));  // a [1,N] row (a bias)
    }
    return s;
  }
  // SKIP: the value that leaves through the shared-memory staging buffer instead (-1: none)
  template <int SKIP>
  __device__ __forceinline__ void put_outputs(const float (&o)[AB_EP_NOUT][8], long long row, long long col) const {
#pragma unroll
    for (int k = 0; k < AB_EP_NOUT; ++k) {
      if (k == SKIP) continue;
      float* dst = k == 0 ? p.C : p.out_ptr[k];
      const long long rs = k == 0 ? p.c_rs : p.out_rs[k];
      if (dst)
        st8<true>(dst + row * rs + col, o[k], ((rs & 7) == 0) && ((reinterpret_cast<uintptr_t>(dst) & 31) == 0));
      if (p.shadow[k]) {
        uint32_t h[4];
#pragma unroll
        for (int t = 0; t < 4; ++t)
          asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h[t]) : "f"(o[k][2 * t + 1]), "f"(o[k][2 * t]));
        uint16_t* sp = static_cast<uint16_t*>(p.shadow[k]) + row * p.shadow_pitch[k] + col;
        __stcs(reinterpret_cast<uint4*>(sp), make_uint4(h[0], h[1], h[2], h[3]));
      }
    }
  }
  // Matrix-shaped reads of a 32-column chunk (the Gemm's z; one [M, N] operand such as h in
  // g * (1 - h^2)) are issued as one batch, ONE CHUNK AHEAD of their use (store_fused*): the
  // loads of all four column groups are in flight together and their DRAM latency passes
  // under the evaluation of the previous chunk.  Loaded group by group right before their
  // use, such an epilogue is latency-bound (16 dependent round trips per tile, tensor pipe
  // 52-66 % active against 71-74 % without such a read, profiles/r02_bench_step_ncu.txt);
  // loaded per chunk but consumed at once, it still waits one DRAM latency per chunk (19 % of
  // the epilogue warps' samples, profiles/r02_region2_fp64_stalls.txt).
  //
  // A [1, N] operand (a bias row) is the same for all 32 rows of a warp: lane l fetches the
  // value of column col0 + l (one coalesced 128-byte read per chunk, a chunk ahead like the
  // matrices) and the evaluation takes column j's value from lane j by shuffle.  Read through
  // ld8 per column group instead, every one of the four groups of a chunk waits for an L2
  // round trip (L1 is swept by the matrix reads): 13 % of the epilogue warps' samples in the
  // region with Y and b2 (profiles/r02_region2_after_pairs.txt).
  // AB_EP_ROWMASK: operands known at code-generation time to be [1, N] rows.  Those are read as
  // 32 values per lane with eight 128-bit loads at a warp-uniform address (one wavefront each, L1
  // hits after the first warp of the CTA), a chunk ahead, instead of one value per lane plus 32
  // SHFL.IDX per chunk at the point of use: the shuffles were the top short-scoreboard / MIO
  // stall of region 1 (profiles/r02_bench_step_ncu_v2.txt).  A row operand that is only
  // recognised at run time keeps the one-register shuffle path.
#ifndef AB_EP_ROWMASK
#define AB_EP_ROWMASK 0
#endif
#ifndef AB_EP_SCALARMASK
#define AB_EP_SCALARMASK 0
#endif
  static __device__ __forceinline__ constexpr int popc4(unsigned m) {  // NVRTC has no __builtin_popcount
    return (int)((m & 1u) + ((m >> 1) & 1u) + ((m >> 2) & 1u) + ((m >> 3) & 1u));
  }
  static constexpr int kRowOps = ((AB_EP_ROWMASK) & 1) + (((AB_EP_ROWMASK) >> 1) & 1) +
                                 (((AB_EP_ROWMASK) >> 2) & 1) + (((AB_EP_ROWMASK) >> 3) & 1);
  static __device__ __forceinline__ constexpr bool is_row_op(int k) { return ((AB_EP_ROWMASK >> k) & 1) != 0; }
  static __device__ __forceinline__ constexpr bool is_scalar_op(int k) { return ((AB_EP_SCALARMASK >> k) & 1) != 0; }
  static __device__ __forceinline__ constexpr int row_slot(int k) {
    return popc4((unsigned)AB_EP_ROWMASK & ((1u << k) - 1u));
  }
  struct ChunkPre {
    // [M, N] reads of the next chunk.  Register-only builds: this lane's row, 32 columns.
    // AB_EP_STAGED builds: the COALESCED layout -- q[i] = row 4 i + lane / 8 of the warp's 32,
    // columns 4 (lane % 8) .. + 3, so that every LDG.128 covers four full 128-byte lines
    // (read row-per-lane, an instruction touches 32 lines, 16 bytes of each: the loads then
    // queue in the LSU like the stores did, profiles/r02_bench_step_ncu_v3.txt) -- and turned
    // into the row-per-lane layout through the staging buffer at the top of fused_eval.
#if AB_EP_CIN
#if AB_EP_STAGED
    float4 cinq[8];
#else
    float cin[32];
#endif
#endif
#if AB_EP_PRE_OP >= 0
#if AB_EP_STAGED
    float4 opq[8];
#else
    float op[32];
#endif
#endif
    float vec[AB_EP_NOPS > 0 ? AB_EP_NOPS : 1];
    float rowv[kRowOps > 0 ? kRowOps : 1][32];
  };
  // EDGE = false: the warp's 32 rows and the tile's columns are all inside [M, N] (no tests)
  template <bool EDGE = true>
  __device__ __forceinline__ void prefetch_chunk(ChunkPre& pre, long long row, long long col0, bool live,
                                                 const FusedScalars& sc, int lane) const {
    const long long r = live ? row : 0;
    (void)r; (void)sc; (void)pre; (void)col0;
#pragma unroll
    for (int k = 0; k < AB_EP_NOPS; ++k) {
      if (is_row_op(k)) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          // N % 8 == 0 and 16-byte aligned rows (the fused launch's contract)
          const float4 q = (!EDGE || col0 + j < p.N) ? __ldg(reinterpret_cast<const float4*>(p.ep_ptr[k] + col0 + j))
                                                     : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
          float* d = &pre.rowv[row_slot(k)][j];
          d[0] = q.x; d[1] = q.y; d[2] = q.z; d[3] = q.w;
        }
      } else if (sc.vec[k]) {
        pre.vec[k] = (!EDGE || col0 + lane < p.N) ? __ldg(p.ep_ptr[k] + col0 + lane) : 0.0f;
      }
    }
#if AB_EP_STAGED
    {
      const long long row0 = row - lane, col = col0 + 4 * (lane & 7);
      (void)row0; (void)col;
#if AB_EP_CIN
      if (p.beta != 0.0f) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const long long grow = row0 + 4 * i + (lane >> 3);
          pre.cinq[i] = (!EDGE || (grow < p.M && col < p.N)) ? __ldcs(reinterpret_cast<const float4*>(p.Cin + grow * p.cin_rs + col))
                                                             : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
      }
#endif
#if AB_EP_PRE_OP >= 0
      {
        // a unit-stride [M, N] matrix (the launch checks it, GemmEpilogueFusion._operands_fit)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const long long grow = row0 + 4 * i + (lane >> 3);
          pre.opq[i] = (!EDGE || (grow < p.M && col < p.N))
                           ? __ldcs(reinterpret_cast<const float4*>(p.ep_ptr[AB_EP_PRE_OP] + grow * p.ep_rs[AB_EP_PRE_OP] + col))
                                                            : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        }
      }
#endif
    }
#else
#if AB_EP_CIN
    if (live && p.beta != 0.0f) {
#pragma unroll
      for (int j = 0; j < 32; j += 8)
        if (col0 + j < p.N) ld8<true>(p.Cin + r * p.cin_rs + col0 + j, *reinterpret_cast<float(*)[8]>(&pre.cin[j]), wide_in);
    }
#endif
#if AB_EP_PRE_OP >= 0
    if (live) {
      const bool wide = ((reinterpret_cast<uintptr_t>(p.ep_ptr[AB_EP_PRE_OP]) & 31) == 0) && ((p.ep_rs[AB_EP_PRE_OP] & 7) == 0);
#pragma unroll
      for (int j = 0; j < 32; j += 8)
        if (col0 + j < p.N)
          ld8<true>(p.ep_ptr[AB_EP_PRE_OP] + r * p.ep_rs[AB_EP_PRE_OP] + col0 + j, *reinterpret_cast<float(*)[8]>(&pre.op[j]), wide);
    }
#endif
#endif
  }
#if AB_EP_STAGED
  // coalesced layout (ChunkPre) -> the staging buffer, rows of the warp's 32 as in the tile
  __device__ __forceinline__ void stage_in(const float4 (&q)[8], int lane) const {
#pragma unroll
    for (int i = 0; i < 8; ++i) sts128(stage + 4u * st_off(4 * i + (lane >> 3), lane & 7), q[i].x, q[i].y, q[i].z, q[i].w);
    __syncwarp();
  }
  // columns j .. j + 7 of this lane's row
  __device__ __forceinline__ void stage_group(int j, float (&out)[8], int lane) const {
    const float4 a = lds128(stage + 4u * st_off(lane, j >> 2)), b = lds128(stage + 4u * st_off(lane, (j >> 2) + 1));
    out[0] = a.x; out[1] = a.y; out[2] = a.z; out[3] = a.w; out[4] = b.x; out[5] = b.y; out[6] = b.z; out[7] = b.w;
  }
  // coalesced layout (ChunkPre) -> this lane's row, through the staging buffer
  __device__ __forceinline__ void restage(const float4 (&q)[8], float (&out)[32], int lane) const {
    stage_in(q, lane);
#pragma unroll
    for (int g = 0; g < 8; g += 2) stage_group(4 * g, *reinterpret_cast<float(*)[8]>(&out[4 * g]), lane);
    __syncwarp();
  }
#endif
  // AB_EP_LAZY: the region reads ONE [M, N] operand (Cin or the read-ahead matrix).  It stays in
  // the staging buffer and each group of 8 columns reads its values right before their use, from
  // this lane's own row -- the slots the group's value is staged to next, which no other lane
  // touches before fused_reduce's __syncwarp.  Read into 32 registers at the top of the chunk
  // instead, they are spilled in the region with Y, b2 and the loss (1.5 KB of local traffic
  // per chunk and warp).
#define AB_EP_LAZY (AB_EP_STAGED && (AB_EP_CIN + (AB_EP_PRE_OP >= 0 ? 1 : 0)) == 1)
  // ---- one 32-column chunk of one accumulator row, in two parts -------------------------
  // fused_eval:   x[32] (raw accumulator values of columns col0 .. col0+31 of `row`) -> the
  //               region's values; consumes the read-ahead buffer `pre`, stores the outputs and
  //               their natural bf16 planes, adds to the thread's total `fs`, and leaves the
  //               value that is reduced / transposed in x[] (0 for rows and columns outside).
  // fused_reduce: the cross-lane part: column sums of the warp's 32 rows and the transposed
  //               bf16 plane.
  // The caller issues the NEXT chunk's reads between the two: `pre` is dead after fused_eval,
  // and the ~300 shuffle/select instructions of fused_reduce give those reads their latency.
  // (Two alternating buffers and a loop body of two chunks did the same at twice the code:
  // ~4900 SASS instructions per iteration, 35 % of the epilogue warps' samples waiting for
  // instruction fetch -- stall_no_inst, profiles/r02_region2_tplane_icache.txt.)
  // UDIV: multiply by the reciprocals of the [1, 1] divisors (FusedScalars::udiv holds)
  template <bool EDGE = true, bool UDIV = false>
  __device__ __forceinline__ void fused_eval(float (&x)[32], long long row, long long col0, bool live,
                                             int lane, const FusedScalars& sc, FF& fs, const ChunkPre& pre) const {
    const long long r = live ? row : 0;
    (void)lane; (void)fs;
#if AB_EP_LAZY
#if AB_EP_CIN
    if (p.beta != 0.0f) stage_in(pre.cinq, lane);
#else
    stage_in(pre.opq, lane);
#endif
#elif AB_EP_STAGED
#if AB_EP_CIN
    float cin_l[32];
    if (p.beta != 0.0f) restage(pre.cinq, cin_l, lane);
#endif
#if AB_EP_PRE_OP >= 0
    float op_l[32];
    restage(pre.opq, op_l, lane);
#endif
#else
#if AB_EP_CIN
    const float (&cin_l)[32] = pre.cin;
#endif
#if AB_EP_PRE_OP >= 0
    const float (&op_l)[32] = pre.op;
#endif
#endif
#pragma unroll
    for (int j = 0; j < 32; j += 8) {
      const long long col = col0 + j;
      // row operands: column j + t's value sits in lane j + t (all 32 lanes take part)
      float ev[AB_EP_NOPS > 0 ? AB_EP_NOPS : 1][8];
#pragma unroll
      for (int k = 0; k < AB_EP_NOPS; ++k) {
        if (is_row_op(k)) {
#pragma unroll
          for (int t = 0; t < 8; ++t) ev[k][t] = pre.rowv[row_slot(k)][j + t];
        } else if (sc.vec[k]) {
#pragma unroll
          for (int t = 0; t < 8; ++t) ev[k][t] = __shfl_sync(0xffffffffu, pre.vec[k], j + t);
        }
      }
      if (!EDGE || (live && col < p.N)) {  // N % 8 == 0: a group of 8 columns is inside or outside as a whole
        float v[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = p.alpha * x[j + t];
        if (p.beta != 0.0f) {
#if AB_EP_CIN
#if AB_EP_LAZY
          float cin_g[8];
          stage_group(j, cin_g, lane);
#pragma unroll
          for (int t = 0; t < 8; ++t) v[t] += p.beta * cin_g[t];
#else
#pragma unroll
          for (int t = 0; t < 8; ++t) v[t] += p.beta * cin_l[j + t];
#endif
#else
          float ci[8];
          ld8<true>(p.Cin + r * p.cin_rs + col, ci, wide_in);
#pragma unroll
          for (int t = 0; t < 8; ++t) v[t] += p.beta * ci[t];
#endif
        }
        float e[4][8];
#pragma unroll
        for (int k = 0; k < AB_EP_NOPS; ++k) {
#if AB_EP_PRE_OP >= 0
          if (k == AB_EP_PRE_OP) {
#if AB_EP_LAZY
            stage_group(j, e[k], lane);
#else
#pragma unroll
            for (int t = 0; t < 8; ++t) e[k][t] = op_l[j + t];
#endif
            continue;
          }
#endif
          if (is_row_op(k) || sc.vec[k]) {
#pragma unroll
            for (int t = 0; t < 8; ++t) e[k][t] = ev[k][t];
          } else if (sc.is[k]) {
#pragma unroll
            for (int t = 0; t < 8; ++t) e[k][t] = sc.v[k];
          } else if (p.ep_cs[k] == 1) {
            ld8<true>(p.ep_ptr[k] + r * p.ep_rs[k] + col, e[k],
                ((reinterpret_cast<uintptr_t>(p.ep_ptr[k]) & 31) == 0) && ((p.ep_rs[k] & 7) == 0));
          } else {
            const float* q = p.ep_ptr[k] + r * p.ep_rs[k] + col * p.ep_cs[k];
#pragma unroll
            for (int t = 0; t < 8; ++t) e[k][t] = q[t * p.ep_cs[k]];
          }
        }
        float o[AB_EP_NOUT][8];
#pragma unroll
        for (int t = 0; t < 8; ++t) { AB_EP_EVAL(v[t], e, t, o, sc.rcp, UDIV); }
#if AB_EP_STAGED
        put_outputs<kStageValue>(o, r, col);
        sts128(stage + 4u * st_off(lane, j >> 2), o[kStageValue][0], o[kStageValue][1], o[kStageValue][2], o[kStageValue][3]);
        sts128(stage + 4u * st_off(lane, (j >> 2) + 1), o[kStageValue][4], o[kStageValue][5], o[kStageValue][6], o[kStageValue][7]);
#else
        put_outputs<-1>(o, r, col);
#if AB_EP_COLSUM >= 0
#pragma unroll
        for (int t = 0; t < 8; ++t) x[j + t] = o[AB_EP_COLSUM][t];
#elif AB_EP_TPLANE >= 0
#pragma unroll
        for (int t = 0; t < 8; ++t) x[j + t] = o[AB_EP_TPLANE][t];
#endif
#endif
#if AB_EP_FULLSUM >= 0
#if AB_EP_EXACT_SUMS
        {
          // four independent pairs per group of 8 (the single running pair was a chain of 8
          // dependent TwoSums per group), folded into the thread's total once per group
          FF q4[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            q4[t].hi = o[AB_EP_FULLSUM][t];
            q4[t].lo = 0.0f;
            ff_add(q4[t], o[AB_EP_FULLSUM][t + 4]);
          }
          ff_add(q4[0], q4[1]);
          ff_add(q4[2], q4[3]);
          ff_add(q4[0], q4[2]);
          ff_add(fs, q4[0]);
        }
#else
        {
          // reduced-precision products (tf32 / bf16 operands): 8 values summed as a float32
          // tree, the groups as float pairs
          const float* w = o[AB_EP_FULLSUM];
          ff_add(fs, __fadd_rn(__fadd_rn(__fadd_rn(w[0], w[1]), __fadd_rn(w[2], w[3])),
                               __fadd_rn(__fadd_rn(w[4], w[5]), __fadd_rn(w[6], w[7]))));
        }
#endif
#endif
      } else {
#if AB_EP_STAGED
        sts128(stage + 4u * st_off(lane, j >> 2), 0.0f, 0.0f, 0.0f, 0.0f);
        sts128(stage + 4u * st_off(lane, (j >> 2) + 1), 0.0f, 0.0f, 0.0f, 0.0f);
#elif AB_EP_COLSUM >= 0 || AB_EP_TPLANE >= 0
#pragma unroll
        for (int t = 0; t < 8; ++t) x[j + t] = 0.0f;
#endif
      }
    }
  }
  // ---- AB_EP_STAGED: the value that is stored / reduced / transposed goes through 4 KB of
  // shared memory per warp (a 32 x 32 float32 chunk, 16-byte groups XOR-swizzled with the row:
  // the SWIZZLE_128B pattern, conflict-free for the row writes of fused_eval, for the row
  // reads of pass 1 and for the column reads of pass 2):
  //   pass 1  lanes 8 i .. 8 i + 7 read one row as 8 float4 and store it as ONE full 128-byte
  //           line (float32 output) / 64 contiguous bytes (bf16 plane).  Stored from the
  //           accumulator layout (lane = row) every STG touches 32 different lines, half a
  //           sector each: the epilogue warps of regions 1 and 2 then wait on the store queue
  //           (long-scoreboard stalls on the address registers of in-flight stores,
  //           profiles/r02_bench_step_ncu_v2.txt);
  //   pass 2  lane c reads column c (32 LDS, one per row): the transpose that took 48 shuffles
  //           and ~130 selects, and the column sum becomes 31 adds without any shuffle.
  // The buffer lives behind the operand ring, which gives up one of its 7 stages for it in the
  // bf16 / tf32 kernels (the hi/lo kernels have the room anyway).
  static constexpr int kStageValue = AB_EP_COLSUM >= 0 ? AB_EP_COLSUM : (AB_EP_TPLANE >= 0 ? AB_EP_TPLANE : 0);
  static __device__ __forceinline__ uint32_t st_off(int r, int g) { return (uint32_t)(r * 32 + ((g ^ (r & 7)) << 2)); }
#if AB_EP_STAGED
  template <bool EDGE = true>
  __device__ __forceinline__ void fused_reduce(float (&x)[32], long long row, long long col0, int lane) const {
    (void)x;
    __syncwarp();
    const long long row0 = row - lane;
    {
      float* dst = kStageValue == 0 ? p.C : p.out_ptr[kStageValue];
      const long long rs = kStageValue == 0 ? p.c_rs : p.out_rs[kStageValue];
      uint16_t* sp = static_cast<uint16_t*>(p.shadow[kStageValue]);
      if (dst != nullptr || sp != nullptr) {
        const int g = lane & 7;
        const long long col = col0 + 4 * g;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = 4 * i + (lane >> 3);
          const float4 v = lds128(stage + 4u * st_off(r, g));
          const long long grow = row0 + r;
          if (!EDGE || (grow < p.M && col < p.N)) {
            if (dst != nullptr) __stcs(reinterpret_cast<float4*>(dst + grow * rs + col), v);
            if (sp != nullptr) {
              uint32_t h0, h1;
              asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h0) : "f"(v.y), "f"(v.x));
              asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h1) : "f"(v.w), "f"(v.z));
              __stcs(reinterpret_cast<uint2*>(sp + grow * p.shadow_pitch[kStageValue] + col), make_uint2(h0, h1));
            }
          }
        }
      }
    }
#if AB_EP_COLSUM >= 0 || AB_EP_TPLANE >= 0
    {
#if AB_EP_TPLANE >= 0
      const bool want_t = p.shadow_t != nullptr;
#else
      const bool want_t = false;
#endif
      if (AB_EP_COLSUM >= 0 || want_t) {
        float v[32];
        const int cg = lane >> 2, cw = lane & 3;
#pragma unroll
        for (int r = 0; r < 32; ++r) v[r] = lds32(stage + 4u * (r * 32 + ((cg ^ (r & 7)) << 2) + cw));
        const long long c = col0 + lane;
#if AB_EP_COLSUM >= 0
        {
          // lane = column: its sum over the warp's 32 rows (rows / columns outside were staged
          // as zeros).  float pairs under the fp32-faithful policy, a float32 tree otherwise
          const long long rb = row >> 5;
#if AB_EP_EXACT_SUMS
          // a tree of float pairs (depth 5): one running pair would be a chain of 31 dependent
          // TwoSums per lane
          FF tp[16];
#pragma unroll
          for (int r = 0; r < 16; ++r) {
            tp[r].hi = v[2 * r];
            tp[r].lo = 0.0f;
            ff_add(tp[r], v[2 * r + 1]);
          }
#pragma unroll
          for (int w = 8; w >= 1; w >>= 1) {
#pragma unroll
            for (int r = 0; r < w; ++r) {
              tp[r] = tp[2 * r];
              ff_add(tp[r], tp[2 * r + 1]);
            }
          }
          const double tot = ff_double(tp[0]);
#else
          float t16[16];
#pragma unroll
          for (int r = 0; r < 16; ++r) t16[r] = __fadd_rn(v[2 * r], v[2 * r + 1]);
#pragma unroll
          for (int w = 8; w >= 1; w >>= 1) {
#pragma unroll
            for (int r = 0; r < w; ++r) t16[r] = __fadd_rn(t16[2 * r], t16[2 * r + 1]);
          }
          const double tot = (double)t16[0];
#endif
          if (!EDGE || (rb * 32 < p.M && c < p.N)) p.colsum_ws[rb * p.N + c] = tot;
        }
#endif
#if AB_EP_TPLANE >= 0
        if (want_t && (!EDGE || (c < p.N && row0 < p.M))) {
          uint16_t* dst = static_cast<uint16_t*>(p.shadow_t) + c * p.shadow_t_pitch + row0;
          if (!EDGE || row0 + 32 <= p.M) {
            uint32_t h[16];
#pragma unroll
            for (int t = 0; t < 16; ++t)
              asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h[t]) : "f"(v[2 * t + 1]), "f"(v[2 * t]));
#pragma unroll
            for (int t = 0; t < 4; ++t)
              __stcs(reinterpret_cast<uint4*>(dst) + t, make_uint4(h[4 * t], h[4 * t + 1], h[4 * t + 2], h[4 * t + 3]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (row0 + i < p.M) {
                uint16_t b;
                asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(b) : "f"(v[i]));
                dst[i] = b;
              }
          }
        }
#endif
      }
    }
#endif
    __syncwarp();  // the buffer is free for the next chunk's values
  }
#else
  template <bool EDGE = true>
  __device__ __forceinline__ void fused_reduce(float (&x)[32], long long row, long long col0, int lane) const {
    (void)x; (void)row; (void)col0; (void)lane;
#if AB_EP_TPLANE >= 0
    // Transposed bf16 plane, first half: rows are lanes, so two vertically adjacent values sit
    // in lanes l and l ^ 1.  Even lanes keep the even columns, odd lanes the odd ones: after
    // one exchange, P[i] of lane l is column 2 i + (l & 1) of the row pair (l & ~1, l | 1),
    // packed (low half = even row).  The remaining four exchanges (below, after the column
    // sums have consumed x[]) work on 16 packed registers instead of 32 floats.
    uint32_t P[16];
    const bool want_t = p.shadow_t != nullptr;
    if (want_t) {
      const bool odd = (lane & 1) != 0;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float mine = odd ? x[2 * i + 1] : x[2 * i];
        const float send = odd ? x[2 * i] : x[2 * i + 1];
        const float got = __shfl_xor_sync(0xffffffffu, send, 1);
        uint32_t h;  // low half <- second source operand
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(got), "f"(mine));
        P[i] = __byte_perm(h, 0u, odd ? 0x1032u : 0x3210u);
      }
    }
#endif
#if AB_EP_COLSUM >= 0
    {
      // 32 x 32 transpose-reduce over the warp's rows: after the step with distance h every
      // lane keeps the half of its columns selected by bit h of its lane index; lane l ends
      // with the sum of column col0 + l.  The reference's CAReduce accumulates float32 sums in
      // float64 (tensor/elemwise.py:1371-1385): under the fp32-faithful policy the 32 rows are
      // added as float pairs (see FF above); under the tf32 / bf16 policies -- the addends
      // carry 2^-11 / 2^-8 relative error themselves -- as a float32 tree.  Either way the
      // partial sum leaves the warp as float64.
      const long long rb = row >> 5;  // row - lane is a multiple of 32
#if AB_EP_EXACT_SUMS
      FF d[16];
      {
        const bool up = (lane & 16) != 0;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float keep = up ? x[16 + i] : x[i];
          const float send = up ? x[i] : x[16 + i];
          d[i].hi = keep;
          d[i].lo = 0.0f;
          ff_add(d[i], __shfl_xor_sync(0xffffffffu, send, 16));
        }
      }
#define AB_COLSUM_STEP(H)                                                      \
      {                                                                        \
        const bool up = (lane & (H)) != 0;                                     \
        _Pragma("unroll") for (int i = 0; i < (H); ++i) {                      \
          const FF keep = up ? d[(H) + i] : d[i];                              \
          const FF send = up ? d[i] : d[(H) + i];                              \
          FF got;                                                              \
          got.hi = __shfl_xor_sync(0xffffffffu, send.hi, (H));                 \
          got.lo = __shfl_xor_sync(0xffffffffu, send.lo, (H));                 \
          d[i] = keep;                                                         \
          ff_add(d[i], got);                                                   \
        }                                                                      \
      }
      AB_COLSUM_STEP(8) AB_COLSUM_STEP(4) AB_COLSUM_STEP(2) AB_COLSUM_STEP(1)
#undef AB_COLSUM_STEP
      if (rb * 32 < p.M && col0 + lane < p.N) p.colsum_ws[rb * p.N + col0 + lane] = ff_double(d[0]);
#else
#define AB_COLSUM_STEP(H)                                                      \
      {                                                                        \
        const bool up = (lane & (H)) != 0;                                     \
        _Pragma("unroll") for (int i = 0; i < (H); ++i) {                      \
          const float keep = up ? x[(H) + i] : x[i];                           \
          const float send = up ? x[i] : x[(H) + i];                           \
          x[i] = __fadd_rn(keep, __shfl_xor_sync(0xffffffffu, send, (H)));     \
        }                                                                      \
      }
      AB_COLSUM_STEP(16) AB_COLSUM_STEP(8) AB_COLSUM_STEP(4) AB_COLSUM_STEP(2) AB_COLSUM_STEP(1)
#undef AB_COLSUM_STEP
      if (rb * 32 < p.M && col0 + lane < p.N) p.colsum_ws[rb * p.N + col0 + lane] = (double)x[0];
#endif
    }
#endif
#if AB_EP_TPLANE >= 0
    if (want_t) {
      // second half: register index bit b <-> lane bit b + 1 (b = 0..3).  Before: lane bits
      // 1..4 = row pair k, register index i = column / 2.  After: lane l = column col0 + l,
      // P[k] = rows (row0 + 2 k, row0 + 2 k + 1): 64 contiguous bytes of the transposed plane.
#define AB_T_STEP(B)                                                            \
      {                                                                         \
        const bool up = (lane & (2 << (B))) != 0;                               \
        _Pragma("unroll") for (int i = 0; i < 16; ++i) {                        \
          if ((i & (1 << (B))) == 0) {                                          \
            const uint32_t send = up ? P[i] : P[i | (1 << (B))];                \
            const uint32_t got = __shfl_xor_sync(0xffffffffu, send, 2 << (B));  \
            if (up) P[i] = got; else P[i | (1 << (B))] = got;                   \
          }                                                                     \
        }                                                                       \
      }
      AB_T_STEP(0) AB_T_STEP(1) AB_T_STEP(2) AB_T_STEP(3)
#undef AB_T_STEP
      const long long row0 = row - lane;
      const long long c = col0 + lane;
      if (c < p.N && row0 < p.M) {
        uint16_t* dst = static_cast<uint16_t*>(p.shadow_t) + c * p.shadow_t_pitch + row0;
        if (row0 + 32 <= p.M) {
#pragma unroll
          for (int t = 0; t < 4; ++t)
            __stcs(reinterpret_cast<uint4*>(dst) + t, make_uint4(P[4 * t], P[4 * t + 1], P[4 * t + 2], P[4 * t + 3]));
        } else {
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (row0 + i < p.M) dst[i] = (uint16_t)((i & 1) ? (P[i >> 1] >> 16) : (P[i >> 1] & 0xffffu));
        }
      }
    }
#endif
  }
#endif  // AB_EP_STAGED
  __device__ __forceinline__ void finish_fullsum(const FF& acc, long long row, long long n0, int lane) const {
#if AB_EP_FULLSUM >= 0
    double fs = ff_double(acc);
#pragma unroll
    for (int h = 16; h >= 1; h >>= 1) fs += __shfl_xor_sync(0xffffffffu, fs, h);
    const long long rb = row >> 5;
    if (lane == 0 && rb * 32 < p.M) p.fullsum_ws[rb * p.fullsum_cols + n0 / (p.block_n >> 1)] = fs;
#endif
  }
  // accumulator already folded into registers (several K segments: the fp32-faithful mode)
  __device__ __forceinline__ void store_fused(float (&acc)[kAccRegs], long long row, long long n0,
                                              int nchunks, int lane, const FusedScalars& sc) const {
    const bool live = row < p.M;
    FF fs = {0.0f, 0.0f};
    // 128 accumulator registers are live here: the chunk's reads are issued and consumed in
    // place (this mode spends 3x the tensor time per tile; its epilogue is not the bottleneck)
#pragma unroll
    for (int c = 0; c < kAccRegs / 32; ++c) {
      if (c < nchunks) {
        ChunkPre pre;
        prefetch_chunk(pre, row, n0 + c * 32, live, sc, lane);
        float (&x)[32] = *reinterpret_cast<float(*)[32]>(&acc[c * 32]);
        fused_eval(x, row, n0 + c * 32, live, lane, sc, fs, pre);
        fused_reduce(x, row, n0 + c * 32, lane);
      }
    }
    finish_fullsum(fs, row, n0, lane);
  }
  // the whole K range sits in one TMEM accumulator (bf16 / tf32 policies): 32 columns at a
  // time straight from TMEM in a rolled loop -- 32 live accumulator registers instead of 128,
  // and the body exists once
  //
  // A tile whose rows (this warp's 32) and columns all lie inside [M, N] -- every tile of a
  // problem whose sizes are multiples of the tile -- runs the chunk loop without any row or
  // column test (EDGE = false); only the tiles on the bottom / right border take the checked
  // loop.  The two loops are separate bodies: a tile never runs instructions of both.
  template <bool EDGE, bool UDIV>
  __device__ __forceinline__ void chunk_loop(uint32_t t_acc, long long row, long long n0, int nchunks,
                                             int lane, const FusedScalars& sc, FF& fs) const {
    const bool live = !EDGE || row < p.M;
    ChunkPre pre;
    prefetch_chunk<EDGE>(pre, row, n0, live, sc, lane);
#pragma unroll 1
    for (int c = 0; c < nchunks; ++c) {
      uint32_t r[32];
      tmem_ld_32x32b_x32(t_acc + (uint32_t)(c * 32), r);
      float x[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(r[j]);
      const long long col0 = n0 + c * 32;
      fused_eval<EDGE, UDIV>(x, row, col0, live, lane, sc, fs, pre);
      if (c + 1 < nchunks) prefetch_chunk<EDGE>(pre, row, col0 + 32, live, sc, lane);
      fused_reduce<EDGE>(x, row, col0, lane);
    }
  }
  __device__ __forceinline__ void store_fused_tmem(uint32_t t_acc, long long row, long long n0, int nchunks,
                                                   int lane, const FusedScalars& sc) const {
    FF fs = {0.0f, 0.0f};
    const bool interior = row - lane + 32 <= p.M && n0 + 32 * nchunks <= p.N;  // warp-uniform
#if AB_EP_UDIV
    if (interior && sc.udiv)
      chunk_loop<false, true>(t_acc, row, n0, nchunks, lane, sc, fs);
    else
#endif
    if (interior)
      chunk_loop<false, false>(t_acc, row, n0, nchunks, lane, sc, fs);
    else
      chunk_loop<true, false>(t_acc, row, n0, nchunks, lane, sc, fs);
    finish_fullsum(fs, row, n0, lane);
  }
#endif  // AB_EPILOGUE
};

// work unit -> (tile, K range); consecutive units of a tile go to different CTAs
// Work unit -> (K range, tile).  Units are K-range major and, inside a K range, follow a grouped
// order (groups of p.group_m tile rows, columns outer, rows inner): the ~74 units in flight
// then form a compact block of the tile grid over ONE K range, so they share ~8 A panels and
// ~9 B panels in L2.  With rows-then-columns order the cfg3 weight-gradient products
// (4096 x 4096 x 65536) re-read their B operand for every tile row: 5.5-5.9 GB of DRAM reads
// per launch against 1 GB of operands (profiles/r02_bench_step_ncu.txt).
#define AB_UNIT_DECODE                                                          \
  const int split = (int)(unit / num_tiles);                                    \
  const long long tile_lin = unit - (long long)split * num_tiles;               \
  const long long tiles_m_ = num_tiles / tiles_n;                               \
  const long long gsz_ = (long long)p.group_m * tiles_n;                        \
  const long long first_m_ = (tile_lin / gsz_) * p.group_m;                     \
  const long long gm_ = min((long long)p.group_m, tiles_m_ - first_m_);         \
  const long long loc_ = tile_lin % gsz_;                                       \
  const long long tile_m = first_m_ + loc_ % gm_;                               \
  const long long tile_n = loc_ / gm_;                                          \
  const int kb_begin = split * p.kb_per_split;                                  \
  const int kb_end = min(kb_begin + p.kb_per_split, num_k_blocks);              \
  (void)split; (void)tile_m; (void)tile_n;

template <int KIND>
__device__ __forceinline__ void gemm_1cta_body(const CUtensorMap& map_a0, const CUtensorMap& map_a1,
                                               const CUtensorMap& map_b0, const CUtensorMap& map_b1,
                                               const GemmParams& p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // dynamic smem base is only guaranteed 16-byte aligned: round up to 1024 for SWIZZLE_128B
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  __shared__ __align__(8) uint64_t full_bar[8];
  __shared__ __align__(8) uint64_t empty_bar[8];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int stage_bytes = p.nparts * (p.a_tile_bytes + p.b_tile_bytes);
  const int num_k_blocks = (int)((p.K + p.k_elems_per_row - 1) / p.k_elems_per_row);
  // persistent tile scheduler: CTA b handles tiles b, b + gridDim.x, ...; N-tiles are
  // consecutive so the CTAs resident at one time share A row panels and all of B in L2
  const long long tiles_n = (p.N + p.block_n - 1) / p.block_n;
  const long long num_tiles = ((p.M + BLOCK_M - 1) / BLOCK_M) * tiles_n;
  const long long num_units = num_tiles * p.k_splits;
  const uint32_t tmem_cols = (uint32_t)(p.acc_stages * p.block_n);

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], kEpiThreads);  // every epilogue thread arrives
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    // allocate the accumulator columns (power of two >= 32): acc_stages x block_n
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&tmem_base_slot)),
                 "r"(tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_slot;

  if (warp < kEpiWarp0) {
  AB_SETMAXNREG_CONTROL();
  if (warp == 0) {
    // ================= TMA producer =================
    if (elect_one()) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_a0)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_b0)) : "memory");
      int stage = 0;
      uint32_t phase = 0;
      const OperandLoad la = operand_load_a(p), lb = operand_load_b(p);
      const int nparts = p.nparts, a_tile_bytes = p.a_tile_bytes, b_tile_bytes = p.b_tile_bytes;
      const int stages = p.stages, k_per_kb = p.k_elems_per_row, block_n = p.block_n;
      for (long long unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        AB_UNIT_DECODE
        const int m0 = (int)(tile_m * BLOCK_M);
        const int n0 = (int)(tile_n * block_n);
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sbase = smem + (size_t)stage * stage_bytes;
          mbar_expect_tx(&full_bar[stage], (uint32_t)stage_bytes);
          const int kc = kb * k_per_kb;
          load_tile(sbase, &map_a0, &full_bar[stage], kc, m0, la);
          load_tile(sbase + nparts * a_tile_bytes, &map_b0, &full_bar[stage], kc, n0, lb);
          if (nparts == 2) {
            load_tile(sbase + a_tile_bytes, &map_a1, &full_bar[stage], kc, m0, la);
            load_tile(sbase + 2 * a_tile_bytes + b_tile_bytes, &map_b1, &full_bar[stage], kc, n0, lb);
          }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t sit = 0;  // accumulator segments issued by this CTA
      // loop invariants in registers (see OperandLoad)
      const int nparts = p.nparts, stages = p.stages, seg_kblocks = p.seg_kblocks;
      const uint32_t acc_stages = (uint32_t)p.acc_stages, block_n = (uint32_t)p.block_n, idesc = p.idesc;
      const uint32_t a_tile_bytes = (uint32_t)p.a_tile_bytes, b_tile_bytes = (uint32_t)p.b_tile_bytes;
      const uint32_t a_kstep = (uint32_t)p.a_kstep, b_kstep = (uint32_t)p.b_kstep;
      const uint32_t a_lbo = p.a_mn ? (uint32_t)p.chunk_bytes : 16u;
      const uint32_t b_lbo = p.b_mn ? (uint32_t)p.chunk_bytes : 16u;
      for (long long unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        AB_UNIT_DECODE
        for (int kb0 = kb_begin; kb0 < kb_end; kb0 += seg_kblocks, ++sit) {
          const int kb1 = min(kb0 + seg_kblocks, kb_end);
          const uint32_t as = sit % acc_stages;
          const uint32_t aphase = (sit / acc_stages) & 1u;
          // wait until the epilogue has drained this accumulator stage
          mbar_wait(&tmem_empty_bar[as], aphase ^ 1);
          tcgen05_fence_after();
          const uint32_t d_tmem = tmem_base + as * block_n;
          for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tcgen05_fence_after();
            const uint32_t sbase = smem_u32(smem + (size_t)stage * stage_bytes);
            const uint32_t a_hi = sbase;
            const uint32_t a_lo = sbase + a_tile_bytes;
            const uint32_t b_hi = sbase + nparts * a_tile_bytes;
            const uint32_t b_lo = b_hi + b_tile_bytes;
#pragma unroll
            for (int k = 0; k < SW_BYTES / 32; ++k) {  // 32 bytes of K per instruction
              const uint32_t ka = k * a_kstep, kb_off = k * b_kstep;
              const uint32_t acc = (kb > kb0 || k > 0) ? 1u : 0u;
              if (nparts == 2) {
                // small cross terms first, the dominant hi*hi term last
                umma<KIND>(d_tmem, make_smem_desc(a_lo + ka, a_lbo), make_smem_desc(b_hi + kb_off, b_lbo), idesc, acc);
                umma<KIND>(d_tmem, make_smem_desc(a_hi + ka, a_lbo), make_smem_desc(b_lo + kb_off, b_lbo), idesc, 1u);
                umma<KIND>(d_tmem, make_smem_desc(a_hi + ka, a_lbo), make_smem_desc(b_hi + kb_off, b_lbo), idesc, 1u);
              } else {
                umma<KIND>(d_tmem, make_smem_desc(a_hi + ka, a_lbo), make_smem_desc(b_hi + kb_off, b_lbo), idesc, acc);
              }
            }
            tcgen05_commit(&empty_bar[stage]);  // frees this smem stage when the MMAs retire
            if (++stage == stages) { stage = 0; phase ^= 1; }
          }
          tcgen05_commit(&tmem_full_bar[as]);  // segment complete
        }
      }
    }
  }
  } else {
    AB_SETMAXNREG_EPILOGUE();
    // ================= epilogue (warps 2..9) =================
    // Two warps share each TMEM lane quarter; each owns half of the tile's columns and
    // keeps them as FP32 register accumulators across the K segments.
    const int q = warp & 3;              // TMEM lane quarter this warp may access
    const int half = (warp - kEpiWarp0) >> 2;    // which half of the columns
    const int half_n = p.block_n >> 1;
    const int nchunks = half_n >> 5;     // 32-column chunks: 1, 2 or 4
#if AB_EP_STAGED
    const EpilogueOut eo(p, smem_u32(smem + (size_t)p.stages * stage_bytes) +
                                (uint32_t)((warp - kEpiWarp0) * kStageBytesPerWarp));
#else
    const EpilogueOut eo(p);
#endif
#ifdef AB_EPILOGUE
    // the region's [1, 1] operands: read once per kernel (a global load per tile otherwise);
    // `lane` through a volatile asm: ptxas otherwise re-reads SR_TID (S2R, ~20 cycles on the
    // short scoreboard) at each of its many uses in the cross-lane code instead of keeping it
    const EpilogueOut::FusedScalars sc = eo.load_scalars();
    uint32_t lane_reg;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane_reg));
    const int lane = (int)lane_reg;
#endif
    float acc[kAccRegs];
    uint32_t sit = 0;
    for (long long unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
        AB_UNIT_DECODE
      const long long m0 = tile_m * BLOCK_M;
      const long long n0 = tile_n * p.block_n + half * half_n;
#ifdef AB_EPILOGUE
      if (KIND == 1 || kb_end - kb_begin <= p.seg_kblocks) {  // bf16 products are never segmented
        // one segment: the epilogue reads TMEM chunk by chunk, then frees the stage
        const uint32_t as = sit % (uint32_t)p.acc_stages;
        const uint32_t aphase = (sit / (uint32_t)p.acc_stages) & 1u;
        ++sit;
        mbar_wait(&tmem_full_bar[as], aphase);
        tcgen05_fence_after();
        const uint32_t t_acc = tmem_base + as * (uint32_t)p.block_n + (uint32_t)(half * half_n) +
                               ((uint32_t)(q * 32) << 16);
        eo.store_fused_tmem(t_acc, m0 + q * 32 + lane, n0, nchunks, lane, sc);
        tcgen05_fence_before();
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&tmem_empty_bar[as]))
                     : "memory");
        continue;
      }
#endif
      for (int kb0 = kb_begin; kb0 < kb_end; kb0 += p.seg_kblocks, ++sit) {
        const uint32_t as = sit % (uint32_t)p.acc_stages;
        const uint32_t aphase = (sit / (uint32_t)p.acc_stages) & 1u;
        mbar_wait(&tmem_full_bar[as], aphase);
        tcgen05_fence_after();
        const uint32_t t_acc = tmem_base + as * (uint32_t)p.block_n + (uint32_t)(half * half_n) +
                               ((uint32_t)(q * 32) << 16);
        fold_segment(acc, t_acc, nchunks, kb0 == kb_begin);
        // the segment is in registers: hand the accumulator stage back to the MMA warp
        tcgen05_fence_before();
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&tmem_empty_bar[as]))
                     : "memory");
      }
#ifdef AB_EPILOGUE
      eo.store_fused(acc, m0 + q * 32 + lane, n0, nchunks, lane, sc);  // fused launches are never split along K
#else
      if (split == 0) eo.store(acc, m0 + q * 32 + lane, n0, nchunks);
      else eo.store_partial(acc, m0 + q * 32 + lane, n0, nchunks, split);
#endif
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(tmem_cols)
                 : "memory");
  }
}

// ------------------------------------------------------------------ 2-CTA variant
// cta_group::2: a cluster of two CTAs (same TPC) computes one 256 x 256 tile.  Each
// CTA stages its own 128 rows of A and HALF of the B tile (128 of the 256 N rows), the
// leader CTA issues tcgen05.mma.cta_group::2 (M = 256) that reads both CTAs' shared
// memory, and each CTA's TMEM receives its 128 accumulator rows.  Per CTA and k-block
// that is 32 KB from L2 instead of 48 KB: the 1-CTA kernel is L2->SM bandwidth bound
// (profiles/r01_gemm_bf16_v2_persistent.txt: lts2xbar 13.7 TB/s, tensor pipe 72 %).
//   * full barriers live in the leader; both CTAs' TMA loads complete_tx on them
//     (cp.async.bulk.tensor...cta_group::2 with the peer bit of the barrier address
//     cleared), the leader arms expect_tx for the bytes of both;
//   * tcgen05.commit.cta_group::2 ... multicast::cluster arrives on the empty /
//     tmem_full barriers of both CTAs;
//   * all 256 epilogue threads arrive on the leader's tmem_empty barrier.
__device__ __forceinline__ void load_tile_2sm(uint8_t* dst, const CUtensorMap* map, uint64_t* bar,
                                              int kc, int mn0, const OperandLoad& o) {
  if (!o.mn_major) {
    tma_load_2d_2sm_hint(dst, map, bar, kc, mn0, o.policy);
  } else if (o.mn3d) {
    tma_load_3d_2sm(dst, map, bar, 0, kc, mn0 / o.mn_per_chunk);
  } else {
    for (int c = 0; c < o.chunks; ++c)
      tma_load_2d_2sm_hint(dst + c * o.chunk_bytes, map, bar, mn0 + c * o.mn_per_chunk, kc, o.policy);
  }
}
// GemmParams here: block_n = 256 (the pair's N tile), b_tile_bytes = 128 rows * 128 B
// (this CTA's half), b_chunks = chunks of the half, idesc encodes M = 256, N = 256.
//
// PAIRS == 2: a cluster of FOUR CTAs = two such pairs stacked along M (a 512 x 256 cluster
// tile) that share the B tile.  The 256 x 256 pair tile asks for 64 B/clk/SM from L2 at full
// tensor rate while the chip delivers ~42 (6300 B/clk over 148 SMs): the mainloop of the
// 2-CTA kernel is L2->SM bound (tensor pipe 72 % active, profiles/r01_gemm_bf16_v4*).  With
// two pairs per cluster each CTA fetches its own 128 A rows and only a QUARTER of the B tile
// (64 of the 256 N rows), which cp.async.bulk.tensor ... .multicast::cluster delivers to the
// CTA of the same position in both pairs: 24 KB instead of 32 KB per CTA and k-block.
//   * a CTA's shared-memory stage is now written by its own producer and by its twin in the
//     other pair, so a stage is free only when BOTH pairs' MMAs have retired it: every
//     leader's tcgen05.commit multicasts to the empty barriers of all four CTAs
//     (count = PAIRS);
//   * tmem_full / tmem_empty stay inside a pair.
template <int PAIRS>
__device__ __forceinline__ void load_b_2sm(uint8_t* dst, const CUtensorMap* map, uint64_t* bar, int kc,
                                           int n0, uint32_t pair, uint16_t mask, const OperandLoad& o,
                                           int b_tile_bytes, int block_n) {
  if (PAIRS == 1) {
    load_tile_2sm(dst, map, bar, kc, n0, o);
  } else if (!o.mn_major) {
    // K-major: box {128 B of K, block_n / 4 rows}; this CTA's quarter lands behind the twin's
    tma_load_2d_2sm_mc(dst + pair * (b_tile_bytes / 2), map, bar, kc, n0 + (int)pair * (block_n / 4), mask);
  } else {
    const int cpq = o.chunks / 2;  // chunks per quarter
    for (int c = (int)pair * cpq; c < ((int)pair + 1) * cpq; ++c)
      tma_load_2d_2sm_mc(dst + c * o.chunk_bytes, map, bar, n0 + c * o.mn_per_chunk, kc, mask);
  }
}

template <int KIND, int PAIRS = 1>
__device__ __forceinline__ void gemm_2cta_body(const CUtensorMap& map_a0, const CUtensorMap& map_a1,
                                               const CUtensorMap& map_b0, const CUtensorMap& map_b1,
                                               const GemmParams& p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  __shared__ __align__(8) uint64_t full_bar[8];
  __shared__ __align__(8) uint64_t empty_bar[8];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();
  const uint32_t rank = crank & 1u;   // position inside the CTA pair
  const uint32_t pair = crank >> 1;   // which pair of the cluster
  const bool leader = rank == 0;
  const int stage_bytes = p.nparts * (p.a_tile_bytes + p.b_tile_bytes);
  const int num_k_blocks = (int)((p.K + p.k_elems_per_row - 1) / p.k_elems_per_row);
  constexpr int TILE_M = 2 * BLOCK_M;        // rows of one pair
  constexpr int CLUSTER_M = PAIRS * TILE_M;  // rows of the cluster tile
  const long long tiles_n = (p.N + p.block_n - 1) / p.block_n;
  const long long num_tiles = ((p.M + CLUSTER_M - 1) / CLUSTER_M) * tiles_n;
  const long long num_units = num_tiles * p.k_splits;
  const long long cluster_id = blockIdx.x / (2 * PAIRS), n_clusters = gridDim.x / (2 * PAIRS);
  const uint32_t tmem_cols = (uint32_t)(p.acc_stages * p.block_n);
  const uint16_t pair_mask = (uint16_t)(3u << (2 * pair));
  const uint16_t all_mask = (uint16_t)((1u << (2 * PAIRS)) - 1u);
  const uint16_t twin_mask = (uint16_t)((1u << rank) | (1u << (rank + 2)));  // same position, both pairs

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], PAIRS);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], 2 * kEpiThreads);  // the epilogue threads of both CTAs
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&tmem_base_slot)),
                 "r"(tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();  // barriers of both CTAs are initialised before any remote signal
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_slot;

  if (warp < kEpiWarp0) {
  AB_SETMAXNREG_CONTROL();
  if (warp == 0) {
    // ================= TMA producer (one per CTA) =================
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      const OperandLoad la = operand_load_a(p), lb = operand_load_b(p);
      const int nparts = p.nparts, a_tile_bytes = p.a_tile_bytes, b_tile_bytes = p.b_tile_bytes;
      const int stages = p.stages, k_per_kb = p.k_elems_per_row, block_n = p.block_n;
      for (long long unit = cluster_id; unit < num_units; unit += n_clusters) {
        AB_UNIT_DECODE
        const int m0 = (int)(tile_m * CLUSTER_M) + (int)pair * TILE_M + (int)rank * BLOCK_M;
        const int n0 = (int)(tile_n * block_n) + (int)rank * (block_n / 2);
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sbase = smem + (size_t)stage * stage_bytes;
          if (leader) mbar_expect_tx(&full_bar[stage], (uint32_t)(2 * stage_bytes));
          const int kc = kb * k_per_kb;
          load_tile_2sm(sbase, &map_a0, &full_bar[stage], kc, m0, la);
          load_b_2sm<PAIRS>(sbase + nparts * a_tile_bytes, &map_b0, &full_bar[stage], kc, n0, pair,
                            twin_mask, lb, b_tile_bytes, block_n);
          if (nparts == 2) {
            load_tile_2sm(sbase + a_tile_bytes, &map_a1, &full_bar[stage], kc, m0, la);
            load_b_2sm<PAIRS>(sbase + 2 * a_tile_bytes + b_tile_bytes, &map_b1, &full_bar[stage], kc,
                              n0, pair, twin_mask, lb, b_tile_bytes, block_n);
          }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (leader CTA only) =================
    if (leader && elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t sit = 0;
      // loop invariants in registers (see OperandLoad)
      const int nparts = p.nparts, stages = p.stages, seg_kblocks = p.seg_kblocks;
      const uint32_t acc_stages = (uint32_t)p.acc_stages, block_n = (uint32_t)p.block_n, idesc = p.idesc;
      const uint32_t a_tile_bytes = (uint32_t)p.a_tile_bytes, b_tile_bytes = (uint32_t)p.b_tile_bytes;
      const uint32_t a_kstep = (uint32_t)p.a_kstep, b_kstep = (uint32_t)p.b_kstep;
      const uint32_t a_lbo = p.a_mn ? (uint32_t)p.chunk_bytes : 16u;
      const uint32_t b_lbo = p.b_mn ? (uint32_t)p.chunk_bytes : 16u;
      for (long long unit = cluster_id; unit < num_units; unit += n_clusters) {
        AB_UNIT_DECODE
        for (int kb0 = kb_begin; kb0 < kb_end; kb0 += seg_kblocks, ++sit) {
          const int kb1 = min(kb0 + seg_kblocks, kb_end);
          const uint32_t as = sit % acc_stages;
          const uint32_t aphase = (sit / acc_stages) & 1u;
          mbar_wait(&tmem_empty_bar[as], aphase ^ 1);
          tcgen05_fence_after();
          const uint32_t d_tmem = tmem_base + as * block_n;
          for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tcgen05_fence_after();
            const uint32_t sbase = smem_u32(smem + (size_t)stage * stage_bytes);
            const uint32_t a_hi = sbase;
            const uint32_t a_lo = sbase + a_tile_bytes;
            const uint32_t b_hi = sbase + nparts * a_tile_bytes;
            const uint32_t b_lo = b_hi + b_tile_bytes;
#pragma unroll
            for (int k = 0; k < SW_BYTES / 32; ++k) {
              const uint32_t ka = k * a_kstep, kbo = k * b_kstep;
              const uint32_t acc = (kb > kb0 || k > 0) ? 1u : 0u;
              if (nparts == 2) {
                umma_2sm<KIND>(d_tmem, make_smem_desc(a_lo + ka, a_lbo), make_smem_desc(b_hi + kbo, b_lbo), idesc, acc);
                umma_2sm<KIND>(d_tmem, make_smem_desc(a_hi + ka, a_lbo), make_smem_desc(b_lo + kbo, b_lbo), idesc, 1u);
                umma_2sm<KIND>(d_tmem, make_smem_desc(a_hi + ka, a_lbo), make_smem_desc(b_hi + kbo, b_lbo), idesc, 1u);
              } else {
                umma_2sm<KIND>(d_tmem, make_smem_desc(a_hi + ka, a_lbo), make_smem_desc(b_hi + kbo, b_lbo), idesc, acc);
              }
            }
            tcgen05_commit_2sm_mask(&empty_bar[stage], all_mask);  // frees the stage in every CTA it is written by
            if (++stage == stages) { stage = 0; phase ^= 1; }
          }
          tcgen05_commit_2sm_mask(&tmem_full_bar[as], pair_mask);  // both CTAs' epilogues may fold the segment
        }
      }
    }
  }
  } else {
    AB_SETMAXNREG_EPILOGUE();
    // ================= epilogue (warps 2..9 of both CTAs) =================
    const int q = warp & 3;
    const int half = (warp - kEpiWarp0) >> 2;
    const int half_n = p.block_n >> 1;
    const int nchunks = half_n >> 5;
#if AB_EP_STAGED
    const EpilogueOut eo(p, smem_u32(smem + (size_t)p.stages * stage_bytes) +
                                (uint32_t)((warp - kEpiWarp0) * kStageBytesPerWarp));
#else
    const EpilogueOut eo(p);
#endif
#ifdef AB_EPILOGUE
    // the region's [1, 1] operands: read once per kernel (a global load per tile otherwise);
    // `lane` through a volatile asm: ptxas otherwise re-reads SR_TID (S2R, ~20 cycles on the
    // short scoreboard) at each of its many uses in the cross-lane code instead of keeping it
    const EpilogueOut::FusedScalars sc = eo.load_scalars();
    uint32_t lane_reg;
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane_reg));
    const int lane = (int)lane_reg;
#endif
    float acc[kAccRegs];
    uint32_t sit = 0;
    for (long long unit = cluster_id; unit < num_units; unit += n_clusters) {
        AB_UNIT_DECODE
      const long long m0 = tile_m * CLUSTER_M + (long long)pair * TILE_M + (long long)rank * BLOCK_M;
      const long long n0 = tile_n * p.block_n + half * half_n;
#ifdef AB_EPILOGUE
      if (KIND == 1 || kb_end - kb_begin <= p.seg_kblocks) {  // bf16 products are never segmented
        const uint32_t as = sit % (uint32_t)p.acc_stages;
        const uint32_t aphase = (sit / (uint32_t)p.acc_stages) & 1u;
        ++sit;
        mbar_wait(&tmem_full_bar[as], aphase);
        tcgen05_fence_after();
        const uint32_t t_acc = tmem_base + as * (uint32_t)p.block_n + (uint32_t)(half * half_n) +
                               ((uint32_t)(q * 32) << 16);
        eo.store_fused_tmem(t_acc, m0 + q * 32 + lane, n0, nchunks, lane, sc);
        tcgen05_fence_before();
        asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(
                         smem_u32(&tmem_empty_bar[as]) & kPeerBitMask)
                     : "memory");
        continue;
      }
#endif
      for (int kb0 = kb_begin; kb0 < kb_end; kb0 += p.seg_kblocks, ++sit) {
        const uint32_t as = sit % (uint32_t)p.acc_stages;
        const uint32_t aphase = (sit / (uint32_t)p.acc_stages) & 1u;
        mbar_wait(&tmem_full_bar[as], aphase);
        tcgen05_fence_after();
        const uint32_t t_acc = tmem_base + as * (uint32_t)p.block_n + (uint32_t)(half * half_n) +
                               ((uint32_t)(q * 32) << 16);
        fold_segment(acc, t_acc, nchunks, kb0 == kb_begin);
        tcgen05_fence_before();
        asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(
                         smem_u32(&tmem_empty_bar[as]) & kPeerBitMask)
                     : "memory");
      }
#ifdef AB_EPILOGUE
      eo.store_fused(acc, m0 + q * 32 + lane, n0, nchunks, lane, sc);  // fused launches are never split along K
#else
      if (split == 0) eo.store(acc, m0 + q * 32 + lane, n0, nchunks);
      else eo.store_partial(acc, m0 + q * 32 + lane, n0, nchunks, split);
#endif
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();  // nobody signals the peer's barriers / reads its smem after this
  if (warp == 1) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"(tmem_cols)
                 : "memory");
  }
}


#if AB_EP_STAGED
extern "C" __global__ void ab_gemm_ep_staged_marker() {}  // tells gemm_run to reserve kStageBytes
#endif
#ifdef AB_EPILOGUE
// NVRTC build: C-linkage entry points (the module is loaded by name from gemm_run)
extern "C" __global__ void __launch_bounds__(kGemmThreads, 1)
ab_gemm_ep_1cta_tf32(const __grid_constant__ CUtensorMap a0, const __grid_constant__ CUtensorMap a1,
                     const __grid_constant__ CUtensorMap b0, const __grid_constant__ CUtensorMap b1,
                     const __grid_constant__ GemmParams p) { gemm_1cta_body<0>(a0, a1, b0, b1, p); }
extern "C" __global__ void __launch_bounds__(kGemmThreads, 1)
ab_gemm_ep_1cta_f16(const __grid_constant__ CUtensorMap a0, const __grid_constant__ CUtensorMap a1,
                    const __grid_constant__ CUtensorMap b0, const __grid_constant__ CUtensorMap b1,
                    const __grid_constant__ GemmParams p) { gemm_1cta_body<1>(a0, a1, b0, b1, p); }
extern "C" __global__ void __launch_bounds__(kGemmThreads, 1)
ab_gemm_ep_2cta_tf32(const __grid_constant__ CUtensorMap a0, const __grid_constant__ CUtensorMap a1,
                     const __grid_constant__ CUtensorMap b0, const __grid_constant__ CUtensorMap b1,
                     const __grid_constant__ GemmParams p) { gemm_2cta_body<0>(a0, a1, b0, b1, p); }
extern "C" __global__ void __launch_bounds__(kGemmThreads, 1)
ab_gemm_ep_2cta_f16(const __grid_constant__ CUtensorMap a0, const __grid_constant__ CUtensorMap a1,
                    const __grid_constant__ CUtensorMap b0, const __grid_constant__ CUtensorMap b1,
                    const __grid_constant__ GemmParams p) { gemm_2cta_body<1>(a0, a1, b0, b1, p); }
extern "C" __global__ void __launch_bounds__(kGemmThreads, 1)
ab_gemm_ep_4cta_tf32(const __grid_constant__ CUtensorMap a0, const __grid_constant__ CUtensorMap a1,
                     const __grid_constant__ CUtensorMap b0, const __grid_constant__ CUtensorMap b1,
                     const __grid_constant__ GemmParams p) { gemm_2cta_body<0, 2>(a0, a1, b0, b1, p); }
extern "C" __global__ void __launch_bounds__(kGemmThreads, 1)
ab_gemm_ep_4cta_f16(const __grid_constant__ CUtensorMap a0, const __grid_constant__ CUtensorMap a1,
                    const __grid_constant__ CUtensorMap b0, const __grid_constant__ CUtensorMap b1,
                    const __grid_constant__ GemmParams p) { gemm_2cta_body<1, 2>(a0, a1, b0, b1, p); }
#endif
