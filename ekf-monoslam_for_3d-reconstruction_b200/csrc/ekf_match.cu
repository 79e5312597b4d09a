// csrc/ekf_match.cu — K3: active-search NCC matcher (Patch::findMatch, Patch.cpp:215-291, and
// computeCorrelation, Patch.cpp:293-329).  SURVEY.md §8(a) rows a11-a13.
//
// One CTA per feature.  The reference scores every in-ellipse candidate with a sequential
// double-precision two-pass NCC, rounds the score to float and keeps the first strict maximum.
// Reproducing that bit for bit does not require running its 5 x w^2 DP operations for every
// candidate: pixels are 8-bit integers, so
//     ncc* = (n Stp - T P) / sqrt((n Stt - T^2)(n Spp - P^2))          (n = w^2)
// is available EXACTLY from integer sums, and the reference's floating-point value differs from it
// by < 1e-13 (121 roundings of 1e-16 relative).  Rounding to float is monotonic, so only candidates
// whose ncc* lies within two float ulps (+ that error bound) of the largest ncc* can be, or tie
// with, the reference's float maximum.  Hence:
//   staging   : the u8 search window (<= 72 x 72) is pulled into shared memory by ONE TMA tile load
//               (cp.async.bulk.tensor over a tensor map of the frame stack, completion on an mbarrier, out-of-frame
//               bytes zero-filled by the copy engine) while the CTA packs the template; the box starts at the 16-byte
//               boundary left of the window (a requirement of the copy engine) and is re-aligned shared -> shared.
//               Frames whose base / row stride are not 16-byte aligned cannot be described by a tensor map and are
//               staged with ordinary loads.
//   fast pass : the window and the template packed 4 bytes per word live in shared
//               memory; each thread scores 4 horizontally adjacent candidates at a time with DP4A
//               (u8 x u8 dot products) on funnel-shifted window words -> Stp, P, Spp; ncc* in double.
//   exact pass: the handful of candidates inside the guard band (normally one) are re-scored with the
//               reference's own operation sequence (__dadd_rn/__dmul_rn, row-major, never contracted)
//               and compared as floats with the reference's first-wins tie-break.
// The result (match coordinates, accept / reject, float score) is bit-identical to the reference's;
// if the guard band ever overflows its list (pathological ties) every candidate takes the exact pass.
//
// That is the CTA matcher (match_one): any template side up to 31.  For template side 11 the TILE matcher of ekf_match_tile.cuh
// runs first — one warp per feature in the batch kernels (match_one_warp2), one CTA per feature ahead of match_one in
// k_match_filter (match_one_tile_cta): candidates scored in registers in 4 x 4 (4 x 2) tiles, ranked by an exact-integer float
// score, and only the few candidates that can lie in the guard band see double precision and the exact pass.  Near-ties it
// cannot decide fall back to match_one (deferred list / marked features / the same CTA).  Same result bits.
#include <cstdlib>

#include <cuda.h>   // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint)

#include "ekf_kernels.h"
#include "ekf_math.cuh"
#include "ekf_match_tile.cuh"

#define MATCH_THREADS 256
#define MATCH_MAX_W 31   // largest template side
#define MATCH_LIST 128   // guard-band list capacity

struct MatchResult {
  float best;  // max NCC (-1 if no candidate)
  int bi, bj;  // argmax (valid if best > -1)
};

// shared-memory plan for template side w and search clamp cl (pixels)
struct MatchSmem {
  int side;      // max window side = 2 cl + w
  int wsb;       // window row stride in bytes (multiple of 4, >= side + 8)
  int tw;        // template words per row
  int ncmax;     // max candidates = (2 cl + 1)^2
  int rawb;      // row stride of the raw TMA box: wsb + 16 (the box starts at the 16-byte boundary left of the window)
  size_t off_tpk, off_tb, off_win, off_raw, off_h1, off_h2, off_b1, off_b2, off_score, off_list, off_red, off_da, off_bar, total;
};
__host__ __device__ inline MatchSmem match_smem_plan(int w, int cl) {
  MatchSmem p;
  p.side = 2 * cl + w;
  p.wsb = (p.side + 8 + 3) & ~3;
  p.rawb = ((p.wsb + 15) & ~15) + 16;
  p.tw = (w + 3) >> 2;
  p.ncmax = (2 * cl + 1) * (2 * cl + 1);
  size_t o = 0;
  p.off_tpk = o; o += (size_t)w * p.tw * 4;                                   // packed template
  p.off_tb = o; o += (size_t)((w * w + 15) & ~15);                            // template bytes
  o = (o + 15) & ~(size_t)15;
  p.off_win = o; o += (size_t)(p.side + 1) * p.wsb;                           // u8 window (+1 spare row)
  // One region, three tenants with disjoint lifetimes (a block barrier between each hand-over): the raw TMA box (until the
  // window is re-aligned), the horizontal box sums (until the vertical pass is done), the ncc* scores (fast pass onwards).
  // Overlaying them takes the CTA from 48 to 32 KB at w = 11, clamp 20: 7 instead of 4 resident CTAs per SM.
  o = (o + 127) & ~(size_t)127;                                               // TMA destination: 128-byte aligned
  const size_t nh = (size_t)p.side * (2 * cl + 1);                            // horizontal sums: window rows x candidate columns
  const size_t raw_bytes = (size_t)p.side * p.rawb;                           // raw TMA box: side rows x rawb bytes
  const size_t h1_bytes = (nh * 2 + 15) & ~(size_t)15, h2_bytes = nh * 4;     // u16 sum of w pixels, u32 sum of w squares
  const size_t score_bytes = (size_t)p.ncmax * 8;                             // ncc* per candidate
  size_t ubytes = raw_bytes > h1_bytes + h2_bytes ? raw_bytes : h1_bytes + h2_bytes;
  if (score_bytes > ubytes) ubytes = score_bytes;
  p.off_raw = o; p.off_h1 = o; p.off_h2 = o + h1_bytes; p.off_score = o;
  o += (ubytes + 15) & ~(size_t)15;
  p.off_b1 = o; o += (size_t)p.ncmax * 4;                                     // P  = sum p   over w x w, per candidate
  p.off_b2 = o; o += (size_t)p.ncmax * 4;                                     // PP = sum p^2 over w x w, per candidate
  o = (o + 7) & ~(size_t)7;
  p.off_list = o; o += (size_t)MATCH_LIST * 4;                                // guard-band candidate keys
  o = (o + 7) & ~(size_t)7;
  p.off_red = o; o += 16 * sizeof(double) + 16 * sizeof(float) + 16 * sizeof(int);
  o = (o + 7) & ~(size_t)7;
  p.off_da = o; o += (size_t)w * w * sizeof(double);                          // (double)(float)t - m1 per template pixel (exact pass)
  p.off_bar = o; o += 8;                                                      // mbarrier of the TMA load
  p.total = o;
  return p;
}

// ---- TMA (cp.async.bulk.tensor) + mbarrier, raw PTX for sm_100a -------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int x, int y, int z, unsigned long long* bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n"
               ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  unsigned done = 0;
  while (!done) {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(done)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
  }
}

// The reference's computeCorrelation for one candidate (window ROI at byte offset `roi`) in its exact operation order.  The
// three accumulation chains of Patch.cpp:316-326 — n1 = sum da da, n2 = sum db db, corr = sum da db, each a sequential sum
// over the pixels in row-major order — are independent, so three lanes of a 4-lane group run one chain each on the SAME
// instruction stream (role 0: n1, 1: n2, 2: corr): a third of the fp64 instructions of one thread running all three, and
// the chain (one DADD of 8.7 cycles per pixel) stays the only serial dependency.  da = (double)(float)t - m1 comes from shared
// memory (formed once per feature with the same expression).  Every lane of the group returns the score.
__device__ __forceinline__ float match_exact_score4(const double* da, const uint8_t* win, int wsb, int roi, int w, int P, int role,
                                                    unsigned gmask, int gbase) {
  const double m2 = __ddiv_rn((double)P, (double)(w * w));
  double acc = 0;
  for (int r = 0; r < w; ++r) {
    const uint8_t* wr = win + roi + r * wsb;
    const double* dr = da + r * w;
#pragma unroll 11
    for (int x = 0; x < w; ++x) {
      const double a = dr[x];
      const double b = __dsub_rn((double)(float)wr[x], m2);
      const double fa = role == 1 ? b : a, fb = role == 0 ? a : b;
      acc = __dadd_rn(acc, __dmul_rn(fa, fb));
    }
  }
  const double n1 = __shfl_sync(gmask, acc, gbase), n2 = __shfl_sync(gmask, acc, gbase + 1), corr = __shfl_sync(gmask, acc, gbase + 2);
  return (float)__ddiv_rn(corr, __dsqrt_rn(__dmul_rn(n2, n1)));
}

// Stp of four horizontally adjacent candidates: u8 x u8 dot products (DP4A) of the packed template
// rows with funnel-shifted window words.  WC > 0 fixes the template side at compile time.
template <int WC>
__device__ __forceinline__ void match_dots4(const uint8_t* win0, int wsb, const unsigned* tpk, int w_rt, unsigned acc[4]) {
  const int w = WC > 0 ? WC : w_rt;
  const int tw = (w + 3) >> 2;
#pragma unroll
  for (int r = 0; r < w; ++r) {
    const unsigned* wr = reinterpret_cast<const unsigned*>(win0 + r * wsb);
    const unsigned* tr = tpk + r * tw;
    unsigned lo = wr[0];
#pragma unroll
    for (int k = 0; k < tw; ++k) {
      const unsigned hi = wr[k + 1];
      const unsigned t = tr[k];
      acc[0] = __dp4a(lo, t, acc[0]);
      acc[1] = __dp4a(__funnelshift_r(lo, hi, 8), t, acc[1]);
      acc[2] = __dp4a(__funnelshift_r(lo, hi, 16), t, acc[2]);
      acc[3] = __dp4a(__funnelshift_r(lo, hi, 24), t, acc[3]);
      lo = hi;
    }
  }
}

// Core search for one feature by one CTA.  All threads must call.
__device__ MatchResult match_one(const MatchJob& jb, int w, float sigma_size, float clampv, unsigned char* smem_raw,
                                 unsigned* phase_io = nullptr, bool init_bar = true) {
  const int tid = threadIdx.x;
  const int half = w / 2, w2 = w * w;
  const MatchSmem pl = match_smem_plan(w, (int)clampv);
  // --- scalar setup, replicated per thread (Patch.cpp:218-241) ---
  const MatchGeom G = match_geometry(jb, w, sigma_size, clampv, pl.side - w + 1);
  const int uc = G.uc, vc = G.vc, i0 = G.i0, j0 = G.j0, nv = G.nv, ilo = G.ilo, jlo = G.jlo, cw = G.cw, ch = G.ch;
  const float x_2_coeff = G.x_2_coeff, y_2_coeff = G.y_2_coeff, yx_coeff = G.yx_coeff, sigma_2 = G.sigma_2;
  const bool any = G.any;
  const int ww = any ? cw + w - 1 : 0, wh = any ? ch + w - 1 : 0;
  const int wsb = pl.wsb, tw = pl.tw;

  unsigned* tpk = reinterpret_cast<unsigned*>(smem_raw + pl.off_tpk);
  uint8_t* tb = smem_raw + pl.off_tb;
  uint8_t* win = smem_raw + pl.off_win;
  unsigned short* Hh1 = reinterpret_cast<unsigned short*>(smem_raw + pl.off_h1);
  unsigned* Hh2 = reinterpret_cast<unsigned*>(smem_raw + pl.off_h2);
  unsigned* H1 = reinterpret_cast<unsigned*>(smem_raw + pl.off_b1);
  unsigned* H2 = reinterpret_cast<unsigned*>(smem_raw + pl.off_b2);
  double* score = reinterpret_cast<double*>(smem_raw + pl.off_score);
  int* list = reinterpret_cast<int*>(smem_raw + pl.off_list);
  double* da = reinterpret_cast<double*>(smem_raw + pl.off_da);
  double* red_d = reinterpret_cast<double*>(smem_raw + pl.off_red);   // [0..7] warp maxima, [8] n1, [9] M*
  float* red_s = reinterpret_cast<float*>(red_d + 16);
  int* red_k = reinterpret_cast<int*>(red_s + 16);                     // [0..7] keys, [8] T, [9] TT, [10] list count

  // --- template: packed words (zero padded), integer sums T = sum t, TT = sum t^2 ---
  unsigned long long* bar = reinterpret_cast<unsigned long long*>(smem_raw + pl.off_bar);
  const bool use_tma = jb.tmap != nullptr;
  if (tid < 16) red_k[tid] = 0;
  if (use_tma && tid == 0 && init_bar) mbar_init(bar, 1);
  __syncthreads();
  uint8_t* raw = smem_raw + pl.off_raw;
  if (use_tma && any && tid == 0) {
    // ONE tile load per feature: the box is `side` rows of rawb bytes whose left edge is the 16-byte boundary at or left of
    // the window (the copy engine needs the innermost coordinate 16-byte aligned: tools/tma_probe2.cu); bytes outside the
    // frame arrive as zeros.  The box lands in `raw` while the CTA packs the template below.
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // the box region was last touched by ordinary accesses (scores of the previous feature)
    mbar_expect_tx(bar, (unsigned)(pl.rawb * pl.side));
    tma_load_3d(raw, jb.tmap, (ilo - half) & ~15, jlo - half, jb.frame_index, bar);
  }
  {
    int pt = 0, ptt = 0;
    for (int e = tid; e < w * tw; e += MATCH_THREADS) {
      const int r = e / tw, k4 = (e - r * tw) * 4;
      unsigned word = 0;
      for (int c = 0; c < 4; ++c)
        if (k4 + c < w) {
          const unsigned v = jb.tmpl[r * w + k4 + c];
          word |= v << (8 * c);
          pt += (int)v; ptt += (int)(v * v);
        }
      tpk[e] = word;
    }
    for (int e = tid; e < w2; e += MATCH_THREADS) tb[e] = jb.tmpl[e];
    for (int o = 16; o > 0; o >>= 1) { pt += __shfl_xor_sync(0xffffffffu, pt, o); ptt += __shfl_xor_sync(0xffffffffu, ptt, o); }
    if ((tid & 31) == 0 && (pt | ptt)) { atomicAdd(&red_k[8], pt); atomicAdd(&red_k[9], ptt); }
  }
  // --- ordinary-load staging (frames a tensor map cannot describe): bytes; columns past ww and the spare row are zero ---
  if (any && !use_tma) {
    const int x0 = ilo - half, y0 = jlo - half;
    if ((((size_t)jb.frame | (size_t)jb.fstride) & 3) == 0) {
      // aligned 4-byte loads, funnel-shifted to the window's own alignment (a quarter of the load instructions of the
      // byte loop, which took a fifth of the kernel); the word past the last needed byte is never touched
      const int sh = x0 & 3, xa = x0 - sh, nwords = wsb >> 2;
      for (int yy = tid / 32; yy <= wh; yy += MATCH_THREADS / 32) {
        const unsigned* srcw = reinterpret_cast<const unsigned*>(jb.frame + (size_t)(y0 + yy) * jb.fstride + xa);
        unsigned* dstw = reinterpret_cast<unsigned*>(win + yy * wsb);
        for (int k = tid & 31; k < nwords; k += 32) {
          unsigned v = 0;
          if (yy < wh && 4 * k < ww) {
            const int last = min(4 * k + 3, ww - 1);          // last window column this word needs
            const unsigned lo = srcw[k];
            const unsigned hi = (sh > 0 && last + sh >= 4 * k + 4) ? srcw[k + 1] : 0u;
            v = __funnelshift_r(lo, hi, 8 * sh);
            const int rem = ww - 4 * k;
            if (rem < 4) v &= (1u << (8 * rem)) - 1u;
          }
          dstw[k] = v;
        }
      }
    } else {
      for (int yy = tid / 32; yy <= wh; yy += MATCH_THREADS / 32) {
        const uint8_t* src = jb.frame + (size_t)(y0 + yy) * jb.fstride + x0;
        for (int xx = tid & 31; xx < wsb; xx += 32) win[yy * wsb + xx] = (yy < wh && xx < ww) ? src[xx] : (uint8_t)0;
      }
    }
  }
  if (use_tma && any) {
    mbar_wait(bar, phase_io ? *phase_io : 0u);   // every consumer thread observes the completion of the tile load
    if (phase_io) *phase_io ^= 1u;            // a persistent CTA re-uses the barrier: the next load completes the other phase
    // raw box -> window at its own alignment (funnel shift by the 0..15 bytes between the box edge and the window), with the
    // same zero padding as the ordinary-load path: columns past ww and rows from wh on are zero
    const int sh = (ilo - half) & 15, shw = sh >> 2, shb = 8 * (sh & 3), nwords = wsb >> 2;
    for (int yy = tid / 32; yy <= wh; yy += MATCH_THREADS / 32) {
      const unsigned* srcw = reinterpret_cast<const unsigned*>(raw + (size_t)min(yy, pl.side - 1) * pl.rawb) + shw;
      unsigned* dstw = reinterpret_cast<unsigned*>(win + yy * wsb);
      for (int k = tid & 31; k < nwords; k += 32) {
        unsigned v = 0;
        if (yy < wh && 4 * k < ww) {
          v = __funnelshift_r(srcw[k], srcw[k + 1], shb);
          const int rem = ww - 4 * k;
          if (rem < 4) v &= (1u << (8 * rem)) - 1u;
        }
        dstw[k] = v;
      }
    }
  }
  __syncthreads();
  const int T = red_k[8], TT = red_k[9];
  const double dn = (double)w2;
  const double m1 = __ddiv_rn((double)T, dn);
  for (int e = tid; e < w2; e += MATCH_THREADS) da[e] = __dsub_rn((double)(float)tb[e], m1);   // read after later barriers
  // --- w x w box sums of p and p^2 for every candidate (exact ints), separable with sliding sums:
  //     a thread produces 4 adjacent outputs from one w-term sum plus three add/subtract slides ---
  if (any) {
    const int gx = (cw + 3) >> 2;
    // linear item index (row, group) advanced without a division per item
    const int dq = MATCH_THREADS % gx, dy = MATCH_THREADS / gx;
    for (int yy = tid / gx, gq = tid - (tid / gx) * gx; yy < wh; ) {
      {
        const uint8_t* pr = win + yy * wsb + 4 * gq;
        unsigned r1 = 0, r2 = 0;
        for (int x = 0; x < w; ++x) { const unsigned v = pr[x]; r1 += v; r2 += v * v; }
        unsigned short* o1 = Hh1 + yy * cw + 4 * gq;
        unsigned* o2 = Hh2 + yy * cw + 4 * gq;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
          if (4 * gq + s < cw) { o1[s] = (unsigned short)r1; o2[s] = r2; }
          const unsigned vin = pr[w + s], vout = pr[s];     // bytes past ww are zero, inside the padded row
          r1 += vin - vout; r2 += vin * vin - vout * vout;
        }
      }
      gq += dq; yy += dy;
      if (gq >= gx) { gq -= gx; ++yy; }
    }
  }
  __syncthreads();
  if (any) {
    const int gv = (ch + 3) >> 2;
    const int di = MATCH_THREADS % cw, dg = MATCH_THREADS / cw;
    for (int gq = tid / cw, iu = tid - (tid / cw) * cw; gq < gv; ) {
      {
        const int jv0 = 4 * gq;
        unsigned r1 = 0, r2 = 0;
        for (int r = 0; r < w; ++r) { r1 += Hh1[(jv0 + r) * cw + iu]; r2 += Hh2[(jv0 + r) * cw + iu]; }
#pragma unroll
        for (int s = 0; s < 4; ++s) {
          if (jv0 + s >= ch) break;
          H1[(jv0 + s) * cw + iu] = r1; H2[(jv0 + s) * cw + iu] = r2;
          if (jv0 + s + 1 < ch) {
            r1 += (unsigned)Hh1[(jv0 + s + w) * cw + iu] - (unsigned)Hh1[(jv0 + s) * cw + iu];
            r2 += Hh2[(jv0 + s + w) * cw + iu] - Hh2[(jv0 + s) * cw + iu];
          }
        }
      }
      iu += di; gq += dg;
      if (iu >= cw) { iu -= cw; ++gq; }
    }
  }
  __syncthreads();
  const double d1 = dn * (double)TT - (double)T * (double)T;   // exact (< 2^53)

  // --- fast pass: ncc* of every in-ellipse candidate ---
  const double kNone = -1.0e300;
  double lmax = kNone;
  if (any) {
    const int gx = (cw + 3) >> 2;
    const double rd1 = (d1 > 0.0) ? rsqrt(d1) : 0.0;
    // group = 4 horizontally adjacent candidates; warps stride over candidate rows, lanes over groups
    const int dq = MATCH_THREADS % gx, dy = MATCH_THREADS / gx;
    for (int jv = tid / gx, gq = tid - (tid / gx) * gx; jv < ch; gq += dq, jv += dy, jv += (gq >= gx) ? 1 : 0, gq -= (gq >= gx) ? gx : 0) {
      const int ja = jlo + jv;
      const float dj = (float)(ja - vc);
      const float ey = __fmul_rn(__fmul_rn(y_2_coeff, dj), dj);
      {
        const int iu4 = gq * 4;
        // ellipse gate in float, same association as Patch.cpp:247
        bool valid[4];
        bool anyv = false;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
          const int iu = iu4 + s;
          const float fdi = (float)(ilo + iu - uc);
          const float e = __fadd_rn(__fadd_rn(__fmul_rn(__fmul_rn(x_2_coeff, fdi), fdi), ey), __fmul_rn(__fmul_rn(yx_coeff, fdi), dj));
          valid[s] = (iu < cw) && (e <= sigma_2);
          anyv |= valid[s];
        }
        if (!anyv) {
#pragma unroll
          for (int s = 0; s < 4; ++s)
            if (iu4 + s < cw) score[jv * cw + iu4 + s] = kNone;
          continue;
        }
        unsigned acc[4] = {0u, 0u, 0u, 0u};
        if (w == 11) match_dots4<11>(win + jv * wsb + iu4, wsb, tpk, w, acc);       // the benchmark / synthetic-scene template size
        else if (w == 21) match_dots4<21>(win + jv * wsb + iu4, wsb, tpk, w, acc);  // reference default (ConfigVSLAM.cpp:31)
        else match_dots4<0>(win + jv * wsb + iu4, wsb, tpk, w, acc);
#pragma unroll
        for (int s = 0; s < 4; ++s) {
          const int iu = iu4 + s;
          if (iu >= cw) continue;
          double v = kNone;
          if (valid[s]) {
            const unsigned P = H1[jv * cw + iu], PP = H2[jv * cw + iu];
            const double d2 = dn * (double)PP - (double)P * (double)P;   // exact (< 2^53)
            if (d1 > 0.0 && d2 > 0.0) {
              const double num = dn * (double)acc[s] - (double)T * (double)P;
              v = (num * rd1) * rsqrt(d2);
              if (v > lmax) lmax = v;
            }  // else: flat template or flat window, 0/0 in the reference, never selected
          }
          score[jv * cw + iu] = v;
        }
      }
    }
  }
  // --- block maximum of ncc* ---
  for (int o = 16; o > 0; o >>= 1) lmax = fmax(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
  if ((tid & 31) == 0) red_d[tid >> 5] = lmax;
  __syncthreads();
  if (tid == 0) {
    double m = red_d[0];
    for (int wv = 1; wv < MATCH_THREADS / 32; ++wv) m = fmax(m, red_d[wv]);
    red_d[9] = m;
  }
  __syncthreads();
  const double Mstar = red_d[9];
  float best = -1.0f;
  int bestkey = 0x7fffffff;
  if (any && Mstar > kNone) {
    // guard band: two float ulps at |M*| plus the bound on |reference - ncc*|
    const float fm = fabsf((float)Mstar);
    const double ulp = (double)(nextafterf(fm, 3.0e38f) - fm);
    const double thr = Mstar - (2.0 * ulp + 4.0e-12);   // ncc* itself carries ~4e-16 (two rsqrt), far inside the bound
    const int ncand = cw * ch;
    for (int c = tid; c < ncand; c += MATCH_THREADS) {
      if (score[c] >= thr) {
        const int slot = atomicAdd(&red_k[10], 1);
        if (slot < MATCH_LIST) list[slot] = c;
      }
    }
    __syncthreads();
    const int nlist = red_k[10];
    const bool overflow = nlist > MATCH_LIST;
    const int nwork = overflow ? ncand : nlist;
    // one 4-lane group per guard-band candidate (see match_exact_score4); whole warps iterate together
    const int lane = tid & 31, role = tid & 3, gbase = lane & ~3;
    const unsigned gmask = 0xfu << gbase;
    for (int q0 = (tid >> 5) * 8; q0 < nwork; q0 += (MATCH_THREADS / 32) * 8) {
      const int q = q0 + (lane >> 2);
      if (q >= nwork) continue;                          // uniform inside a 4-lane group
      const int c = overflow ? q : list[q];
      if (overflow && !(score[c] > kNone)) continue;
      const int jv = c / cw, iu = c - jv * cw;
      const int P = (int)H1[c];
      const float sc = match_exact_score4(da, win, wsb, jv * wsb + iu, w, P, role, gmask, gbase);
      const int key = (ilo + iu - i0) * nv + (jlo + jv - j0);  // position in the reference's scan order (u outer, v inner)
      if (role == 0 && (sc > best || (sc == best && key < bestkey))) { best = sc; bestkey = key; }
    }
  }
  // --- arg-max: higher score wins, ties go to the earlier key (strict '>' in a sequential scan) ---
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int ok = __shfl_xor_sync(0xffffffffu, bestkey, o);
    if (ob > best || (ob == best && ok < bestkey)) { best = ob; bestkey = ok; }
  }
  if ((tid & 31) == 0) { red_s[tid >> 5] = best; red_k[tid >> 5] = bestkey; }
  __syncthreads();
  best = red_s[0]; bestkey = red_k[0];
  for (int wv = 1; wv < MATCH_THREADS / 32; ++wv) {
    const float ob = red_s[wv];
    const int ok = red_k[wv];
    if (ob > best || (ob == best && ok < bestkey)) { best = ob; bestkey = ok; }
  }
  MatchResult res;
  res.best = best; res.bi = 0; res.bj = 0;
  if (bestkey != 0x7fffffff && nv > 0) {
    res.bi = i0 + bestkey / nv;
    res.bj = j0 + bestkey % nv;
  }
  return res;
}

static size_t match_smem_bytes(int w, float clampv) { return match_smem_plan(w, (int)clampv).total; }

// Tensor map of a stack of u8 frames (x = column, y = row, z = frame) whose box is the matcher's staging window for template
// side w and search clamp `clamp`.  The driver's encoder is looked up at run time (no link-time dependency on libcuda).
typedef CUresult (*EkfEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
void match_make_tensor_map(EkfTensorMap* out, const uint8_t* frames, int width, int height, int stride, int n_frames, int w, int clamp) {
  static_assert(sizeof(CUtensorMap) <= sizeof(out->opaque), "EkfTensorMap too small");
  out->ok = 0;
  static EkfEncodeTiled enc = nullptr;
  static bool looked = false;
  if (!looked) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
      enc = (EkfEncodeTiled)fn;
    else
      cudaGetLastError();
    looked = true;
  }
  const char* off = getenv("EKF_MATCH_TMA");
  if (!enc || (off && atoi(off) == 0)) return;
  if (!frames || (((size_t)frames | (size_t)stride) & 15) != 0 || width < 1 || height < 1 || n_frames < 1) return;
  const MatchSmem pl = match_smem_plan(w, clamp);
  if (pl.rawb > 256 || pl.side > 256) return;
  const cuuint64_t gdim[3] = {(cuuint64_t)width, (cuuint64_t)height, (cuuint64_t)n_frames};
  const cuuint64_t gstr[2] = {(cuuint64_t)stride, (cuuint64_t)stride * (cuuint64_t)height};
  const cuuint32_t box[3] = {(cuuint32_t)pl.rawb, (cuuint32_t)pl.side, 1u};
  const cuuint32_t est[3] = {1u, 1u, 1u};
  const CUresult r = enc(reinterpret_cast<CUtensorMap*>(out->opaque), CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void*)frames, gdim, gstr, box, est,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  out->ok = (r == CUDA_SUCCESS) ? 1 : 0;
}
static const CUtensorMap& as_cu(const EkfTensorMap& m) { return *reinterpret_cast<const CUtensorMap*>(m.opaque); }

template <int W, int R>
__device__ bool match_one_tile_cta(const MatchJob& jb, float sigma_size, float clampv, unsigned char* smem_raw, MatchResult& res);   // below

// Filter-attached matcher: the loop V:870-880 with one CTA per feature.
__device__ __forceinline__ void match_filter_feature(FeatTab ft, int f, FrameView fr, const DevCfg& cfg, unsigned char* smem_raw,
                                                     const CUtensorMap* tmap, unsigned* phase_io = nullptr, bool init_bar = true,
                                                     bool try_tile = false, int frame_index = 0) {
  const int w = cfg.window, w2 = w * w;
  MatchJob jb;
  jb.tmap = tmap; jb.frame_index = frame_index;
  jb.frame = fr.px; jb.fw = fr.w; jb.fh = fr.h; jb.fstride = fr.stride;
  jb.tmpl = ft.mpatch + (size_t)f * cfg.tstride;
  jb.hu = ft.h[2 * f]; jb.hv = ft.h[2 * f + 1];
  for (int c = 0; c < 4; ++c) jb.S[c] = ft.S2[4 * f + c];
  MatchResult r;
  // template side 11: the tile matcher first; near-ties (uniform verdict) fall through to match_one in the same CTA
  if (!(try_tile && w == 11 && match_one_tile_cta<11, 2>(jb, cfg.sigma_size_f, cfg.search_clamp, smem_raw, r))) {
    if (try_tile) __syncthreads();   // the tile matcher's shared memory is re-used from here on
    r = match_one(jb, w, cfg.sigma_size_f, cfg.search_clamp, smem_raw, phase_io, init_bar);
  }
  __syncthreads();
  const bool accept = !(r.best < cfg.ncc_threshold);  // Patch.cpp:278
  if (accept) {
    // matching_patch <- matched ROI (Patch.cpp:285)
    const int x0 = r.bi - w / 2, y0 = r.bj - w / 2;
    for (int e = threadIdx.x; e < w2; e += MATCH_THREADS)
      ft.mpatch[(size_t)f * cfg.tstride + e] = fr.px[(size_t)(y0 + e / w) * fr.stride + x0 + (e % w)];
  }
  if (threadIdx.x == 0) {
    ft.n_tot[f] += 1;  // Patch.cpp:218
    ft.last_ncc[f] = r.best;
    if (!accept) {
      ft.center[2 * f] = -1.0f; ft.center[2 * f + 1] = -1.0f;
      ft.innov[f] = 0; ft.li[f] = 0; ft.hi[f] = 0;
    } else {
      ft.center[2 * f] = (float)r.bi; ft.center[2 * f + 1] = (float)r.bj;
      ft.z[2 * f] = (double)(float)r.bi; ft.z[2 * f + 1] = (double)(float)r.bj;
    }
  }
}
__global__ void __launch_bounds__(MATCH_THREADS, 4) k_match_filter(FeatTab ft, int N, FrameView fr, DevCfg cfg,
                                                                const __grid_constant__ CUtensorMap tmap, int use_tma, int tile) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int f = blockIdx.x;
  if (f >= N || !ft.innov[f]) return;
  match_filter_feature(ft, f, fr, cfg, smem_raw, use_tma ? &tmap : nullptr, nullptr, true, tile != 0);
}
// ------------------------------------------------------------------------------------------------
// Warp-per-feature path for SMALL search windows (candidate grid <= 16 x 16, template side <= 15): the batched filters
// (BASELINE config 3) match 4096 x 30 features per step whose converged windows hold ~200 candidates — a 256-thread CTA per
// feature spends its time in block barriers and idle lanes (4.1 of the 7.5 ms step).  Here one WARP owns a feature: window
// and template in a private 1.7 KB slice of shared memory, every lane scores up to eight candidates (Stp, P, PP by DP4A on
// funnel-shifted window words — exact integers, the same ncc* and guard band as match_one), the guard-band candidates take
// the reference's exact operation sequence on 4-lane groups, and only __syncwarp separates the phases.  Same result bits
// as match_one by construction: the fast pass only SELECTS the candidates whose exact float score is compared.  A feature
// with a larger window (or a guard band of more than 16 candidates) is not touched: its index goes to a list that a
// persistent grid of CTAs works off with match_one.
// ------------------------------------------------------------------------------------------------
#define MW_GRID 16
#define MW_MAXW 15
#define MW_WARPS 8
#define MW_ROWS (MW_GRID + MW_MAXW - 1)   // 30 window rows
#define MW_WS 40                          // window row stride in bytes (30 columns + slack for whole-word reads)
#define MW_LIST 16
struct MatchWarpSmem {
  unsigned win[MW_ROWS * MW_WS / 4];
  unsigned tpk[MW_MAXW * 4];
  unsigned char tb[MW_MAXW * MW_MAXW + 15];
  int list[MW_LIST];
  int cnt;
};

// exact score of one candidate on a 4-lane group: match_exact_score4 with da formed on the fly from the template bytes
__device__ __forceinline__ float match_exact_score4_tb(const unsigned char* tb, double m1, const uint8_t* win, int wsb, int roi, int w,
                                                       int P, int role, unsigned gmask, int gbase) {
  const double m2 = __ddiv_rn((double)P, (double)(w * w));
  double acc = 0;
  for (int r = 0; r < w; ++r) {
    const uint8_t* wr = win + roi + r * wsb;
    const unsigned char* tr = tb + r * w;
    for (int x = 0; x < w; ++x) {
      const double a = __dsub_rn((double)(float)tr[x], m1);
      const double b = __dsub_rn((double)(float)wr[x], m2);
      const double fa = role == 1 ? b : a, fb = role == 0 ? a : b;
      acc = __dadd_rn(acc, __dmul_rn(fa, fb));
    }
  }
  const double n1 = __shfl_sync(gmask, acc, gbase), n2 = __shfl_sync(gmask, acc, gbase + 1), corr = __shfl_sync(gmask, acc, gbase + 2);
  return (float)__ddiv_rn(corr, __dsqrt_rn(__dmul_rn(n2, n1)));
}

// One warp, one feature.  Returns false (nothing written, nothing decided) when the feature does not fit this path.
__device__ bool match_one_warp(const MatchJob& jb, int w, float sigma_size, float clampv, MatchWarpSmem& sm, MatchResult& res) {
  const int lane = threadIdx.x & 31;
  const int half = w / 2, w2 = w * w, tw = (w + 3) >> 2;
  const MatchGeom G = match_geometry(jb, w, sigma_size, clampv, 2 * (int)clampv + 1);
  if (w > MW_MAXW || G.cw > MW_GRID || G.ch > MW_GRID) return false;
  res.best = -1.0f; res.bi = 0; res.bj = 0;
  if (!G.any) return true;
  const int cw = G.cw, ch = G.ch, ww = cw + w - 1, wh = ch + w - 1;
  uint8_t* win = reinterpret_cast<uint8_t*>(sm.win);
  // --- template: packed words (zero padded), bytes, T = sum t, TT = sum t^2 ---
  int T = 0, TT = 0;
  for (int e = lane; e < w * tw; e += 32) {
    const int r = e / tw, k4 = (e - r * tw) * 4;
    unsigned word = 0;
    for (int c = 0; c < 4; ++c)
      if (k4 + c < w) {
        const unsigned v = jb.tmpl[r * w + k4 + c];
        word |= v << (8 * c);
        T += (int)v; TT += (int)(v * v);
      }
    sm.tpk[e] = word;
  }
  for (int e = lane; e < w2; e += 32) sm.tb[e] = jb.tmpl[e];
  for (int o = 16; o > 0; o >>= 1) { T += __shfl_xor_sync(0xffffffffu, T, o); TT += __shfl_xor_sync(0xffffffffu, TT, o); }
  // --- window: bytes, columns past ww zero ---
  {
    const int x0 = G.ilo - half, y0 = G.jlo - half;
    const int nwords = MW_WS / 4;
    if ((((size_t)jb.frame | (size_t)jb.fstride) & 3) == 0) {
      const int sh = x0 & 3, xa = x0 - sh;
      for (int e = lane; e < wh * nwords; e += 32) {
        const int yy = e / nwords, k = e - yy * nwords;
        const unsigned* srcw = reinterpret_cast<const unsigned*>(jb.frame + (size_t)(y0 + yy) * jb.fstride + xa);
        unsigned v = 0;
        if (4 * k < ww) {
          const int last = min(4 * k + 3, ww - 1);
          const unsigned lo = srcw[k];
          const unsigned hi = (sh > 0 && last + sh >= 4 * k + 4) ? srcw[k + 1] : 0u;
          v = __funnelshift_r(lo, hi, 8 * sh);
          const int rem = ww - 4 * k;
          if (rem < 4) v &= (1u << (8 * rem)) - 1u;
        }
        sm.win[e] = v;
      }
    } else {
      for (int e = lane; e < wh * MW_WS; e += 32) {
        const int yy = e / MW_WS, xx = e - yy * MW_WS;
        win[e] = (xx < ww) ? jb.frame[(size_t)(y0 + yy) * jb.fstride + x0 + xx] : (uint8_t)0;
      }
    }
  }
  __syncwarp();
  const double dn = (double)w2;
  const double m1 = __ddiv_rn((double)T, dn);
  const double d1 = dn * (double)TT - (double)T * (double)T;   // exact (< 2^53)
  const double rd1 = (d1 > 0.0) ? rsqrt(d1) : 0.0;
  const double kNone = -1.0e300;
  // --- fast pass: ncc* of every in-ellipse candidate; lane -> candidates lane, lane + 32, ... (row-major over the grid) ---
  const int ncand = cw * ch;
  const unsigned lastmask = (w & 3) ? ((1u << (8 * (w & 3))) - 1u) : 0xffffffffu;   // bytes of the last template word of a row
  double sc[8];
  int Pq[8];
  double lmax = kNone;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    sc[q] = kNone; Pq[q] = 0;
    const int c = lane + 32 * q;
    if (c < ncand) {
      const int jv = c / cw, iu = c - jv * cw;
      const float dj = (float)(G.jlo + jv - G.vc);
      const float ey = __fmul_rn(__fmul_rn(G.y_2_coeff, dj), dj);
      const float fdi = (float)(G.ilo + iu - G.uc);
      const float e = __fadd_rn(__fadd_rn(__fmul_rn(__fmul_rn(G.x_2_coeff, fdi), fdi), ey), __fmul_rn(__fmul_rn(G.yx_coeff, fdi), dj));
      if (e <= G.sigma_2) {
        unsigned stp = 0, P = 0, PP = 0;
        const int shb = 8 * (iu & 3);
        for (int r = 0; r < w; ++r) {
          const unsigned* wr = sm.win + ((jv + r) * MW_WS + (iu & ~3)) / 4;
          const unsigned* tr = sm.tpk + r * tw;
          unsigned lo = wr[0];
          for (int k = 0; k < tw; ++k) {
            const unsigned hi = wr[k + 1];
            unsigned x = __funnelshift_r(lo, hi, shb);
            if (k == tw - 1) x &= lastmask;
            stp = __dp4a(x, tr[k], stp);
            P = __dp4a(x, 0x01010101u, P);
            PP = __dp4a(x, x, PP);
            lo = hi;
          }
        }
        Pq[q] = (int)P;
        const double d2 = dn * (double)PP - (double)P * (double)P;   // exact (< 2^53)
        if (d1 > 0.0 && d2 > 0.0) {
          const double num = dn * (double)stp - (double)T * (double)P;
          const double v = (num * rd1) * rsqrt(d2);
          sc[q] = v;
          if (v > lmax) lmax = v;
        }
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) lmax = fmax(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
  const double Mstar = lmax;
  float best = -1.0f;
  int bestkey = 0x7fffffff;
  if (Mstar > kNone) {
    const float fm = fabsf((float)Mstar);
    const double ulp = (double)(nextafterf(fm, 3.0e38f) - fm);
    const double thr = Mstar - (2.0 * ulp + 4.0e-12);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      if (sc[q] >= thr) {
        const int slot = atomicAdd(&sm.cnt, 1);
        if (slot < MW_LIST) sm.list[slot] = (lane + 32 * q) | (Pq[q] << 8);
      }
    }
    __syncwarp();
    const int nlist = sm.cnt;
    if (nlist > MW_LIST) return false;   // pathological ties: leave it to match_one (nothing has been written)
    const int role = lane & 3, gbase = lane & ~3;
    const unsigned gmask = 0xfu << gbase;
    for (int q0 = 0; q0 < nlist; q0 += 8) {
      const int q = q0 + (lane >> 2);
      if (q >= nlist) continue;                         // uniform inside a 4-lane group
      const int c = sm.list[q] & 255, P = sm.list[q] >> 8;
      const int jv = c / cw, iu = c - jv * cw;
      const float s1 = match_exact_score4_tb(sm.tb, m1, win, MW_WS, jv * MW_WS + iu, w, P, role, gmask, gbase);
      const int key = (G.ilo + iu - G.i0) * G.nv + (G.jlo + jv - G.j0);
      if (role == 0 && (s1 > best || (s1 == best && key < bestkey))) { best = s1; bestkey = key; }
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int ok = __shfl_xor_sync(0xffffffffu, bestkey, o);
    if (ob > best || (ob == best && ok < bestkey)) { best = ob; bestkey = ok; }
  }
  res.best = best;
  if (bestkey != 0x7fffffff && G.nv > 0) {
    res.bi = G.i0 + bestkey / G.nv;
    res.bj = G.j0 + bestkey % G.nv;
  }
  return true;
}

// ------------------------------------------------------------------------------------------------
// Warp-per-feature path for FULL windows (candidate grid up to 41 x 41 at the reference's +-20 px clamp), template side W <= 12
// fixed at compile time: the register-tiled scoring core of ekf_match_tile.cuh.  Only the u8 window (54 rows x 76 bytes), the
// packed template and the band list sit in shared memory (4.6 KB per warp); the lanes take 4 x 4-candidate tiles round-robin,
// rank them by an exact-integer float score, and only the band candidates see double precision and the reference's exact pass.
// No block barrier anywhere.  Returns false (nothing written, nothing decided) when the feature needs the CTA matcher.
// ------------------------------------------------------------------------------------------------
// The reference's computeCorrelation for one candidate on a 4-lane group, template side fixed at compile time and no selects in
// the loop: every lane runs acc += (A[x] - mA) * (B[x] - mB) over the pixels in row-major order with its own operand pair —
// role 0: template x template (n1), role 1: window x window (n2), roles 2 / 3: template x window (corr).  (double)(float) of
// an 8-bit pixel is the pixel, so the conversion is direct; sums and products are the reference's, one rounding each.
template <int W>
__device__ __forceinline__ float match_exact_score3(const unsigned char* tb, double m1, const uint8_t* win, int wsb, int roi, int P,
                                                    int role, unsigned gmask, int gbase) {
  const double m2 = __ddiv_rn((double)P, (double)(W * W));
  const uint8_t* srcA = role == 1 ? win + roi : tb;
  const uint8_t* srcB = role == 0 ? tb : win + roi;
  const int strA = role == 1 ? wsb : W, strB = role == 0 ? W : wsb;
  const double mA = role == 1 ? m2 : m1, mB = role == 0 ? m1 : m2;
  double acc = 0;
  for (int r = 0; r < W; ++r) {
    const uint8_t* pa = srcA + r * strA;
    const uint8_t* pb = srcB + r * strB;
#pragma unroll
    for (int x = 0; x < W; ++x) {
      const double a = __dsub_rn((double)pa[x], mA);
      const double b = __dsub_rn((double)pb[x], mB);
      acc = __dadd_rn(acc, __dmul_rn(a, b));
    }
  }
  const double n1 = __shfl_sync(gmask, acc, gbase), n2 = __shfl_sync(gmask, acc, gbase + 1), corr = __shfl_sync(gmask, acc, gbase + 2);
  return (float)__ddiv_rn(corr, __dsqrt_rn(__dmul_rn(n2, n1)));
}

#define MW2_WARPS 8
template <int W>
struct MatchWarp2Smem {
  unsigned win[(MT_MAXGRID + W - 1 + MT_R - 1) * MT_WSW];
  unsigned tpk[W * ((W + 3) / 4)];
  unsigned char tb[((W * W + 15) & ~15) + 16];
  uint4 list[MT_LIST];   // {candidate index, Stp, P, PP}
  int cnt;
};

template <int W, bool TSMEM, bool SLIDE>
__device__ bool match_one_warp2(const MatchJob& jb, float sigma_size, float clampv, MatchWarp2Smem<W>& sm, MatchResult& res) {
  constexpr int TW = (W + 3) / 4, W2 = W * W;
  const int lane = threadIdx.x & 31;
  if (!(clampv <= 20.0f)) return false;
  const MatchGeom G = match_geometry(jb, W, sigma_size, clampv, MT_MAXGRID);
  res.best = -1.0f; res.bi = 0; res.bj = 0;
  if (!G.any) return true;
  const int cw = G.cw, ch = G.ch;
  // --- template: packed words (zero padded), bytes, T = sum t, TT = sum t^2 ---
  int T = 0, TT = 0;
  for (int e = lane; e < W * TW; e += 32) {
    const int r = e / TW, k4 = (e - r * TW) * 4;
    unsigned word = 0;
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (k4 + c < W) {
        const unsigned v = jb.tmpl[r * W + k4 + c];
        word |= v << (8 * c);
        T += (int)v; TT += (int)(v * v);
      }
    sm.tpk[e] = word;
  }
  for (int e = lane; e < W2; e += 32) sm.tb[e] = jb.tmpl[e];
  for (int o = 16; o > 0; o >>= 1) { T += __shfl_xor_sync(0xffffffffu, T, o); TT += __shfl_xor_sync(0xffffffffu, TT, o); }
  mt_stage_window(sm.win, jb, G, W, lane, 32);
  __syncwarp();
  const double dn = (double)W2;
  const double m1 = __ddiv_rn((double)T, dn);
  const double d1 = dn * (double)TT - (double)T * (double)T;   // exact (< 2^53)
  if (!(d1 > 0.0)) return true;                                 // flat template: 0/0 in the reference for every candidate
  const double rd1 = rsqrt(d1);
  // --- ranking pass: tiles round-robin over the lanes ---
  MTTop top;
  top.reset();
  {
    unsigned Treg[TSMEM ? 1 : W * TW];   // TSMEM: the template words are shared-memory operands (broadcast loads) instead of 33 registers
    if (!TSMEM) {
#pragma unroll
      for (int e = 0; e < W * TW; ++e) Treg[e] = sm.tpk[e];
    }
    MTGate g;
    g.x2c = G.x_2_coeff; g.y2c = G.y_2_coeff; g.yxc = G.yx_coeff; g.sigma2 = G.sigma_2;
    g.du0 = G.ilo - G.uc; g.dv0 = G.jlo - G.vc; g.cw = cw; g.ch = ch; g.T = T; g.rd1f = (float)rd1;
    const int ntx = (cw + 3) >> 2, nty = (ch + MT_R - 1) / MT_R;
    int ty = lane / ntx, tx = lane - ty * ntx;
    const int dty = 32 / ntx, dtx = 32 - dty * ntx;
    while (ty < nty) {
      if (TSMEM) mt_tile<W, MT_R, SLIDE>(sm.win, tx, ty, sm.tpk, g, top);
      else mt_tile<W, MT_R, SLIDE>(sm.win, tx, ty, reinterpret_cast<const unsigned (&)[W * TW]>(Treg), g, top);
      tx += dtx; ty += dty;
      if (tx >= ntx) { tx -= ntx; ++ty; }
    }
  }
  float F = top.a0;
  for (int o = 16; o > 0; o >>= 1) F = fmaxf(F, __shfl_xor_sync(0xffffffffu, F, o));
  if (!(F > -INFINITY)) return true;                            // no candidate inside the ellipse with a textured window
  const float thrF = F - MT_BAND;
  const bool crowded = top.a2 >= thrF;                          // a lane may have dropped a band candidate
  if (__any_sync(0xffffffffu, crowded)) return false;
  if (top.a0 >= thrF) {
    const int slot = atomicAdd(&sm.cnt, 1);
    if (slot < MT_LIST) sm.list[slot] = make_uint4((unsigned)top.i0, top.s0, (unsigned)top.p0, (unsigned)top.q0);
  }
  if (top.a1 >= thrF) {
    const int slot = atomicAdd(&sm.cnt, 1);
    if (slot < MT_LIST) sm.list[slot] = make_uint4((unsigned)top.i1, top.s1, (unsigned)top.p1, (unsigned)top.q1);
  }
  __syncwarp();
  const int nlist = sm.cnt;
  if (nlist > MT_LIST) return false;
  // --- ncc* in double of the band candidates, its maximum, the guard band (as match_one) ---
  const double kNone = -1.0e300;
  double v = kNone;
  if (lane < nlist) {
    const uint4 c = sm.list[lane];
    v = mt_ncc_star(W2, c.y, (int)c.z, (int)c.w, T, rd1);
  }
  double Mstar = v;
  for (int o = 16; o > 0; o >>= 1) Mstar = fmax(Mstar, __shfl_xor_sync(0xffffffffu, Mstar, o));
  const float fm = fabsf((float)Mstar);
  const double ulp = (double)(nextafterf(fm, 3.0e38f) - fm);
  const double thr = Mstar - (2.0 * ulp + 4.0e-12);
  // --- exact pass: one 4-lane group per guard-band candidate ---
  float best = -1.0f;
  int bestkey = 0x7fffffff;
  const uint8_t* winb = reinterpret_cast<const uint8_t*>(sm.win);
  const int role = lane & 3, gbase = lane & ~3;
  const unsigned gmask = 0xfu << gbase;
  for (int q0 = 0; q0 < nlist; q0 += 8) {
    const int q = q0 + (lane >> 2);
    if (q >= nlist) continue;                           // uniform inside a 4-lane group
    const uint4 c = sm.list[q];
    if (!(mt_ncc_star(W2, c.y, (int)c.z, (int)c.w, T, rd1) >= thr)) continue;   // same value in the four lanes
    const int jv = (int)c.x / cw, iu = (int)c.x - jv * cw;
    const float s1 = match_exact_score3<W>(sm.tb, m1, winb, MT_WSW * 4, jv * MT_WSW * 4 + iu, (int)c.z, role, gmask, gbase);
    const int key = (G.ilo + iu - G.i0) * G.nv + (G.jlo + jv - G.j0);
    if (role == 0 && (s1 > best || (s1 == best && key < bestkey))) { best = s1; bestkey = key; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int ok = __shfl_xor_sync(0xffffffffu, bestkey, o);
    if (ob > best || (ob == best && ok < bestkey)) { best = ob; bestkey = ok; }
  }
  res.best = best;
  if (bestkey != 0x7fffffff && G.nv > 0) {
    res.bi = G.i0 + bestkey / G.nv;
    res.bj = G.j0 + bestkey % G.nv;
  }
  return true;
}

// ------------------------------------------------------------------------------------------------
// The same scoring core for ONE feature per CTA (the single-filter path: a few hundred features per frame, where the latency
// of a feature counts, not the throughput): MATCH_THREADS threads take the 4 x 2-candidate tiles of the feature (231 tiles
// of a 41 x 41 grid: one round), the band list is shared, warp 0 finishes.  Four block barriers instead of match_one's
// seven phases through shared memory.  The verdict is uniform over the CTA: false = match_one must run (nothing written).
// ------------------------------------------------------------------------------------------------
template <int W>
struct MatchTileCtaSmem {
  MatchWarp2Smem<W> w;
  int T, TT;
  float fmax[MATCH_THREADS / 32];
  float best;
  int bi, bj;
};
template <int W, int R>
__device__ bool match_one_tile_cta(const MatchJob& jb, float sigma_size, float clampv, unsigned char* smem_raw, MatchResult& res) {
  constexpr int TW = (W + 3) / 4, W2 = W * W;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  MatchTileCtaSmem<W>& cs = *reinterpret_cast<MatchTileCtaSmem<W>*>(smem_raw);
  MatchWarp2Smem<W>& sm = cs.w;
  res.best = -1.0f; res.bi = 0; res.bj = 0;
  if (!(clampv <= 20.0f)) return false;
  const MatchGeom G = match_geometry(jb, W, sigma_size, clampv, MT_MAXGRID);
  if (!G.any) return true;
  const int cw = G.cw, ch = G.ch;
  if (tid == 0) { sm.cnt = 0; cs.T = 0; cs.TT = 0; }
  __syncthreads();
  // --- template: packed words, bytes, T, TT ---
  {
    int pt = 0, ptt = 0;
    for (int e = tid; e < W * TW; e += MATCH_THREADS) {
      const int r = e / TW, k4 = (e - r * TW) * 4;
      unsigned word = 0;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (k4 + c < W) {
          const unsigned v = jb.tmpl[r * W + k4 + c];
          word |= v << (8 * c);
          pt += (int)v; ptt += (int)(v * v);
        }
      sm.tpk[e] = word;
    }
    for (int e = tid; e < W2; e += MATCH_THREADS) sm.tb[e] = jb.tmpl[e];
    for (int o = 16; o > 0; o >>= 1) { pt += __shfl_xor_sync(0xffffffffu, pt, o); ptt += __shfl_xor_sync(0xffffffffu, ptt, o); }
    if (lane == 0 && (pt | ptt)) { atomicAdd(&cs.T, pt); atomicAdd(&cs.TT, ptt); }
  }
  mt_stage_window(sm.win, jb, G, W, tid, MATCH_THREADS);
  __syncthreads();
  const int T = cs.T, TT = cs.TT;
  const double dn = (double)W2;
  const double m1 = __ddiv_rn((double)T, dn);
  const double d1 = dn * (double)TT - (double)T * (double)T;   // exact (< 2^53)
  if (!(d1 > 0.0)) return true;                                 // flat template
  const double rd1 = rsqrt(d1);
  // --- ranking pass ---
  MTTop top;
  top.reset();
  {
    const int ntx = (cw + 3) >> 2, nty = (ch + R - 1) / R;
    const int ntiles = ntx * nty;
    if (tid < ntiles) {
      MTGate g;
      g.x2c = G.x_2_coeff; g.y2c = G.y_2_coeff; g.yxc = G.yx_coeff; g.sigma2 = G.sigma_2;
      g.du0 = G.ilo - G.uc; g.dv0 = G.jlo - G.vc; g.cw = cw; g.ch = ch; g.T = T; g.rd1f = (float)rd1;
      for (int t = tid; t < ntiles; t += MATCH_THREADS) {
        const int ty = t / ntx, tx = t - ty * ntx;
        mt_tile<W, R>(sm.win, tx, ty, sm.tpk, g, top);   // template words straight from shared memory (broadcast): 64 registers, 4 CTAs per SM
      }
    }
  }
  float F = top.a0;
  for (int o = 16; o > 0; o >>= 1) F = fmaxf(F, __shfl_xor_sync(0xffffffffu, F, o));
  if (lane == 0) cs.fmax[warp] = F;
  __syncthreads();
#pragma unroll
  for (int wv = 0; wv < MATCH_THREADS / 32; ++wv) F = fmaxf(F, cs.fmax[wv]);
  if (!(F > -INFINITY)) return true;
  const float thrF = F - MT_BAND;
  if (__syncthreads_or(top.a2 >= thrF)) return false;           // a thread may have dropped a band candidate
  if (top.a0 >= thrF) {
    const int slot = atomicAdd(&sm.cnt, 1);
    if (slot < MT_LIST) sm.list[slot] = make_uint4((unsigned)top.i0, top.s0, (unsigned)top.p0, (unsigned)top.q0);
  }
  if (top.a1 >= thrF) {
    const int slot = atomicAdd(&sm.cnt, 1);
    if (slot < MT_LIST) sm.list[slot] = make_uint4((unsigned)top.i1, top.s1, (unsigned)top.p1, (unsigned)top.q1);
  }
  __syncthreads();
  const int nlist = sm.cnt;
  if (nlist > MT_LIST) return false;
  if (warp == 0) {
    // --- ncc* in double of the band candidates, the guard band, the exact pass (as match_one_warp2) ---
    const double kNone = -1.0e300;
    double v = kNone;
    if (lane < nlist) {
      const uint4 c = sm.list[lane];
      v = mt_ncc_star(W2, c.y, (int)c.z, (int)c.w, T, rd1);
    }
    double Mstar = v;
    for (int o = 16; o > 0; o >>= 1) Mstar = fmax(Mstar, __shfl_xor_sync(0xffffffffu, Mstar, o));
    const float fm = fabsf((float)Mstar);
    const double ulp = (double)(nextafterf(fm, 3.0e38f) - fm);
    const double thr = Mstar - (2.0 * ulp + 4.0e-12);
    float best = -1.0f;
    int bestkey = 0x7fffffff;
    const uint8_t* winb = reinterpret_cast<const uint8_t*>(sm.win);
    const int role = lane & 3, gbase = lane & ~3;
    const unsigned gmask = 0xfu << gbase;
    for (int q0 = 0; q0 < nlist; q0 += 8) {
      const int q = q0 + (lane >> 2);
      if (q >= nlist) continue;
      const uint4 c = sm.list[q];
      if (!(mt_ncc_star(W2, c.y, (int)c.z, (int)c.w, T, rd1) >= thr)) continue;
      const int jv = (int)c.x / cw, iu = (int)c.x - jv * cw;
      const float s1 = match_exact_score3<W>(sm.tb, m1, winb, MT_WSW * 4, jv * MT_WSW * 4 + iu, (int)c.z, role, gmask, gbase);
      const int key = (G.ilo + iu - G.i0) * G.nv + (G.jlo + jv - G.j0);
      if (role == 0 && (s1 > best || (s1 == best && key < bestkey))) { best = s1; bestkey = key; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int ok = __shfl_xor_sync(0xffffffffu, bestkey, o);
      if (ob > best || (ob == best && ok < bestkey)) { best = ob; bestkey = ok; }
    }
    if (lane == 0) {
      cs.best = best; cs.bi = 0; cs.bj = 0;
      if (bestkey != 0x7fffffff && G.nv > 0) {
        cs.bi = G.i0 + bestkey / G.nv;
        cs.bj = G.j0 + bestkey % G.nv;
      }
    }
  }
  __syncthreads();
  res.best = cs.best; res.bi = cs.bi; res.bj = cs.bj;
  return true;
}

// write-back of one matched (or rejected) feature by its warp: Patch.cpp:278-289; the new template comes from the frame
__device__ __forceinline__ void match_warp_commit(FeatTab ft, int f, FrameView fr, const DevCfg& cfg, const MatchResult& r) {
  const int lane = threadIdx.x & 31, w = cfg.window, w2 = w * w;
  const bool accept = !(r.best < cfg.ncc_threshold);  // Patch.cpp:278
  if (accept) {   // matching_patch <- matched ROI (Patch.cpp:285)
    const int x0 = r.bi - w / 2, y0 = r.bj - w / 2;
    for (int e = lane; e < w2; e += 32)
      ft.mpatch[(size_t)f * cfg.tstride + e] = fr.px[(size_t)(y0 + e / w) * fr.stride + x0 + (e % w)];
  }
  if (lane == 0) {
    ft.n_tot[f] += 1;  // Patch.cpp:218
    ft.last_ncc[f] = r.best;
    if (!accept) {
      ft.center[2 * f] = -1.0f; ft.center[2 * f + 1] = -1.0f;
      ft.innov[f] = 0; ft.li[f] = 0; ft.hi[f] = 0;
    } else {
      ft.center[2 * f] = (float)r.bi; ft.center[2 * f + 1] = (float)r.bj;
      ft.z[2 * f] = (double)(float)r.bi; ft.z[2 * f + 1] = (double)(float)r.bj;
    }
  }
}

// The frame filter b searches: camera cam_of[b] of the batch's contiguous frame stack.  The camera is also the z coordinate of
// the stack's tensor map, which only the CTA matcher reads.  The batched matcher kernels take CAMS = false with one camera, and
// then compile to the code that reads the one frame from the kernel's parameters.
__device__ __forceinline__ FrameView batch_frame(FrameView fr, int cam) {
  fr.px += (size_t)cam * fr.h * fr.stride;
  return fr;
}
// SIZES (ekf_batch_set_frame_sizes): camera c's frame is the top-left fsize[4c + 2] x fsize[4c + 3] of its slot, and the window
// clipping uses that size.  cam_of may then be null (one camera).  Without sizes the kernels take SIZES = false, today's code.
template <bool CAMS, bool SIZES>
__device__ __forceinline__ FrameView batch_frame_of(FrameView fr, const int* __restrict__ cam_of, const int* __restrict__ fsize, int b) {
  if constexpr (SIZES) {
    const int c = cam_of ? cam_of[b] : 0;
    fr = batch_frame(fr, c);
    fr.w = fsize[4 * c + 2]; fr.h = fsize[4 * c + 3];
  } else if constexpr (CAMS) {
    fr = batch_frame(fr, cam_of[b]);
  }
  return fr;
}

// ACT (ekf_batch_step_filters): the pairs run over the B = n listed filters, the list's entry i being filter act[i]; the deferred
// list keeps the pair of the filter itself, b * Ncap + f.  Without a list the kernels are the code they were before.
template <bool ACT>
__device__ __forceinline__ int batch_pair_filter(const int* __restrict__ act, int i) {
  if constexpr (ACT) return act[i];
  else return i;
}

// Batched filters, pass 1 with the full-window warp matcher (template side 11): one warp per (filter, feature)
template <int MINB, bool TSMEM, bool SLIDE, bool CAMS, bool SIZES, bool ACT>
__global__ void __launch_bounds__(MW2_WARPS * 32, MINB) k_match_filter_batch_warp2(FeatTab base, int Ncap, const int* __restrict__ Nper, int B,
                                                                                FrameView fr, DevCfg cfg, int* __restrict__ defer_list,
                                                                                int* __restrict__ defer_cnt, const int* __restrict__ cam_of,
                                                                                const int* __restrict__ fsize, const int* __restrict__ act) {
  __shared__ MatchWarp2Smem<11> wsm[MW2_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long pair_i = (long long)blockIdx.x * MW2_WARPS + warp;
  if (pair_i >= (long long)B * Ncap) return;
  const int i = (int)(pair_i / Ncap), f = (int)(pair_i - (long long)i * Ncap), b = batch_pair_filter<ACT>(act, i);
  const long long pair = ACT ? (long long)b * Ncap + f : pair_i;
  const FeatTab ft = feattab_slice(base, b, Ncap, cfg.tstride);
  if (f >= Nper[b] || !ft.innov[f]) return;
  MatchJob jb;
  fr = batch_frame_of<CAMS, SIZES>(fr, cam_of, fsize, b);
  jb.tmap = nullptr; jb.frame_index = 0;
  jb.frame = fr.px; jb.fw = fr.w; jb.fh = fr.h; jb.fstride = fr.stride;
  jb.tmpl = ft.mpatch + (size_t)f * cfg.tstride;
  jb.hu = ft.h[2 * f]; jb.hv = ft.h[2 * f + 1];
  for (int c = 0; c < 4; ++c) jb.S[c] = ft.S2[4 * f + c];
  if (lane == 0) wsm[warp].cnt = 0;
  __syncwarp();
  MatchResult r;
  if (!match_one_warp2<11, TSMEM, SLIDE>(jb, cfg.sigma_size_f, cfg.search_clamp, wsm[warp], r)) {
    if (lane == 0) defer_list[atomicAdd(defer_cnt, 1)] = (int)pair;
    return;
  }
  __syncwarp();
  match_warp_commit(ft, f, fr, cfg, r);
}

// Batched filters, pass 1: one warp per (filter, feature); features that do not fit go to defer_list.
template <bool CAMS, bool SIZES, bool ACT>
__global__ void __launch_bounds__(MW_WARPS * 32) k_match_filter_batch_warp(FeatTab base, int Ncap, const int* __restrict__ Nper, int B,
                                                                           FrameView fr, DevCfg cfg, int* __restrict__ defer_list,
                                                                           int* __restrict__ defer_cnt, int warp_path,
                                                                           const int* __restrict__ cam_of, const int* __restrict__ fsize,
                                                                           const int* __restrict__ act) {
  __shared__ MatchWarpSmem wsm[MW_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long pair_i = (long long)blockIdx.x * MW_WARPS + warp;
  if (pair_i >= (long long)B * Ncap) return;
  const int i = (int)(pair_i / Ncap), f = (int)(pair_i - (long long)i * Ncap), b = batch_pair_filter<ACT>(act, i);
  const long long pair = ACT ? (long long)b * Ncap + f : pair_i;
  const FeatTab ft = feattab_slice(base, b, Ncap, cfg.tstride);
  if (f >= Nper[b] || !ft.innov[f]) return;
  const int w = cfg.window, w2 = w * w;
  MatchJob jb;
  fr = batch_frame_of<CAMS, SIZES>(fr, cam_of, fsize, b);
  jb.tmap = nullptr; jb.frame_index = 0;
  jb.frame = fr.px; jb.fw = fr.w; jb.fh = fr.h; jb.fstride = fr.stride;
  jb.tmpl = ft.mpatch + (size_t)f * cfg.tstride;
  jb.hu = ft.h[2 * f]; jb.hv = ft.h[2 * f + 1];
  for (int c = 0; c < 4; ++c) jb.S[c] = ft.S2[4 * f + c];
  if (lane == 0) wsm[warp].cnt = 0;
  __syncwarp();
  MatchResult r;
  if (!warp_path || !match_one_warp(jb, w, cfg.sigma_size_f, cfg.search_clamp, wsm[warp], r)) {
    if (lane == 0) defer_list[atomicAdd(defer_cnt, 1)] = (int)pair;
    return;
  }
  __syncwarp();
  const bool accept = !(r.best < cfg.ncc_threshold);  // Patch.cpp:278
  if (accept) {   // matching_patch <- matched ROI (Patch.cpp:285)
    const int x0 = r.bi - w / 2, y0 = r.bj - w / 2;
    for (int e = lane; e < w2; e += 32)
      ft.mpatch[(size_t)f * cfg.tstride + e] = fr.px[(size_t)(y0 + e / w) * fr.stride + x0 + (e % w)];
  }
  if (lane == 0) {
    ft.n_tot[f] += 1;  // Patch.cpp:218
    ft.last_ncc[f] = r.best;
    if (!accept) {
      ft.center[2 * f] = -1.0f; ft.center[2 * f + 1] = -1.0f;
      ft.innov[f] = 0; ft.li[f] = 0; ft.hi[f] = 0;
    } else {
      ft.center[2 * f] = (float)r.bi; ft.center[2 * f + 1] = (float)r.bj;
      ft.z[2 * f] = (double)(float)r.bi; ft.z[2 * f + 1] = (double)(float)r.bj;
    }
  }
}
// pass 2: a persistent grid of CTAs works off the deferred (filter, feature) pairs with match_one
template <bool CAMS, bool SIZES>
__global__ void __launch_bounds__(MATCH_THREADS) k_match_filter_batch_deferred(FeatTab base, int Ncap, FrameView fr, DevCfg cfg,
                                                                               const __grid_constant__ CUtensorMap tmap, int use_tma,
                                                                               const int* __restrict__ defer_list,
                                                                               const int* __restrict__ defer_cnt,
                                                                               const int* __restrict__ cam_of,
                                                                               const int* __restrict__ fsize) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int n = *defer_cnt;
  unsigned phase = 0;
  bool first = true;
  for (int i = blockIdx.x; i < n; i += gridDim.x) {
    const int pair = defer_list[i];
    const int b = pair / Ncap, f = pair - b * Ncap;
    const FeatTab ft = feattab_slice(base, b, Ncap, cfg.tstride);
    const int cam = ((CAMS || SIZES) && cam_of) ? cam_of[b] : 0;
    match_filter_feature(ft, f, batch_frame_of<CAMS, SIZES>(fr, cam_of, fsize, b), cfg, smem_raw, use_tma ? &tmap : nullptr, &phase,
                         first, false, cam);
    first = false;
    __syncthreads();
  }
}

// Stateless batch (BASELINE config 5): grid = frames x features.
__global__ void __launch_bounds__(MATCH_THREADS) k_match_batch(const uint8_t* __restrict__ frames, int width, int height,
                                                               int stride, const uint8_t* __restrict__ templates, int fpf,
                                                               int w, const double* __restrict__ hh, const double* __restrict__ Sm,
                                                               float sigma_size, float thr, float clampv,
                                                               int32_t* __restrict__ out_uv, float* __restrict__ out_score, int total,
                                                               const __grid_constant__ CUtensorMap tmap, int use_tma) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int idx = blockIdx.x;
  if (idx >= total) return;
  MatchJob jb;
  jb.tmap = use_tma ? &tmap : nullptr; jb.frame_index = idx / fpf;
  jb.frame = frames + (size_t)(idx / fpf) * height * stride;
  jb.fw = width; jb.fh = height; jb.fstride = stride;
  jb.tmpl = templates + (size_t)idx * w * w;
  jb.hu = hh[2 * idx]; jb.hv = hh[2 * idx + 1];
  for (int c = 0; c < 4; ++c) jb.S[c] = Sm[4 * idx + c];
  const MatchResult r = match_one(jb, w, sigma_size, clampv, smem_raw);
  if (threadIdx.x == 0) {
    const bool accept = !(r.best < thr);
    out_uv[2 * idx] = accept ? r.bi : -1;
    out_uv[2 * idx + 1] = accept ? r.bj : -1;
    out_score[idx] = r.best;
  }
}

// Stateless batch with the full-window warp matcher (template side 11): one warp per (frame, feature).  A feature that needs
// the CTA matcher is MARKED in out_uv and worked off by the persistent grid of k_match_batch_marked.
#define MATCH_MARK ((int32_t)0x80000000)
template <int MINB, bool TSMEM, bool SLIDE>
__global__ void __launch_bounds__(MW2_WARPS * 32, MINB) k_match_batch_warp2(const uint8_t* __restrict__ frames, int width, int height, int stride,
                                                                         const uint8_t* __restrict__ templates, int fpf,
                                                                         const double* __restrict__ hh, const double* __restrict__ Sm,
                                                                         float sigma_size, float thr, float clampv,
                                                                         int32_t* __restrict__ out_uv, float* __restrict__ out_score, int total) {
  __shared__ MatchWarp2Smem<11> wsm[MW2_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int idx = blockIdx.x * MW2_WARPS + warp;
  if (idx >= total) return;
  MatchJob jb;
  jb.tmap = nullptr; jb.frame_index = idx / fpf;
  jb.frame = frames + (size_t)(idx / fpf) * height * stride;
  jb.fw = width; jb.fh = height; jb.fstride = stride;
  jb.tmpl = templates + (size_t)idx * 121;
  jb.hu = hh[2 * idx]; jb.hv = hh[2 * idx + 1];
  for (int c = 0; c < 4; ++c) jb.S[c] = Sm[4 * idx + c];
  if (lane == 0) wsm[warp].cnt = 0;
  __syncwarp();
  MatchResult r;
  const bool done = match_one_warp2<11, TSMEM, SLIDE>(jb, sigma_size, clampv, wsm[warp], r);
  if (lane == 0) {
    if (!done) {
      out_uv[2 * idx] = MATCH_MARK;
    } else {
      const bool accept = !(r.best < thr);
      out_uv[2 * idx] = accept ? r.bi : -1;
      out_uv[2 * idx + 1] = accept ? r.bj : -1;
      out_score[idx] = r.best;
    }
  }
}
__global__ void __launch_bounds__(MATCH_THREADS) k_match_batch_marked(const uint8_t* __restrict__ frames, int width, int height,
                                                                      int stride, const uint8_t* __restrict__ templates, int fpf,
                                                                      int w, const double* __restrict__ hh, const double* __restrict__ Sm,
                                                                      float sigma_size, float thr, float clampv,
                                                                      int32_t* __restrict__ out_uv, float* __restrict__ out_score, int total,
                                                                      const __grid_constant__ CUtensorMap tmap, int use_tma) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  unsigned phase = 0;
  bool first = true;
  for (int idx = blockIdx.x; idx < total; idx += gridDim.x) {
    if (out_uv[2 * idx] != MATCH_MARK) continue;   // uniform over the CTA
    MatchJob jb;
    jb.tmap = use_tma ? &tmap : nullptr; jb.frame_index = idx / fpf;
    jb.frame = frames + (size_t)(idx / fpf) * height * stride;
    jb.fw = width; jb.fh = height; jb.fstride = stride;
    jb.tmpl = templates + (size_t)idx * w * w;
    jb.hu = hh[2 * idx]; jb.hv = hh[2 * idx + 1];
    for (int c = 0; c < 4; ++c) jb.S[c] = Sm[4 * idx + c];
    const MatchResult r = match_one(jb, w, sigma_size, clampv, smem_raw, &phase, first);
    first = false;
    __syncthreads();   // every thread has read the mark before thread 0 overwrites it
    if (threadIdx.x == 0) {
      const bool accept = !(r.best < thr);
      out_uv[2 * idx] = accept ? r.bi : -1;
      out_uv[2 * idx + 1] = accept ? r.bj : -1;
      out_score[idx] = r.best;
    }
    __syncthreads();
  }
}

// EKF_MATCH_W2VAR: build of the warp tile matcher — 0 template words in registers, 2 CTAs per SM (128 registers); 1 template
// words as shared-memory operands, 2 CTAs; 2 shared-memory operands, 3 CTAs per SM (80 registers); + 4: window sums of the three
// right-hand candidates by sliding (mt_tile SLIDE).  Measured (tools/match_ab.py, 12 800 features per launch): 0 / 1 / 2 / 4 / 5 / 6 =
// 52.3 / 55.2 / 54.4 / 51.9 / 55.6 / 53.4 M matches/s — DP4A and IMAD share one pipe (tools/idp_rate_probe: 2 warp-instructions per
// cycle per SM each and together), so sliding buys nothing; default 1.
static int match_w2_variant() {
  const char* e = getenv("EKF_MATCH_W2VAR");   // read per call: tools/match_ab.py switches it inside one process
  return e ? atoi(e) : 1;
}

void launch_match_filter(cudaStream_t st, FeatTab ft, int N, FrameView fr, const DevCfg& cfg, const EkfTensorMap* tmap, long long* launches) {
  if (N <= 0) return;
  static PerDeviceOnce once;   // opt in to the largest supported window once per device
  size_t smem = match_smem_bytes(cfg.window, cfg.search_clamp);
  if (smem < sizeof(MatchTileCtaSmem<11>)) smem = sizeof(MatchTileCtaSmem<11>);   // the tile matcher's fixed-size window buffer
  if (once.ensure([] { return cudaFuncSetAttribute(k_match_filter, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   (int)match_smem_bytes(MATCH_MAX_W, 20.0f)); }) != cudaSuccess) return;   // the error stays in cudaGetLastError() for the caller
  static const EkfTensorMap none{};
  const EkfTensorMap& tm = (tmap && tmap->ok) ? *tmap : none;
  static const int tile = [] { const char* e = getenv("EKF_MATCH_WARP"); return (e ? atoi(e) : 2) >= 2; }();   // the tile matcher ahead of match_one
  k_match_filter<<<N, MATCH_THREADS, smem, st>>>(ft, N, fr, cfg, as_cu(tm), tm.ok, tile);
  *launches += 1;
}

void launch_match_filter_batch(cudaStream_t st, FeatTab base, int Ncap, const int* Nper, int B, FrameView fr, const DevCfg& cfg,
                               const EkfTensorMap* tmap, int* defer_list, int* defer_cnt, long long* launches, const int* cam_of,
                               const int* fsize, const int* act) {
  if (B <= 0 || Ncap <= 0) return;
  static PerDeviceOnce once;   // opt in to the largest supported window once per device
  const size_t smem = match_smem_bytes(cfg.window, cfg.search_clamp);
  if (once.ensure([] {
        const int bytes = (int)match_smem_bytes(MATCH_MAX_W, 20.0f);
        cudaError_t e = cudaFuncSetAttribute(k_match_filter_batch_deferred<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_match_filter_batch_deferred<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        return e != cudaSuccess ? e : cudaFuncSetAttribute(k_match_filter_batch_deferred<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
      }) != cudaSuccess) return;   // the error stays in cudaGetLastError() for the caller
  static const EkfTensorMap none{};
  const EkfTensorMap& tm = (tmap && tmap->ok) ? *tmap : none;
  // pass 1: a warp per (filter, feature) for small windows; pass 2: a persistent grid of CTAs for the deferred rest
  cudaMemsetAsync(defer_cnt, 0, sizeof(int), st);
  const long long pairs = (long long)B * Ncap;
  // EKF_MATCH_WARP: 2 (default) full-window warp matcher where the template side allows it, 1 the small-window warp matcher only,
  // 0 every feature takes the CTA matcher (A/B timing, tests)
  static const int warp_path = [] { const char* e = getenv("EKF_MATCH_WARP"); return e ? atoi(e) : 2; }();
  if (warp_path >= 2 && cfg.window == 11 && cfg.search_clamp <= 20.0f) {
    const unsigned grid = (unsigned)((pairs + MW2_WARPS - 1) / MW2_WARPS);
    const int var = match_w2_variant();
#define MW2_LAUNCH_ACT(MINB, TS, SL, ACT)                                                                                               \
  if (fsize) k_match_filter_batch_warp2<MINB, TS, SL, true, true, ACT><<<grid, MW2_WARPS * 32, 0, st>>>(base, Ncap, Nper, B, fr, cfg, defer_list, defer_cnt, cam_of, fsize, act); \
  else if (cam_of) k_match_filter_batch_warp2<MINB, TS, SL, true, false, ACT><<<grid, MW2_WARPS * 32, 0, st>>>(base, Ncap, Nper, B, fr, cfg, defer_list, defer_cnt, cam_of, fsize, act); \
  else k_match_filter_batch_warp2<MINB, TS, SL, false, false, ACT><<<grid, MW2_WARPS * 32, 0, st>>>(base, Ncap, Nper, B, fr, cfg, defer_list, defer_cnt, cam_of, fsize, act)
#define MW2_LAUNCH(MINB, TS, SL)                   \
  if (act) { MW2_LAUNCH_ACT(MINB, TS, SL, true); } \
  else { MW2_LAUNCH_ACT(MINB, TS, SL, false); }
    switch (var) {
      case 0: MW2_LAUNCH(2, false, false); break;
      case 2: MW2_LAUNCH(3, true, false); break;
      case 4: MW2_LAUNCH(2, false, true); break;
      case 5: MW2_LAUNCH(2, true, true); break;
      case 6: MW2_LAUNCH(3, true, true); break;
      default: MW2_LAUNCH(2, true, false); break;   // 1
    }
#undef MW2_LAUNCH
#undef MW2_LAUNCH_ACT
  } else {
    const unsigned grid = (unsigned)((pairs + MW_WARPS - 1) / MW_WARPS);
#define MW_LAUNCH(ACT)                                                                                                                \
  if (fsize) k_match_filter_batch_warp<true, true, ACT><<<grid, MW_WARPS * 32, 0, st>>>(base, Ncap, Nper, B, fr, cfg, defer_list, defer_cnt, warp_path, cam_of, fsize, act); \
  else if (cam_of) k_match_filter_batch_warp<true, false, ACT><<<grid, MW_WARPS * 32, 0, st>>>(base, Ncap, Nper, B, fr, cfg, defer_list, defer_cnt, warp_path, cam_of, fsize, act); \
  else k_match_filter_batch_warp<false, false, ACT><<<grid, MW_WARPS * 32, 0, st>>>(base, Ncap, Nper, B, fr, cfg, defer_list, defer_cnt, warp_path, cam_of, fsize, act)
    if (act) { MW_LAUNCH(true); }
    else { MW_LAUNCH(false); }
#undef MW_LAUNCH
  }
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int per_sm = 4;   // persistent grid: as many CTAs as are resident at this shared-memory footprint
  auto* const deferred = fsize ? k_match_filter_batch_deferred<true, true>
                               : cam_of ? k_match_filter_batch_deferred<true, false> : k_match_filter_batch_deferred<false, false>;   // the one launched
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, deferred, MATCH_THREADS, smem) != cudaSuccess || per_sm < 1) {
    cudaGetLastError();
    per_sm = 4;
  }
  deferred<<<sms * per_sm, MATCH_THREADS, smem, st>>>(base, Ncap, fr, cfg, as_cu(tm), tm.ok, defer_list, defer_cnt, cam_of, fsize);
  *launches += 2;
}

int launch_match_batch(cudaStream_t st, const uint8_t* frames, int n_frames, int width, int height, int stride,
                       const uint8_t* templates, int fpf, int w, const double* h, const double* S, float sigma_size,
                       float thr, float clampv, int32_t* out_uv, float* out_score) {
  if (w > MATCH_MAX_W || w < 1 || clampv > 20.0f || !(clampv >= 0.0f)) return -1;
  const int total = n_frames * fpf;
  if (total <= 0) return 0;
  static PerDeviceOnce once;   // opt in to the largest supported window once per device
  const size_t smem = match_smem_bytes(w, clampv);
  if (once.ensure([] { return cudaFuncSetAttribute(k_match_batch, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                   (int)match_smem_bytes(MATCH_MAX_W, 20.0f)); }) != cudaSuccess) return -1;
  EkfTensorMap tm;
  match_make_tensor_map(&tm, frames, width, height, stride, n_frames, w, (int)clampv);
  static const int warp_path = [] { const char* e = getenv("EKF_MATCH_WARP"); return e ? atoi(e) : 2; }();
  if (warp_path >= 2 && w == 11) {
    // a warp per feature; what it cannot decide is marked and taken by a persistent grid of CTA matchers
    static PerDeviceOnce once2;
    if (once2.ensure([] { return cudaFuncSetAttribute(k_match_batch_marked, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                      (int)match_smem_bytes(MATCH_MAX_W, 20.0f)); }) != cudaSuccess) return -1;
    const int grid2 = (total + MW2_WARPS - 1) / MW2_WARPS, var = match_w2_variant();
#define MW2_LAUNCH(MINB, TS, SL) \
  k_match_batch_warp2<MINB, TS, SL><<<grid2, MW2_WARPS * 32, 0, st>>>(frames, width, height, stride, templates, fpf, h, S, sigma_size, thr, clampv, out_uv, out_score, total)
    switch (var) {
      case 0: MW2_LAUNCH(2, false, false); break;
      case 2: MW2_LAUNCH(3, true, false); break;
      case 4: MW2_LAUNCH(2, false, true); break;
      case 5: MW2_LAUNCH(2, true, true); break;
      case 6: MW2_LAUNCH(3, true, true); break;
      default: MW2_LAUNCH(2, true, false); break;   // 1
    }
#undef MW2_LAUNCH
    int dev = 0, sms = 148, per_sm = 4;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_match_batch_marked, MATCH_THREADS, smem) != cudaSuccess || per_sm < 1) {
      cudaGetLastError();
      per_sm = 4;
    }
    const int grid = total < sms * per_sm ? total : sms * per_sm;
    k_match_batch_marked<<<grid, MATCH_THREADS, smem, st>>>(frames, width, height, stride, templates, fpf, w, h, S, sigma_size, thr,
                                                           clampv, out_uv, out_score, total, as_cu(tm), tm.ok);
    return 0;
  }
  k_match_batch<<<total, MATCH_THREADS, smem, st>>>(frames, width, height, stride, templates, fpf, w, h, S, sigma_size, thr,
                                                   clampv, out_uv, out_score, total, as_cu(tm), tm.ok);
  return 0;
}
