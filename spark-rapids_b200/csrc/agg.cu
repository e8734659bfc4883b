// agg.cu — a3/a4/a5: reductions and hash group-by, fused with the child filter and the pre-step
// projection (one kernel: predicate -> project -> aggregate).
//
// Reference: AggHelper.performReduction / performGroupByAggregation (GpuAggregateExec.scala:540-585),
// GpuAggFirstPassIterator (:730-742), CudfSum/Count/Min/Max (aggregateFunctions.scala:38-68),
// GpuDecimalSum / GpuDecimal128Sum / GpuExtractChunk32 / GpuAssembleSumChunks (:607-700, 1106-1290).
//
// The reference expands a DECIMAL128 sum into four 32-bit chunk sums plus isEmpty/overflow columns
// (~30 cudf aggregations for TPC-H q1) because cudf cannot sum 128-bit values with overflow
// detection.  Here every decimal sum is accumulated exactly in a 128- or 192-bit two's-complement
// accumulator (64-bit limbs + carry), which is observably identical: the exact sum, NULL when it
// does not fit the result precision, NULL for an empty / all-null group.
//
// Two regimes, one accumulate routine:
//   * shared-memory table per CTA (<= SMEM_SLOTS groups): rows of a warp that hit the same group
//     are combined with __match_any_sync + REDUX (__reduce_add_sync on 16-bit pieces) so only one
//     lane per group per warp touches the accumulator; CTAs merge into the global table once.
//   * global open-addressing table (any cardinality): insert by CAS on a representative row index,
//     key equality against that row, RED/ATOM on per-slot accumulators.
#include "prim.cuh"
#include "rowops.cuh"
#include "vm.cuh"

namespace b2 {

constexpr int AG_MAX_AGGS = 24;
constexpr int SMEM_SLOTS_MAX = 2048;  // groups per CTA table (power of two, sized per plan)
constexpr uint32_t KEY_READY = 0x80000000u;
constexpr int32_t SLOT_EMPTY = -1;

struct AggD {
  int32_t kind;      // b2_agg_kind
  int32_t out_idx;   // program output feeding this aggregate (-1: none)
  int32_t in_mt;     // machine type of the input
  int32_t nlimbs;    // 64-bit limbs of the accumulator
  int32_t limb_off;  // first limb inside the slot's accumulator block
  int32_t track_valid;  // count valid inputs (nullable input or keyless reduction)
  int32_t valid_off;
  int32_t is_float;
};
struct AggPlan {
  int32_t nkeys, naggs, limbs, nvalids, has_pred;
  int32_t smem_slots;   // slots of the per-CTA table (power of two)
  int32_t fast_keys;    // all keys fixed width, <= 8 bytes together: packed copy kept in the slot
  KeyCols keys;
  AggD aggs[AG_MAX_AGGS];
};
struct GTable {
  int32_t* slots;     // representative row per slot, SLOT_EMPTY when free
  uint64_t* acc;      // [cap][limbs]
  uint32_t* nvalid;   // [cap][nvalids]
  uint32_t mask;      // cap - 1
  int32_t* overflow;  // set when a shared-memory table filled up
  uint64_t* keys;     // fast keys: packed key per slot
  uint32_t* knull;    // fast keys: null mask | KEY_READY once keys[slot] is visible
};

// order-preserving maps to u64 for MIN/MAX (Spark float order: NaN greatest, aggregateFunctions.scala:368-465)
__device__ __forceinline__ uint64_t ord_i64(int64_t v) { return (uint64_t)v ^ 0x8000000000000000ull; }
__device__ __forceinline__ uint64_t ord_f64(double d) {
  if (d != d) return 0xffffffffffffffffull;
  if (d == 0.0) d = 0.0;
  uint64_t b = (uint64_t)__double_as_longlong(d);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ inline double unord_f64(uint64_t k) {
  if (k == 0xffffffffffffffffull) { uint64_t n = 0x7ff8000000000000ull; double d; memcpy(&d, &n, 8); return d; }
  uint64_t b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
  double d; memcpy(&d, &b, 8); return d;
}

__device__ __forceinline__ uint64_t init_limb(const AggD& a) {
  return a.kind == B2_AGG_MIN ? 0xffffffffffffffffull : 0ull;
}

// multi-limb two's-complement add with carry via 64-bit atomics (exact mod 2^(64*n), order free)
__device__ __forceinline__ void acc_add_limbs(uint64_t* acc, int nlimbs, uint64_t l0, uint64_t l1, uint64_t l2) {
  unsigned long long* a = reinterpret_cast<unsigned long long*>(acc);
  if (nlimbs == 1) { if (l0) atomicAdd(&a[0], (unsigned long long)l0); return; }
  if (l0 == 0 && l1 == 0 && l2 == 0) return;
  uint64_t old0 = atomicAdd(&a[0], (unsigned long long)l0);
  uint64_t c0 = (old0 + l0) < old0 ? 1 : 0;
  uint64_t s1 = l1 + c0;
  uint64_t c1a = s1 < l1 ? 1 : 0;
  if (nlimbs == 2) { if (s1) atomicAdd(&a[1], (unsigned long long)s1); return; }
  uint64_t old1 = atomicAdd(&a[1], (unsigned long long)s1);
  uint64_t c1 = c1a + ((old1 + s1) < old1 ? 1 : 0);
  uint64_t s2 = l2 + c1;
  if (s2) atomicAdd(&a[2], (unsigned long long)s2);
}

// Accumulate one warp-slice (32 rows) into per-slot accumulators.  Two regimes per slice:
//   few distinct groups in the warp (<= 4, e.g. TPC-H q1): for each group the members' values are
//     summed with full-mask REDUX (hardware) on 16-bit pieces and ONE lane updates the accumulator;
//   many distinct groups: every lane updates its own slot (little contention by construction).
// (A REDUX over an arbitrary lane subset is a software loop on this architecture: 20% of the
//  kernel's stall samples in profiles/r1_agg_keyed_ncu_summary.txt before this split.)
__device__ __forceinline__ u128 warp_sum_u64(uint64_t x) {
  const uint32_t s0 = __reduce_add_sync(0xffffffffu, (uint32_t)(x & 0xffff));
  const uint32_t s1 = __reduce_add_sync(0xffffffffu, (uint32_t)((x >> 16) & 0xffff));
  const uint32_t s2 = __reduce_add_sync(0xffffffffu, (uint32_t)((x >> 32) & 0xffff));
  const uint32_t s3 = __reduce_add_sync(0xffffffffu, (uint32_t)((x >> 48) & 0xffff));
  return (u128)s0 + ((u128)s1 << 16) + ((u128)s2 << 32) + ((u128)s3 << 48);
}

__device__ __forceinline__ void accumulate_slice(const AggPlan& plan, const VMCtx& cx, int i, int64_t g,
                                                 bool active, int32_t slot, uint64_t* acc_base, uint32_t* nv_base) {
  const int lane = threadIdx.x & 31;
  const uint32_t m = __match_any_sync(0xffffffffu, slot);
  const bool leader = active && lane == (__ffs(m) - 1);
  const uint32_t leaders = __ballot_sync(0xffffffffu, leader);
  const bool few = __popc(leaders) <= 4;
  uint64_t* acc = active ? acc_base + (int64_t)slot * plan.limbs : nullptr;
  uint32_t* nvalid = active ? nv_base + (int64_t)slot * plan.nvalids : nullptr;
  for (int k = 0; k < plan.naggs; k++) {
    const AggD& a = plan.aggs[k];
    bool valid = active;
    Opnd opk;
    if (a.out_idx >= 0) opk = resolve(cx, cx.hdr->outs[a.out_idx], mt_width(a.in_mt));
    if (a.out_idx >= 0 && active) valid = opnd_valid(opk, i, g);
    // value of this row as sign-extended (lo, hi) or as an ordered key / double
    uint64_t lo = 0, hi = 0;
    double dv = 0.0;
    if (valid && a.out_idx >= 0) {
      switch (a.in_mt) {
        case MT_I8: lo = (uint64_t)(int64_t)opnd_ld<int8_t>(opk, i); break;
        case MT_I16: lo = (uint64_t)(int64_t)opnd_ld<int16_t>(opk, i); break;
        case MT_I32: lo = (uint64_t)(int64_t)opnd_ld<int32_t>(opk, i); break;
        case MT_I64: lo = (uint64_t)opnd_ld<int64_t>(opk, i); break;
        case MT_I128: { const i128 v = opnd_ld<i128>(opk, i); lo = (uint64_t)v; hi = (uint64_t)(v >> 64); } break;
        case MT_F32: dv = (double)opnd_ld<float>(opk, i); break;
        default: dv = opnd_ld<double>(opk, i); break;
      }
      if (a.in_mt < MT_I128) hi = ((int64_t)lo < 0) ? ~0ull : 0ull;
    }
    const bool int_sum = a.kind == B2_AGG_SUM && !a.is_float;
    const bool counting = a.kind == B2_AGG_COUNT || a.kind == B2_AGG_COUNT_ALL;
    if (few && (int_sum || counting || a.track_valid)) {
      // one pass per distinct group of this slice
      uint32_t rem = leaders;
      while (rem) {
        const int L = __ffs(rem) - 1;
        rem &= rem - 1;
        const int32_t gs = __shfl_sync(0xffffffffu, slot, L);
        const bool mem = active && slot == gs;
        const uint32_t vc = __popc(__ballot_sync(0xffffffffu, mem && valid));
        if (a.track_valid && lane == L && vc) atomicAdd(&nvalid[a.valid_off], vc);
        if (counting) { if (lane == L && vc) atomicAdd(reinterpret_cast<unsigned long long*>(&acc[a.limb_off]), (unsigned long long)vc); }
        else if (int_sum) {
          const bool mv = mem && valid;
          const uint32_t nneg = __popc(__ballot_sync(0xffffffffu, mv && (int64_t)hi < 0));
          const u128 slo = warp_sum_u64(mv ? lo : 0);
          if (a.in_mt == MT_I128) {
            const u128 shi = warp_sum_u64(mv ? hi : 0);
            if (lane == L) {
              const u128 mid = (slo >> 64) + (u128)(uint64_t)shi;
              acc_add_limbs(&acc[a.limb_off], 3, (uint64_t)slo, (uint64_t)mid, (uint64_t)(mid >> 64) + (uint64_t)(shi >> 64) - (uint64_t)nneg);
            }
          } else if (lane == L) {
            acc_add_limbs(&acc[a.limb_off], a.nlimbs, (uint64_t)slo, (uint64_t)(slo >> 64) - (uint64_t)nneg, 0);
          }
        }
      }
    } else if (valid) {
      if (a.track_valid) atomicAdd(&nvalid[a.valid_off], 1u);
      if (counting) atomicAdd(reinterpret_cast<unsigned long long*>(&acc[a.limb_off]), 1ull);
      else if (int_sum) acc_add_limbs(&acc[a.limb_off], a.nlimbs, lo, hi, (int64_t)hi < 0 ? ~0ull : 0ull);
    }
    if (!valid) continue;
    if (a.kind == B2_AGG_SUM && a.is_float) atomicAdd(reinterpret_cast<double*>(&acc[a.limb_off]), dv);
    else if (a.kind == B2_AGG_MIN || a.kind == B2_AGG_MAX) {
      const uint64_t key = a.is_float ? ord_f64(dv) : ord_i64((int64_t)lo);
      unsigned long long* p = reinterpret_cast<unsigned long long*>(&acc[a.limb_off]);
      if (a.kind == B2_AGG_MIN) atomicMin(p, (unsigned long long)key); else atomicMax(p, (unsigned long long)key);
    }
  }
}

// Keyless reduction: every thread folds its own rows into private shared-memory accumulators
// (no atomics, no warp collectives); the CTA combines them once at the end.
__device__ __forceinline__ void accumulate_private(const AggPlan& plan, const VMCtx& cx, uint32_t active_mask, uint64_t* priv, uint32_t* privv) {
  const int K = cx.K;
  for (int k = 0; k < plan.naggs; k++) {
    const AggD& a = plan.aggs[k];
    Opnd op;
    if (a.out_idx >= 0) op = resolve(cx, cx.hdr->outs[a.out_idx], mt_width(a.in_mt));
    uint64_t* p0 = &priv[a.limb_off * VM_NT + threadIdx.x];
    uint32_t nvalid = 0;
    uint64_t l0 = p0[0], l1 = a.nlimbs > 1 ? p0[VM_NT] : 0, l2 = a.nlimbs > 2 ? p0[2 * VM_NT] : 0;
    for (int j = 0; j < K; j++) {
      if (!((active_mask >> j) & 1u)) continue;
      const int i = threadIdx.x + j * VM_NT;
      const int64_t g = cx.tile_base + i;
      if (a.out_idx >= 0 && !opnd_valid(op, i, g)) continue;
      nvalid++;
      switch (a.kind) {
        case B2_AGG_COUNT: case B2_AGG_COUNT_ALL: l0 += 1; break;
        case B2_AGG_SUM: {
          if (a.is_float) {
            const double v = a.in_mt == MT_F32 ? (double)opnd_ld<float>(op, i) : opnd_ld<double>(op, i);
            l0 = (uint64_t)__double_as_longlong(__longlong_as_double((long long)l0) + v);
            break;
          }
          uint64_t lo, hi;
          switch (a.in_mt) {
            case MT_I8: lo = (uint64_t)(int64_t)opnd_ld<int8_t>(op, i); hi = (int64_t)lo < 0 ? ~0ull : 0; break;
            case MT_I16: lo = (uint64_t)(int64_t)opnd_ld<int16_t>(op, i); hi = (int64_t)lo < 0 ? ~0ull : 0; break;
            case MT_I32: lo = (uint64_t)(int64_t)opnd_ld<int32_t>(op, i); hi = (int64_t)lo < 0 ? ~0ull : 0; break;
            case MT_I64: lo = (uint64_t)opnd_ld<int64_t>(op, i); hi = (int64_t)lo < 0 ? ~0ull : 0; break;
            default: { const i128 v = opnd_ld<i128>(op, i); lo = (uint64_t)v; hi = (uint64_t)(v >> 64); } break;
          }
          const uint64_t s0 = l0 + lo;
          const uint64_t c0 = s0 < l0;
          l0 = s0;
          if (a.nlimbs > 1) {
            const uint64_t t1 = l1 + hi, c1a = t1 < l1;
            const uint64_t s1 = t1 + c0, c1b = s1 < t1;
            l1 = s1;
            if (a.nlimbs > 2) l2 += ((int64_t)hi < 0 ? ~0ull : 0ull) + c1a + c1b;
          }
        } break;
        case B2_AGG_MIN: case B2_AGG_MAX: {
          uint64_t key;
          switch (a.in_mt) {
            case MT_I8: key = ord_i64(opnd_ld<int8_t>(op, i)); break;
            case MT_I16: key = ord_i64(opnd_ld<int16_t>(op, i)); break;
            case MT_I32: key = ord_i64(opnd_ld<int32_t>(op, i)); break;
            case MT_I64: key = ord_i64(opnd_ld<int64_t>(op, i)); break;
            case MT_F32: key = ord_f64((double)opnd_ld<float>(op, i)); break;
            default: key = ord_f64(opnd_ld<double>(op, i)); break;
          }
          l0 = a.kind == B2_AGG_MIN ? (key < l0 ? key : l0) : (key > l0 ? key : l0);
        } break;
        default: break;
      }
    }
    p0[0] = l0;
    if (a.nlimbs > 1) p0[VM_NT] = l1;
    if (a.nlimbs > 2) p0[2 * VM_NT] = l2;
    if (a.track_valid && nvalid) privv[a.valid_off * VM_NT + threadIdx.x] += nvalid;
  }
}

// keys that fit 8 bytes together — fixed-width columns and SHORT strings (1 length byte + chars) —
// identify the group exactly as (packed bits, null mask).  Returns false for a row whose string is
// too long for its budget: that row takes the generic compare path.
__device__ __forceinline__ bool pack_keys(const KeyCols& ks, int64_t r, uint64_t& bits, uint32_t& nulls) {
  bits = 0; nulls = 0;
  int shift = 0;
  for (int i = 0; i < ks.n; i++) {
    const KeyCol& k = ks.c[i];
    if (!row_valid(k.valid, r)) nulls |= 1u << i;
    else if (k.dtype == B2_STRING) {
      const int32_t b = k.offsets[r], len = k.offsets[r + 1] - b;
      if (len > k.pack - 1) return false;
      uint64_t v = (uint64_t)(len + 1);
      const uint8_t* p = reinterpret_cast<const uint8_t*>(k.data) + b;
      for (int q = 0; q < len; q++) v |= (uint64_t)p[q] << (8 * (q + 1));
      bits |= v << shift;
    } else bits |= key_bits(k, r) << shift;
    shift += 8 * k.pack;
  }
  return true;
}

// find-or-insert row `row` in the global table; returns the slot
__device__ __forceinline__ uint32_t global_insert(const GTable& gt, const KeyCols& keys, int64_t row, bool fast) {
  if (keys.n == 0) { gt.slots[0] = 0; return 0; }
  if (fast) {
    uint64_t kb; uint32_t kn;
    const bool packed = pack_keys(keys, row, kb, kn);
    uint32_t idx = (packed ? (uint32_t)mix64(kb ^ ((uint64_t)kn << 56) ^ 0x9e3779b97f4a7c15ull) : row_hash(keys, row)) & gt.mask;
    while (true) {
      int32_t cur = gt.slots[idx];
      if (cur == SLOT_EMPTY) {
        const int32_t old = atomicCAS(&gt.slots[idx], SLOT_EMPTY, (int32_t)row);
        if (old == SLOT_EMPTY) {
          if (packed) {
            gt.keys[idx] = kb;
            __threadfence();
            *reinterpret_cast<volatile uint32_t*>(&gt.knull[idx]) = kn | KEY_READY;
          }
          return idx;
        }
        cur = old;
      }
      const uint32_t tag = *reinterpret_cast<volatile uint32_t*>(&gt.knull[idx]);
      bool same;
      if (packed && (tag & KEY_READY)) { __threadfence(); same = (tag & ~KEY_READY) == kn && *reinterpret_cast<volatile uint64_t*>(&gt.keys[idx]) == kb; }
      else same = cur == (int32_t)row || rows_equal(keys, row, keys, cur, true);
      if (same) return idx;
      idx = (idx + 1) & gt.mask;
    }
  }
  uint32_t idx = row_hash(keys, row) & gt.mask;
  while (true) {
    int32_t cur = gt.slots[idx];
    if (cur == SLOT_EMPTY) {
      int32_t old = atomicCAS(&gt.slots[idx], SLOT_EMPTY, (int32_t)row);
      if (old == SLOT_EMPTY) return idx;
      cur = old;
    }
    if (cur == (int32_t)row || rows_equal(keys, row, keys, cur, true)) return idx;
    idx = (idx + 1) & gt.mask;
  }
}

__global__ void init_table_kernel(GTable gt, const __grid_constant__ AggPlan plan, int64_t cap) {
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < cap; s += (int64_t)gridDim.x * blockDim.x) {
    gt.slots[s] = SLOT_EMPTY;
    if (gt.knull) gt.knull[s] = 0;
    for (int k = 0; k < plan.naggs; k++)
      for (int l = 0; l < plan.aggs[k].nlimbs; l++) gt.acc[s * plan.limbs + plan.aggs[k].limb_off + l] = init_limb(plan.aggs[k]);
    for (int v = 0; v < plan.nvalids; v++) gt.nvalid[s * plan.nvalids + v] = 0;
  }
}

// Group-sorted tile, blocked: thread t owns C consecutive sorted positions, so it sees one group (two at
// a boundary).  It folds its rows into a private 192-bit partial per aggregate (plain adds, no collectives);
// when the whole warp ended on the same group the 32 partials are combined with 12 REDUX and ONE lane
// touches the table, otherwise each lane flushes its own run.
struct AggPart { uint64_t l0, l1, l2, mm; double d; uint32_t cnt; };
__device__ __forceinline__ void part_reset(AggPart& p, const AggD& a) { p.l0 = p.l1 = p.l2 = 0; p.cnt = 0; p.d = 0.0; p.mm = init_limb(a); }
__device__ __forceinline__ void part_flush(const AggPlan& plan, const AggD& a, const AggPart& p, int32_t slot, uint64_t* s_acc, uint32_t* s_nvalid) {
  if (slot < 0 || p.cnt == 0) return;
  uint64_t* acc = s_acc + (int64_t)slot * plan.limbs + a.limb_off;
  if (a.track_valid) atomicAdd(&s_nvalid[(int64_t)slot * plan.nvalids + a.valid_off], p.cnt);
  if (a.kind == B2_AGG_COUNT || a.kind == B2_AGG_COUNT_ALL) atomicAdd(reinterpret_cast<unsigned long long*>(acc), (unsigned long long)p.cnt);
  else if (a.kind == B2_AGG_SUM && a.is_float) atomicAdd(reinterpret_cast<double*>(acc), p.d);
  else if (a.kind == B2_AGG_SUM) acc_add_limbs(acc, a.nlimbs, p.l0, p.l1, p.l2);
  else if (a.kind == B2_AGG_MIN) atomicMin(reinterpret_cast<unsigned long long*>(acc), (unsigned long long)p.mm);
  else if (a.kind == B2_AGG_MAX) atomicMax(reinterpret_cast<unsigned long long*>(acc), (unsigned long long)p.mm);
}
__device__ __forceinline__ void accumulate_sorted(const AggPlan& plan, const VMCtx& cx, const uint16_t* s_perm, const uint16_t* s_rowslot, int total,
                                                  uint64_t* s_acc, uint32_t* s_nvalid) {
  const int C = (total + VM_NT - 1) / VM_NT;
  const int p0 = threadIdx.x * C, p1 = min(p0 + C, total);
  const int lane = threadIdx.x & 31;
  for (int k = 0; k < plan.naggs; k++) {
    const AggD& a = plan.aggs[k];
    Opnd op;
    if (a.out_idx >= 0) op = resolve(cx, cx.hdr->outs[a.out_idx], mt_width(a.in_mt));
    AggPart part; part_reset(part, a);
    int32_t run = -1;
    for (int p = p0; p < p1; p++) {
      const int i = s_perm[p];
      const int32_t slot = (int32_t)s_rowslot[i];
      if (slot != run) { part_flush(plan, a, part, run, s_acc, s_nvalid); part_reset(part, a); run = slot; }
      const int64_t g = cx.tile_base + i;
      if (a.out_idx >= 0 && !opnd_valid(op, i, g)) continue;
      part.cnt++;
      if (a.kind == B2_AGG_SUM && !a.is_float) {
        uint64_t lo, hi;
        switch (a.in_mt) {
          case MT_I8: lo = (uint64_t)(int64_t)opnd_ld<int8_t>(op, i); hi = (int64_t)lo < 0 ? ~0ull : 0; break;
          case MT_I16: lo = (uint64_t)(int64_t)opnd_ld<int16_t>(op, i); hi = (int64_t)lo < 0 ? ~0ull : 0; break;
          case MT_I32: lo = (uint64_t)(int64_t)opnd_ld<int32_t>(op, i); hi = (int64_t)lo < 0 ? ~0ull : 0; break;
          case MT_I64: lo = (uint64_t)opnd_ld<int64_t>(op, i); hi = (int64_t)lo < 0 ? ~0ull : 0; break;
          default: { const i128 v = opnd_ld<i128>(op, i); lo = (uint64_t)v; hi = (uint64_t)(v >> 64); } break;
        }
        const uint64_t s0 = part.l0 + lo, c0 = s0 < part.l0;
        const uint64_t t1 = part.l1 + hi, c1a = t1 < part.l1;
        const uint64_t s1 = t1 + c0, c1b = s1 < t1;
        part.l0 = s0; part.l1 = s1; part.l2 += ((int64_t)hi < 0 ? ~0ull : 0ull) + c1a + c1b;
      } else if (a.kind == B2_AGG_SUM) {
        part.d += a.in_mt == MT_F32 ? (double)opnd_ld<float>(op, i) : opnd_ld<double>(op, i);
      } else if (a.kind == B2_AGG_MIN || a.kind == B2_AGG_MAX) {
        uint64_t key;
        switch (a.in_mt) {
          case MT_I8: key = ord_i64(opnd_ld<int8_t>(op, i)); break;
          case MT_I16: key = ord_i64(opnd_ld<int16_t>(op, i)); break;
          case MT_I32: key = ord_i64(opnd_ld<int32_t>(op, i)); break;
          case MT_I64: key = ord_i64(opnd_ld<int64_t>(op, i)); break;
          case MT_F32: key = ord_f64((double)opnd_ld<float>(op, i)); break;
          default: key = ord_f64(opnd_ld<double>(op, i)); break;
        }
        part.mm = a.kind == B2_AGG_MIN ? (key < part.mm ? key : part.mm) : (key > part.mm ? key : part.mm);
      }
    }
    // last run of every lane: one combined update when the warp agrees on the group
    const int32_t wslot = __reduce_max_sync(0xffffffffu, run);
    const bool uniform = __ballot_sync(0xffffffffu, run != wslot && run != -1) == 0;
    const bool int_sum = a.kind == B2_AGG_SUM && !a.is_float;
    if (uniform && wslot >= 0 && (int_sum || a.kind == B2_AGG_COUNT || a.kind == B2_AGG_COUNT_ALL)) {
      const uint32_t cnt = __reduce_add_sync(0xffffffffu, part.cnt);
      AggPart w; part_reset(w, a); w.cnt = cnt;
      if (int_sum) {
        const u128 S0 = warp_sum_u64(part.l0), S1 = warp_sum_u64(part.l1);
        const uint64_t S2 = (uint64_t)warp_sum_u64(part.l2);
        const u128 mid = (S0 >> 64) + (u128)(uint64_t)S1;
        w.l0 = (uint64_t)S0; w.l1 = (uint64_t)mid; w.l2 = (uint64_t)(mid >> 64) + (uint64_t)(S1 >> 64) + S2;
      }
      if (lane == 0) part_flush(plan, a, w, wslot, s_acc, s_nvalid);
    } else {
      part_flush(plan, a, part, run, s_acc, s_nvalid);
    }
  }
}

// find-or-insert row g in the CTA's shared-memory table; -1 when the table is too full (overflow flagged)
__device__ __forceinline__ int32_t smem_find_slot(const AggPlan& plan, int64_t g, int32_t* s_slots, uint64_t* s_keys, uint32_t* s_knull, int SLOTS,
                                                  int32_t* overflow, uint32_t* s_nocc) {
  uint64_t kb = 0; uint32_t kn = 0;
  const bool packed = plan.fast_keys && pack_keys(plan.keys, g, kb, kn);
  uint32_t idx = (packed ? (uint32_t)mix64(kb ^ ((uint64_t)kn << 56) ^ 0x9e3779b97f4a7c15ull) : row_hash(plan.keys, g)) & (SLOTS - 1);
  int probes = 0;
  // a table this full is abandoned at once: walking long probe chains (row compares through global memory for unpacked
  // keys) only to overflow a few rows later made the 256 K-row cardinality probe of TPC-H q3 cost 1.8 ms
  if (*reinterpret_cast<volatile uint32_t*>(s_nocc) > (uint32_t)(SLOTS - SLOTS / 8)) { atomicExch(overflow, 1); return -1; }
  while (true) {
    int32_t cur = s_slots[idx];
    if (cur == SLOT_EMPTY) {
      const int32_t old = atomicCAS(&s_slots[idx], SLOT_EMPTY, (int32_t)g);
      if (old == SLOT_EMPTY) {  // mine: publish the packed key for later probes (key, fence, then the READY flag: a reader
                                // that does not see the flag yet compares the rows themselves; racecheck reports this
                                // flag+fence hand-off as a hazard pair, see profiles/r1_racecheck.txt)
        if (packed) {
          s_keys[idx] = kb;
          __threadfence_block();
          *reinterpret_cast<volatile uint32_t*>(&s_knull[idx]) = kn | KEY_READY;
        }
        atomicAdd(s_nocc, 1u);
        return (int32_t)idx;
      }
      cur = old;
    }
    bool same;
    const uint32_t tag = plan.fast_keys ? *reinterpret_cast<volatile uint32_t*>(&s_knull[idx]) : 0u;
    if (packed && (tag & KEY_READY)) { __threadfence_block(); same = (tag & ~KEY_READY) == kn && *reinterpret_cast<volatile uint64_t*>(&s_keys[idx]) == kb; }
    else same = cur == (int32_t)g || rows_equal(plan.keys, g, plan.keys, cur, true);  // generic compare / key not published yet
    if (same) return (int32_t)idx;
    idx = (idx + 1) & (SLOTS - 1);
    if (++probes >= SLOTS / 2) { atomicExch(overflow, 1); return -1; }
  }
}

// SMEM = true: per-CTA shared table + merge; false: straight to the global table
template <bool SMEM>
__global__ void __launch_bounds__(VM_NT, 4) aggregate_kernel(const VMProgramHeader* __restrict__ g_hdr, const VMInstr* __restrict__ g_code,
                                                          const __grid_constant__ VMInputs in, const __grid_constant__ AggPlan plan,
                                                          GTable gt, int64_t nrows, int smem_regs_bytes) {
  __shared__ VMShared sh;
  extern __shared__ __align__(16) char dyn[];
  char* regs = dyn;
  // shared table lives after the VM registers
  int32_t* s_slots = reinterpret_cast<int32_t*>(dyn + smem_regs_bytes);
  const int SLOTS = plan.smem_slots;
  uint64_t* s_acc = reinterpret_cast<uint64_t*>(dyn + smem_regs_bytes + SLOTS * 4);
  uint32_t* s_nvalid = reinterpret_cast<uint32_t*>(s_acc + (SMEM ? SLOTS * plan.limbs : 0));
  // keyless reductions: one private accumulator set per thread, [limb][thread] / [valid][thread]
  // after the table: keyless private accumulators, or the packed keys of the slots (fast keys)
  uint64_t* s_priv = reinterpret_cast<uint64_t*>(s_nvalid + SLOTS * plan.nvalids + (SLOTS * plan.nvalids & 1));
  uint32_t* s_privv = reinterpret_cast<uint32_t*>(s_priv + plan.limbs * VM_NT);
  uint64_t* s_keys = s_priv;                                             // [SLOTS]
  uint32_t* s_knull = reinterpret_cast<uint32_t*>(s_keys + SLOTS);       // [SLOTS], KEY_READY once s_keys is valid
  const bool keyless = SMEM && plan.nkeys == 0;
  // keyed: sort area after the packed keys: counts/offsets per slot, slot per row, permutation, scalars
  uint32_t* s_cnt = s_knull + SLOTS;
  uint32_t* s_total = s_cnt + SLOTS;
  uint32_t* s_nocc = s_total + 1;
  uint16_t* s_rowslot = reinterpret_cast<uint16_t*>(s_nocc + 1);
  const RInstr* code = vm_load_program(sh, g_hdr, g_code, in, regs);
  uint16_t* s_perm = s_rowslot + sh.hdr.tile_rows;
  if (SMEM && threadIdx.x == 0 && !keyless) *s_nocc = 0;
  const int lane = threadIdx.x & 31;
  // a keyless reduction always has its single group, even over zero rows (GpuAggregateExec.scala:1107-1126)
  if (plan.nkeys == 0 && blockIdx.x == 0 && threadIdx.x == 0) gt.slots[0] = 0;
  if (SMEM) {
    for (int s = threadIdx.x; s < SLOTS; s += VM_NT) {
      s_slots[s] = SLOT_EMPTY;
      if (plan.fast_keys && plan.nkeys > 0) s_knull[s] = 0;
      for (int k = 0; k < plan.naggs; k++)
        for (int l = 0; l < plan.aggs[k].nlimbs; l++) s_acc[s * plan.limbs + plan.aggs[k].limb_off + l] = init_limb(plan.aggs[k]);
      for (int v = 0; v < plan.nvalids; v++) s_nvalid[s * plan.nvalids + v] = 0;
    }
    if (keyless) {
      for (int k = 0; k < plan.naggs; k++)
        for (int l = 0; l < plan.aggs[k].nlimbs; l++) s_priv[(plan.aggs[k].limb_off + l) * VM_NT + threadIdx.x] = init_limb(plan.aggs[k]);
      for (int v = 0; v < plan.nvalids; v++) s_privv[v * VM_NT + threadIdx.x] = 0;
    }
    __syncthreads();
  }
  const int64_t ntiles = (nrows + sh.hdr.tile_rows - 1) / sh.hdr.tile_rows;
  const int first_post = plan.has_pred ? sh.hdr.npred : 0;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    if (SMEM && *reinterpret_cast<volatile int32_t*>(gt.overflow)) break;  // someone overflowed: the launch is void
    VMCtx cx = vm_ctx(&sh.hdr, &in, regs, tile, nrows);
    uint32_t active_mask = 0;
    if (plan.has_pred) {
      // predicate first; the projection only runs for rows that survive it (per-thread row mask)
      vm_run(tile_info(cx), code, 0, first_post);
      const Opnd pred = resolve(cx, sh.hdr.outs[0], 1);
      for (int j = 0; j < cx.K; j++) {
        const int i = threadIdx.x + j * VM_NT;
        const int64_t g = cx.tile_base + i;
        const bool a = g < nrows && opnd_valid(pred, i, g) && opnd_ld<int8_t>(pred, i) != 0;
        active_mask |= (uint32_t)a << j;
      }
      // the row mask only pays off when few rows survive: every VM op is side-effect free, so when most
      // rows pass the projection runs unmasked (fast row loops) and the filtered rows are simply not aggregated
      const int passed = __syncthreads_count(active_mask != 0) ;
      cx.rowmask = (passed * 4 > VM_NT) ? 0xffffffffu : active_mask;
    } else {
      for (int j = 0; j < cx.K; j++) active_mask |= (uint32_t)(cx.tile_base + threadIdx.x + j * VM_NT < nrows) << j;
    }
    vm_run(tile_info(cx), code, first_post, sh.hdr.ninstr);
    if (keyless) {
      accumulate_private(plan, cx, active_mask, s_priv, s_privv);
      continue;
    }
    if (SMEM) {
      // group-sorted tile: when the CTA has seen few groups relative to the tile, rows are counting-sorted
      // by slot in shared memory so that a warp slice holds one or two groups instead of a random mix —
      // the per-(group, aggregate) REDUX work then drops by the number of groups per slice
      const int T = cx.tile_rows;
      if ((int)(*s_nocc) * 16 <= T) {
        for (int k = threadIdx.x; k < SLOTS; k += VM_NT) s_cnt[k] = 0;
        __syncthreads();
        for (int j = 0; j < cx.K; j++) {
          const int i = threadIdx.x + j * VM_NT;
          int32_t slot = -1;
          if ((active_mask >> j) & 1u) slot = smem_find_slot(plan, cx.tile_base + i, s_slots, s_keys, s_knull, SLOTS, gt.overflow, s_nocc);
          s_rowslot[i] = (uint16_t)(slot < 0 ? 0xffff : slot);
          if (slot >= 0) atomicAdd(&s_cnt[slot], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 32) {  // exclusive scan of the slot counts, SLOTS/32 consecutive slots per lane
          const int per = SLOTS / 32;
          uint32_t sum = 0;
          for (int k = 0; k < per; k++) sum += s_cnt[lane * per + k];
          uint32_t inc = sum;
          for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
          uint32_t run = inc - sum;
          for (int k = 0; k < per; k++) { const uint32_t c = s_cnt[lane * per + k]; s_cnt[lane * per + k] = run; run += c; }
          if (lane == 31) *s_total = inc;
        }
        __syncthreads();
        for (int j = 0; j < cx.K; j++) {
          const int i = threadIdx.x + j * VM_NT;
          const uint32_t sl = s_rowslot[i];
          if (sl != 0xffff) s_perm[atomicAdd(&s_cnt[sl], 1u)] = (uint16_t)i;
        }
        __syncthreads();
        accumulate_sorted(plan, cx, s_perm, s_rowslot, (int)*s_total, s_acc, s_nvalid);
        __syncthreads();
        continue;
      }
    }
#pragma unroll 1
    for (int j = 0; j < cx.K; j++) {
      const int i = threadIdx.x + j * VM_NT;
      const int64_t g = cx.tile_base + i;
      bool active = (active_mask >> j) & 1u;
      if (__ballot_sync(0xffffffffu, active) == 0) continue;  // nothing selected in these 32 rows
      int32_t slot = -1;
      if (active) {
        if (SMEM) slot = smem_find_slot(plan, g, s_slots, s_keys, s_knull, SLOTS, gt.overflow, s_nocc);
        else slot = (int32_t)global_insert(gt, plan.keys, g, plan.fast_keys != 0);
        if (slot < 0) active = false;
      }
      accumulate_slice(plan, cx, i, g, active && slot >= 0, active ? slot : -1, SMEM ? s_acc : gt.acc, SMEM ? s_nvalid : gt.nvalid);
    }
  }
  if (keyless) {
    s_slots[0] = 0;
    __syncthreads();
    for (int k = 0; k < plan.naggs; k++) {
      const AggD& a = plan.aggs[k];
      unsigned long long* p = reinterpret_cast<unsigned long long*>(&s_acc[a.limb_off]);
      const uint64_t l0 = s_priv[a.limb_off * VM_NT + threadIdx.x];
      if (a.kind == B2_AGG_MIN) atomicMin(p, (unsigned long long)l0);
      else if (a.kind == B2_AGG_MAX) atomicMax(p, (unsigned long long)l0);
      else if (a.is_float) atomicAdd(reinterpret_cast<double*>(p), __longlong_as_double((long long)l0));
      else acc_add_limbs(&s_acc[a.limb_off], a.nlimbs, l0, a.nlimbs > 1 ? s_priv[(a.limb_off + 1) * VM_NT + threadIdx.x] : 0,
                         a.nlimbs > 2 ? s_priv[(a.limb_off + 2) * VM_NT + threadIdx.x] : 0);
    }
    for (int v = 0; v < plan.nvalids; v++)
      if (s_privv[v * VM_NT + threadIdx.x]) atomicAdd(&s_nvalid[v], s_privv[v * VM_NT + threadIdx.x]);
  }
  if (SMEM) {
    __syncthreads();
    if (*reinterpret_cast<volatile int32_t*>(gt.overflow)) return;
    for (int s = threadIdx.x; s < SLOTS; s += VM_NT) {
      const int32_t row = s_slots[s];
      if (row == SLOT_EMPTY) continue;
      const uint32_t gs = global_insert(gt, plan.keys, row, plan.fast_keys != 0);
      uint64_t* ga = &gt.acc[(int64_t)gs * plan.limbs];
      const uint64_t* sa = &s_acc[s * plan.limbs];
      for (int k = 0; k < plan.naggs; k++) {
        const AggD& a = plan.aggs[k];
        unsigned long long* p = reinterpret_cast<unsigned long long*>(&ga[a.limb_off]);
        if (a.kind == B2_AGG_MIN) atomicMin(p, (unsigned long long)sa[a.limb_off]);
        else if (a.kind == B2_AGG_MAX) atomicMax(p, (unsigned long long)sa[a.limb_off]);
        else if (a.is_float) atomicAdd(reinterpret_cast<double*>(p), __longlong_as_double((long long)sa[a.limb_off]));
        else acc_add_limbs(&ga[a.limb_off], a.nlimbs, sa[a.limb_off], a.nlimbs > 1 ? sa[a.limb_off + 1] : 0, a.nlimbs > 2 ? sa[a.limb_off + 2] : 0);
      }
      for (int v = 0; v < plan.nvalids; v++)
        if (s_nvalid[s * plan.nvalids + v]) atomicAdd(&gt.nvalid[(int64_t)gs * plan.nvalids + v], s_nvalid[s * plan.nvalids + v]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
__global__ void occupied_flags_kernel(const int32_t* __restrict__ slots, int64_t cap, int32_t* __restrict__ flags) {
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < cap; s += (int64_t)gridDim.x * blockDim.x)
    flags[s] = slots[s] != SLOT_EMPTY;
}

struct AggOut {
  void* data[AG_MAX_AGGS];
  uint32_t* valid[AG_MAX_AGGS];  // zero-initialised
  int32_t out_dtype[AG_MAX_AGGS];
  int32_t out_precision[AG_MAX_AGGS];
};

__device__ __forceinline__ i128 pow10_128(int e) {
  i128 r = 1;
  for (int i = 0; i < e; i++) r *= 10;
  return r;
}

// finalise the accumulators of ONE group into row o of the output columns (shared by the hash-table and the radix paths)
__device__ __forceinline__ void finalize_group(const AggPlan& plan, const uint64_t* __restrict__ gacc, const uint32_t* __restrict__ gnvalid, int64_t o,
                                               const AggOut& out) {
  for (int k = 0; k < plan.naggs; k++) {
    const AggD& a = plan.aggs[k];
    const uint64_t* acc = &gacc[a.limb_off];
    bool valid = true;
    if (a.track_valid) valid = gnvalid[a.valid_off] > 0;
    switch (a.kind) {
      case B2_AGG_COUNT: case B2_AGG_COUNT_ALL:
        reinterpret_cast<int64_t*>(out.data[k])[o] = (int64_t)acc[0]; valid = true; break;
      case B2_AGG_SUM:
        if (a.is_float) {
          double d = __longlong_as_double((long long)acc[0]);
          if (out.out_dtype[k] == B2_FLOAT32) reinterpret_cast<float*>(out.data[k])[o] = (float)d;
          else reinterpret_cast<double*>(out.data[k])[o] = d;
        } else if (a.nlimbs == 1) {
          reinterpret_cast<int64_t*>(out.data[k])[o] = (int64_t)acc[0];  // long sum wraps (aggregateFunctions.scala:1041-1104)
        } else {
          // exact 128/192-bit sum -> decimal; NULL when it needs more than out_precision digits
          i128 v = (i128)(((u128)acc[1] << 64) | acc[0]);
          bool fits = true;
          if (a.nlimbs == 3) {
            const int64_t ext = (int64_t)acc[2];
            fits = (ext == 0 && (int64_t)acc[1] >= 0) || (ext == -1 && (int64_t)acc[1] < 0);
          }
          const i128 lim = pow10_128(out.out_precision[k]);
          if (!fits || v >= lim || v <= -lim) valid = false;
          if (out.out_dtype[k] == B2_DECIMAL128) reinterpret_cast<i128*>(out.data[k])[o] = valid ? v : (i128)0;
          else reinterpret_cast<int64_t*>(out.data[k])[o] = valid ? (int64_t)v : 0;
        }
        break;
      case B2_AGG_MIN: case B2_AGG_MAX: {
        const uint64_t key = acc[0];
        if (a.in_mt == MT_F32) reinterpret_cast<float*>(out.data[k])[o] = (float)unord_f64(key);
        else if (a.in_mt == MT_F64) reinterpret_cast<double*>(out.data[k])[o] = unord_f64(key);
        else {
          const int64_t v = (int64_t)(key ^ 0x8000000000000000ull);
          switch (a.in_mt) {
            case MT_I8: reinterpret_cast<int8_t*>(out.data[k])[o] = (int8_t)v; break;
            case MT_I16: reinterpret_cast<int16_t*>(out.data[k])[o] = (int16_t)v; break;
            case MT_I32: reinterpret_cast<int32_t*>(out.data[k])[o] = (int32_t)v; break;
            default: reinterpret_cast<int64_t*>(out.data[k])[o] = v; break;
          }
        }
      } break;
      default: break;
    }
    if (valid && out.valid[k]) atomicOr(&out.valid[k][o >> 5], 1u << (o & 31));
  }
}

__global__ void finalize_kernel(GTable gt, const __grid_constant__ AggPlan plan, int64_t cap, const int32_t* __restrict__ pos,
                                const __grid_constant__ AggOut out, int32_t* __restrict__ rep_rows) {
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < cap; s += (int64_t)gridDim.x * blockDim.x) {
    const int32_t row = gt.slots[s];
    if (row == SLOT_EMPTY) continue;
    const int32_t o = pos[s];
    rep_rows[o] = row;
    finalize_group(plan, &gt.acc[s * plan.limbs], &gt.nvalid[s * plan.nvalids], o, out);
  }
}

// A floating-point group key gathered from the group's representative row may be -0.0 or any NaN payload, whichever row won
// the slot; the group itself was formed on key_bits.  Writing key_bits back gives +0.0 and the canonical NaN, as Spark's
// NormalizeFloatingNumbers does before grouping and as the radix regime's packed keys already are.
__global__ void normalize_float_key_kernel(KeyCol k, int64_t n) {
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t b = key_bits(k, r);
    if (k.width == 4) reinterpret_cast<uint32_t*>(const_cast<void*>(k.data))[r] = (uint32_t)b;
    else reinterpret_cast<uint64_t*>(const_cast<void*>(k.data))[r] = b;
  }
}

// ================================================================================================================================
// Radix-partitioned group-by for high cardinalities (millions of groups: TPC-H q3's (l_orderkey, o_orderdate, o_shippriority)).
// The global open-addressing table of the regime above pays several random HBM accesses per row and is sized for the worst
// case (2 x rows slots).  Here the rows are first materialised (fused predicate + projection, keys packed into <= 16 bytes),
// then radix-partitioned by key hash (one or two stable passes of hash.cu's tile-histogram scatter) into partitions of
// ~1000 rows, and ONE persistent kernel aggregates each partition in a SHARED-MEMORY hash table: the partition's rows are
// streamed into shared memory by TMA bulk copies (cp.async.bulk + mbarrier, double buffered) while the previous chunk is
// being inserted; a finished partition's groups are appended to the compact group arrays and the table is reset.  No global
// hash table exists, every row moves through HBM a fixed number of times, all probing happens in shared memory.
// Reference it replaces: cudf hash groupby behind AggHelper.performGroupByAggregation (GpuAggregateExec.scala:562-585).
constexpr int RG_MAX_VALS = 5;
constexpr int RG_NT = 512;
constexpr int RG_CHUNK = 1024;        // rows per staged chunk (<= 4 x RG_NT: see `claimed` in radix_agg_kernel)
constexpr uint32_t RG_READY = 0x80000000u;
struct RGVal { int32_t out_idx, in_mt, width, pad; };
struct RGPlan {
  int32_t nvals, has_k1, use_vbits, pad;
  RGVal val[RG_MAX_VALS];
  int32_t agg_val[AG_MAX_AGGS];     // aggregate -> value slot, -1 for COUNT(*)
  int32_t key_shift[MAX_KEYS];      // bit offset of each key column inside the packed 128-bit key
};
struct RGRows {   // materialised rows, structure of arrays
  uint32_t* h; uint64_t* k0; uint64_t* k1; char* v[RG_MAX_VALS]; uint32_t* vbits;
};
__device__ __forceinline__ uint64_t rg_hash(uint64_t k0, uint64_t k1) { return mix64(k0 ^ mix64(k1 ^ 0x9e3779b97f4a7c15ull)); }

__global__ void __launch_bounds__(VM_NT, 4) radix_rows_kernel(const VMProgramHeader* __restrict__ g_hdr, const VMInstr* __restrict__ g_code,
                                                              const __grid_constant__ VMInputs in, const __grid_constant__ AggPlan plan,
                                                              const __grid_constant__ RGPlan rp, RGRows rows, int64_t nrows,
                                                              unsigned long long* __restrict__ counter) {
  __shared__ VMShared sh;
  extern __shared__ __align__(16) char regs[];
  const RInstr* code = vm_load_program(sh, g_hdr, g_code, in, regs);
  const int64_t ntiles = (nrows + sh.hdr.tile_rows - 1) / sh.hdr.tile_rows;
  const int first_post = plan.has_pred ? sh.hdr.npred : 0;
  const int lane = threadIdx.x & 31;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    VMCtx cx = vm_ctx(&sh.hdr, &in, regs, tile, nrows);
    uint32_t active_mask = 0;
    if (plan.has_pred) {
      vm_run(tile_info(cx), code, 0, first_post);
      const Opnd pred = resolve(cx, sh.hdr.outs[0], 1);
      for (int j = 0; j < cx.K; j++) {
        const int i = threadIdx.x + j * VM_NT;
        const int64_t g = cx.tile_base + i;
        active_mask |= (uint32_t)(g < nrows && opnd_valid(pred, i, g) && opnd_ld<int8_t>(pred, i) != 0) << j;
      }
    } else {
      for (int j = 0; j < cx.K; j++) active_mask |= (uint32_t)(cx.tile_base + threadIdx.x + j * VM_NT < nrows) << j;
    }
    vm_run(tile_info(cx), code, first_post, sh.hdr.ninstr);
    Opnd ops[RG_MAX_VALS];
    for (int s = 0; s < rp.nvals; s++) ops[s] = resolve(cx, sh.hdr.outs[rp.val[s].out_idx], mt_width(rp.val[s].in_mt));
    for (int j = 0; j < cx.K; j++) {
      const int i = threadIdx.x + j * VM_NT;
      const int64_t g = cx.tile_base + i;
      const bool active = (active_mask >> j) & 1u;
      const uint32_t b = __ballot_sync(0xffffffffu, active);
      if (b == 0) continue;
      int64_t pos = g;
      if (plan.has_pred) {   // compaction: order is irrelevant to an aggregation, one atomic per warp slice
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(counter, (unsigned long long)__popc(b));
        base = __shfl_sync(0xffffffffu, base, 0);
        pos = (int64_t)base + __popc(b & ((1u << lane) - 1u));
      }
      if (!active) continue;
      u128 bits = 0;
      for (int k = 0; k < plan.nkeys; k++) bits |= (u128)key_bits(plan.keys.c[k], g) << rp.key_shift[k];
      const uint64_t k0 = (uint64_t)bits, k1 = (uint64_t)(bits >> 64);
      rows.h[pos] = (uint32_t)(rg_hash(k0, k1) >> 32);
      rows.k0[pos] = k0;
      if (rp.has_k1) rows.k1[pos] = k1;
      uint32_t vb = 0;
      for (int s = 0; s < rp.nvals; s++) {
        const bool valid = opnd_valid(ops[s], i, g);
        vb |= (uint32_t)valid << s;
        if (rp.val[s].width == 16) {
          reinterpret_cast<i128*>(rows.v[s])[pos] = valid ? opnd_ld<i128>(ops[s], i) : (i128)0;
        } else {
          int64_t x = 0;
          if (valid) switch (rp.val[s].in_mt) {
            case MT_I8: x = opnd_ld<int8_t>(ops[s], i); break;
            case MT_I16: x = opnd_ld<int16_t>(ops[s], i); break;
            case MT_I32: x = opnd_ld<int32_t>(ops[s], i); break;
            default: x = opnd_ld<int64_t>(ops[s], i); break;
          }
          reinterpret_cast<int64_t*>(rows.v[s])[pos] = x;
        }
      }
      if (rp.use_vbits) rows.vbits[pos] = vb;
    }
  }
}

__global__ void rg_digit_kernel(const uint32_t* __restrict__ h, int64_t n, int shift, uint32_t mask, int32_t* __restrict__ pid) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) pid[i] = (int32_t)((h[i] >> shift) & mask);
}
// rows are sorted by q = h & (P - 1): off[q] = first row of partition q, off[P] = n
__global__ void rg_offsets_kernel(const uint32_t* __restrict__ h, int64_t n, uint32_t pmask, int32_t* __restrict__ off) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t q = h[i] & pmask, qp = i ? (int64_t)(h[i - 1] & pmask) : -1;
    for (int64_t x = qp + 1; x <= q; x++) off[x] = (int32_t)i;
    if (i == n - 1) for (int64_t x = q + 1; x <= (int64_t)pmask + 1; x++) off[x] = (int32_t)n;
  }
}

struct RGAgg {
  RGRows rows;
  const int32_t* off;
  int32_t P, C;
  int64_t m;
  uint64_t* gk0; uint64_t* gk1; uint64_t* gacc; uint32_t* gnvalid;
  unsigned long long* gcount;
  int32_t* overflow;
};

__global__ void __launch_bounds__(RG_NT, 1) radix_agg_kernel(const __grid_constant__ AggPlan plan, const __grid_constant__ RGPlan rp, const __grid_constant__ RGAgg a) {
  extern __shared__ __align__(128) char rg_dyn[];
  __shared__ __align__(8) uint64_t s_bar[2];
  __shared__ uint32_t s_nused[2];
  const int C = a.C;
  // table: packed keys, accumulators, state (0 = empty, else (claiming stage index + 1) [| RG_READY once the key is published])
  uint64_t* t_k0 = reinterpret_cast<uint64_t*>(rg_dyn);
  uint64_t* t_k1 = t_k0 + C;
  uint64_t* t_acc = t_k1 + (rp.has_k1 ? C : 0);
  uint32_t* t_state = reinterpret_cast<uint32_t*>(t_acc + (size_t)C * plan.limbs);
  uint32_t* t_nvalid = t_state + C;
  uint16_t* t_used = reinterpret_cast<uint16_t*>(t_nvalid + (size_t)C * plan.nvalids);   // log of the claimed slots
  char* stage0 = reinterpret_cast<char*>(((uintptr_t)(t_used + C) + 127) & ~(uintptr_t)127);
  // one stage buffer: k0 | k1 | v[0..] | vbits, each CH rows (+ slack so that 16-byte rounded copies stay inside)
  constexpr int CH = RG_CHUNK;
  int soff_k1 = CH * 8 + 16, soff_v[RG_MAX_VALS], soff_vb, sbytes;
  {
    int o = soff_k1 + (rp.has_k1 ? CH * 8 + 16 : 0);
    for (int s = 0; s < rp.nvals; s++) { soff_v[s] = o; o += CH * rp.val[s].width + 16; }
    soff_vb = o; o += rp.use_vbits ? CH * 4 + 16 : 0;
    sbytes = (o + 127) & ~127;
  }
  for (int s = threadIdx.x; s < C; s += RG_NT) {
    t_state[s] = 0;
    for (int k = 0; k < plan.naggs; k++)
      for (int l = 0; l < plan.aggs[k].nlimbs; l++) t_acc[(size_t)s * plan.limbs + plan.aggs[k].limb_off + l] = init_limb(plan.aggs[k]);
    for (int v = 0; v < plan.nvalids; v++) t_nvalid[(size_t)s * plan.nvalids + v] = 0;
  }
  // this CTA's partitions and the row stream that covers them (starts on a 4-row boundary: every array offset is 16-byte aligned)
  const int pA = (int)((int64_t)a.P * blockIdx.x / gridDim.x), pB = (int)((int64_t)a.P * (blockIdx.x + 1) / gridDim.x);
  const int64_t r_lo = a.off[pA], r_hi = a.off[pB];
  const int64_t a0 = r_lo & ~(int64_t)3;
  const int64_t nchunks = r_hi > r_lo ? (r_hi - a0 + CH - 1) / CH : 0;
  // the arrays a chunk is made of (base pointer, element width, offset inside a stage buffer): built once, so that the thread
  // that issues the TMA copies runs a short rolled loop (the inlined, unrolled form was ~600 instructions per chunk on the
  // critical path of warp 0)
  __shared__ const char* s_abase[RG_MAX_VALS + 3];
  __shared__ int s_awidth[RG_MAX_VALS + 3], s_aoff[RG_MAX_VALS + 3], s_narr;
  if (threadIdx.x == 0) {
    int k = 0;
    s_abase[k] = reinterpret_cast<const char*>(a.rows.k0); s_awidth[k] = 8; s_aoff[k] = 0; k++;
    if (rp.has_k1) { s_abase[k] = reinterpret_cast<const char*>(a.rows.k1); s_awidth[k] = 8; s_aoff[k] = soff_k1; k++; }
    for (int s = 0; s < rp.nvals; s++) { s_abase[k] = a.rows.v[s]; s_awidth[k] = rp.val[s].width; s_aoff[k] = soff_v[s]; k++; }
    if (rp.use_vbits) { s_abase[k] = reinterpret_cast<const char*>(a.rows.vbits); s_awidth[k] = 4; s_aoff[k] = soff_vb; k++; }
    s_narr = k;
  }
  __syncthreads();
  auto issue = [&](int64_t c, int buf) {   // one thread: TMA copies of chunk c into stage buffer buf
    const int64_t start = a0 + c * CH;
    const int64_t rows = min((int64_t)CH, a.m - start);
    char* sb = stage0 + (size_t)buf * sbytes;
    const int narr = s_narr;
    uint32_t total = 0;
#pragma unroll 1
    for (int k = 0; k < narr; k++) total += (uint32_t)((rows * s_awidth[k] + 15) & ~15LL);
    fence_proxy_async();
    mbar_expect_tx(&s_bar[buf], total);
#pragma unroll 1
    for (int k = 0; k < narr; k++)
      tma_bulk_g2s(sb + s_aoff[k], s_abase[k] + start * s_awidth[k], (uint32_t)((rows * s_awidth[k] + 15) & ~15LL), &s_bar[buf]);
  };
  if (threadIdx.x == 0) {
    s_nused[0] = 0; s_nused[1] = 0;
    mbar_init(&s_bar[0], 1); mbar_init(&s_bar[1], 1);
    mbar_fence_init();
    if (nchunks > 0) issue(0, 0);
  }
  __syncthreads();
  uint32_t phase[2] = {0, 0};
  int p = pA;
  uint32_t nu = 0;      // claimed slots (= groups alive in the table), block-uniform
  const int lane = threadIdx.x & 31;
  const uint32_t lt = (1u << lane) - 1u;
  // every logged group -> the compact group arrays, every logged slot reset: the table is EMPTY afterwards.  Only called at a
  // partition boundary (all rows of every group in the table have been seen).  A partial flush is not possible with linear
  // probing: resetting some slots breaks the probe chains of the groups that stay.
  auto flush_all = [&]() {
    __syncthreads();
    const uint32_t n_used = s_nused[0];
    for (uint32_t u0 = threadIdx.x & ~31u; u0 < n_used; u0 += RG_NT) {
      const uint32_t u = u0 + lane;
      const bool valid = u < n_used;
      const int sl = valid ? t_used[u] : 0;
      const uint32_t bal = __ballot_sync(0xffffffffu, valid);
      unsigned long long o = 0;
      if (lane == 0) o = atomicAdd(a.gcount, (unsigned long long)__popc(bal));
      o = __shfl_sync(0xffffffffu, o, 0) + __popc(bal & lt);
      if (valid) {
        a.gk0[o] = t_k0[sl];
        if (rp.has_k1) a.gk1[o] = t_k1[sl];
        for (int l = 0; l < plan.limbs; l++) a.gacc[o * plan.limbs + l] = t_acc[(size_t)sl * plan.limbs + l];
        for (int v = 0; v < plan.nvalids; v++) a.gnvalid[o * plan.nvalids + v] = t_nvalid[(size_t)sl * plan.nvalids + v];
        t_state[sl] = 0;
        for (int k = 0; k < plan.naggs; k++)
          for (int l = 0; l < plan.aggs[k].nlimbs; l++) t_acc[(size_t)sl * plan.limbs + plan.aggs[k].limb_off + l] = init_limb(plan.aggs[k]);
        for (int v = 0; v < plan.nvalids; v++) t_nvalid[(size_t)sl * plan.nvalids + v] = 0;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) s_nused[0] = 0;
    __syncthreads();
  };
  // A chunk's rows are aggregated all at once, whatever partitions they belong to (different partitions are just different
  // keys to the table); the partition order of the rows only bounds how many groups are alive at a time.  When the log of
  // claimed slots has grown past C/4 the chunk is cut at the next partition boundary and the table flushed there.  Two
  // barriers per chunk + three per flush, instead of four per partition (~480 rows) before.
  for (int64_t c = 0; c < nchunks; c++) {
    const int buf = (int)(c & 1);
    if (threadIdx.x == 0 && c + 1 < nchunks) issue(c + 1, buf ^ 1);
    mbar_wait(&s_bar[buf], phase[buf]);
    phase[buf] ^= 1;
    const char* sb = stage0 + (size_t)buf * sbytes;
    const uint64_t* s_k0 = reinterpret_cast<const uint64_t*>(sb);
    const uint64_t* s_k1 = reinterpret_cast<const uint64_t*>(sb + soff_k1);
    const uint32_t* s_vb = reinterpret_cast<const uint32_t*>(sb + soff_vb);
    const int64_t cs = a0 + c * CH;
    const int64_t lo = max(cs, r_lo), hi = min(cs + CH, r_hi);
    uint16_t claimed[4];   // slots this thread claimed in the current segment (a thread sees CH / RG_NT = 2 rows of a chunk)
    int nclaimed = 0;
    auto aggregate_rows = [&](int64_t from, int64_t to) {
      nclaimed = 0;
      // at most CH / RG_NT (= 2) rows per thread: fixed trip count, unrolled, so that both rows' probes overlap (with the
      // runtime bound the compiler kept them serial in one build and interleaved them in another: 2.25 vs 2.0 ms)
#pragma unroll
      for (int it = 0; it < CH / RG_NT; it++) {
        const int64_t r = from + (int64_t)it * RG_NT + threadIdx.x;
        if (r >= to) continue;
        const int li = (int)(r - cs);
        const uint64_t k0 = s_k0[li], k1 = rp.has_k1 ? s_k1[li] : 0;
        uint32_t idx = (uint32_t)rg_hash(k0, k1) & (uint32_t)(C - 1);
        int probes = 0;
        bool found = false;
        // A slot claimed in THIS segment carries the claiming row's stage index and is compared through the (read-only) stage
        // buffer; its key is written to the table without any fence and only read after the barrier that ends the segment,
        // when the claimer also sets RG_READY.  No memory fence and no volatile key read per row.
        while (!found) {
          uint32_t st = *reinterpret_cast<volatile uint32_t*>(&t_state[idx]);
          if (st == 0) {
            const uint32_t old = atomicCAS(&t_state[idx], 0u, (uint32_t)(li + 1));
            if (old == 0) {
              t_k0[idx] = k0;
              if (rp.has_k1) t_k1[idx] = k1;
              t_used[atomicAdd(&s_nused[0], 1u)] = (uint16_t)idx;
              if (nclaimed < 4) claimed[nclaimed] = (uint16_t)idx;
              nclaimed++;
              found = true;
              break;
            }
            st = old;
          }
          bool same;
          if (st & RG_READY) same = t_k0[idx] == k0 && (!rp.has_k1 || t_k1[idx] == k1);
          else { const int lj = (int)st - 1; same = s_k0[lj] == k0 && (!rp.has_k1 || s_k1[lj] == k1); }
          if (same) { found = true; break; }
          idx = (idx + 1) & (uint32_t)(C - 1);
          if (++probes > C / 2) { atomicExch(a.overflow, 1); break; }
        }
        if (!found) continue;
        const uint32_t vb = rp.use_vbits ? s_vb[li] : 0xffffffffu;
        uint64_t* acc = t_acc + (size_t)idx * plan.limbs;
        uint32_t* nv = t_nvalid + (size_t)idx * plan.nvalids;
        for (int k = 0; k < plan.naggs; k++) {
          const AggD& ag = plan.aggs[k];
          const int vs = rp.agg_val[k];
          const bool valid = vs < 0 || ((vb >> vs) & 1u);
          if (!valid) continue;
          if (ag.track_valid) atomicAdd(&nv[ag.valid_off], 1u);
          if (ag.kind == B2_AGG_COUNT || ag.kind == B2_AGG_COUNT_ALL) { atomicAdd(reinterpret_cast<unsigned long long*>(&acc[ag.limb_off]), 1ull); continue; }
          uint64_t lo64, hi64;
          if (rp.val[vs].width == 16) { const i128 x = reinterpret_cast<const i128*>(sb + soff_v[vs])[li]; lo64 = (uint64_t)x; hi64 = (uint64_t)(x >> 64); }
          else { lo64 = (uint64_t)reinterpret_cast<const int64_t*>(sb + soff_v[vs])[li]; hi64 = (int64_t)lo64 < 0 ? ~0ull : 0ull; }
          if (ag.kind == B2_AGG_SUM) acc_add_limbs(&acc[ag.limb_off], ag.nlimbs, lo64, hi64, (int64_t)hi64 < 0 ? ~0ull : 0ull);
          else if (ag.kind == B2_AGG_MIN) atomicMin(reinterpret_cast<unsigned long long*>(&acc[ag.limb_off]), (unsigned long long)ord_i64((int64_t)lo64));
          else if (ag.kind == B2_AGG_MAX) atomicMax(reinterpret_cast<unsigned long long*>(&acc[ag.limb_off]), (unsigned long long)ord_i64((int64_t)lo64));
        }
      }
    };
    int64_t from = lo;
    if (nu >= (uint32_t)(C / 4)) {
      while (p < pB && (int64_t)a.off[p + 1] <= lo) p++;   // a.off[p] <= lo < a.off[p + 1]
      if (p < pB) {
        const int64_t bnd = (int64_t)a.off[p] == lo ? lo : (int64_t)a.off[p + 1];   // the first partition boundary at or after lo
        if (bnd <= hi) {
          aggregate_rows(lo, bnd);
          flush_all();
          from = bnd;
        }
      }
    }
    aggregate_rows(from, hi);
    if (c + 1 == nchunks) { flush_all(); nclaimed = 0; }
    __syncthreads();   // the chunk is aggregated: every key is in the table, the stage buffer may be refilled
    for (int q = 0; q < nclaimed && q < 4; q++) t_state[claimed[q]] |= RG_READY;   // from now on compared through the table
    nu = s_nused[0];
    __syncthreads();   // nobody claims a slot of the next chunk before everybody has read the count
  }
}

struct RGKeyOut { void* data[MAX_KEYS]; int32_t width[MAX_KEYS]; };
__global__ void radix_finalize_kernel(const __grid_constant__ AggPlan plan, const __grid_constant__ RGPlan rp, int64_t ngroups, const uint64_t* __restrict__ gk0,
                                      const uint64_t* __restrict__ gk1, const uint64_t* __restrict__ gacc, const uint32_t* __restrict__ gnvalid,
                                      const __grid_constant__ AggOut out, const __grid_constant__ RGKeyOut ko) {
  for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < ngroups; o += (int64_t)gridDim.x * blockDim.x) {
    const u128 bits = ((u128)(rp.has_k1 ? gk1[o] : 0ull) << 64) | gk0[o];
    for (int k = 0; k < plan.nkeys; k++) {
      const uint64_t v = (uint64_t)(bits >> rp.key_shift[k]);
      switch (ko.width[k]) {
        case 1: reinterpret_cast<uint8_t*>(ko.data[k])[o] = (uint8_t)v; break;
        case 2: reinterpret_cast<uint16_t*>(ko.data[k])[o] = (uint16_t)v; break;
        case 4: reinterpret_cast<uint32_t*>(ko.data[k])[o] = (uint32_t)v; break;
        default: reinterpret_cast<uint64_t*>(ko.data[k])[o] = v; break;
      }
    }
    finalize_group(plan, &gacc[o * plan.limbs], &gnvalid[o * plan.nvalids], o, out);
  }
}

// ------------------------------------------------------------------------------------------------
void check_program_inputs(const Program* p, const Table* t);
void fill_inputs(VMInputs& in, const Table* t);
int vm_grid(int64_t nrows, int smem_bytes, int tile_rows);
Table* gather_table(const Table* t, const int32_t* d_map, int64_t n, bool nullify_oob, const std::vector<int>* only_cols);
Program* make_passthrough_program(const Table* t, const std::vector<int>& cols);

static int mt_of_dtype(int dtype) {
  switch (dtype) {
    case B2_BOOL8: case B2_INT8: return MT_I8;
    case B2_INT16: return MT_I16;
    case B2_INT32: case B2_DATE32: case B2_DECIMAL32: return MT_I32;
    case B2_INT64: case B2_TIMESTAMP_US: case B2_DECIMAL64: return MT_I64;
    case B2_DECIMAL128: return MT_I128;
    case B2_FLOAT32: return MT_F32;
    case B2_FLOAT64: return MT_F64;
  }
  throw Error(B2_ERR_UNSUPPORTED, "aggregation over dtype " + std::to_string(dtype));
}


// result columns of the aggregates for `ngroups` groups
static void make_agg_outputs(const AggPlan& plan, const Program* prog, const b2_agg_spec* specs, int naggs, int64_t ngroups, ColsGuard& outs, AggOut& ao) {
  memset(&ao, 0, sizeof(ao));
  for (int k = 0; k < naggs; k++) {
    int odt = specs[k].out_dtype;
    if (plan.aggs[k].kind == B2_AGG_COUNT || plan.aggs[k].kind == B2_AGG_COUNT_ALL) odt = B2_INT64;
    if (plan.aggs[k].kind == B2_AGG_MIN || plan.aggs[k].kind == B2_AGG_MAX) odt = prog->out_dtype[plan.aggs[k].out_idx];
    bool nullable = plan.aggs[k].track_valid || (plan.aggs[k].kind == B2_AGG_SUM && plan.aggs[k].nlimbs >= 2);
    int oscale = (plan.aggs[k].kind == B2_AGG_MIN || plan.aggs[k].kind == B2_AGG_MAX) ? prog->out_scale[plan.aggs[k].out_idx] : specs[k].out_scale;
    Column* c = new_column(odt, oscale, ngroups, nullable);
    outs.v.push_back(c);
    ao.data[k] = c->data.p; ao.valid[k] = c->valid.as<uint32_t>();
    ao.out_dtype[k] = odt; ao.out_precision[k] = specs[k].out_precision;
    if (c->valid.p) CUDA_CHECK(cudaMemsetAsync(c->valid.p, 0, c->valid.bytes, stream()));
  }
}

// the radix-partitioned regime; nullptr = not applicable (or a partition overflowed its table): the caller falls back
static Table* radix_groupby(const Program* prog, const Table* t, const AggPlan& plan, const b2_agg_spec* specs, const std::vector<int>& key_table_cols,
                            const VMInputs& in) {
  if (getenv("B2_AGG_NO_RADIX")) return nullptr;
  const int64_t n = t->rows;
  const int nkeys = plan.nkeys, naggs = plan.naggs;
  RGPlan rp; memset(&rp, 0, sizeof(rp));
  int kb = 0;
  for (int k = 0; k < nkeys; k++) {
    const KeyCol& c = plan.keys.c[k];
    if (c.dtype == B2_STRING || c.width == 16 || c.valid) return nullptr;   // fixed-width NOT NULL keys, <= 16 bytes together
    rp.key_shift[k] = 8 * kb; kb += c.width;
  }
  if (kb > 16 || kb == 0) return nullptr;
  rp.has_k1 = kb > 8;
  for (int k = 0; k < naggs; k++) {
    const AggD& a = plan.aggs[k];
    if (a.is_float) return nullptr;
    if (a.kind != B2_AGG_SUM && a.kind != B2_AGG_COUNT && a.kind != B2_AGG_COUNT_ALL && a.kind != B2_AGG_MIN && a.kind != B2_AGG_MAX) return nullptr;
    rp.agg_val[k] = -1;
    if (a.out_idx < 0) continue;
    int slot = -1;
    for (int s2 = 0; s2 < rp.nvals; s2++) if (rp.val[s2].out_idx == a.out_idx) slot = s2;
    if (slot < 0) {
      if (rp.nvals >= RG_MAX_VALS) return nullptr;
      slot = rp.nvals++;
      rp.val[slot].out_idx = a.out_idx; rp.val[slot].in_mt = a.in_mt; rp.val[slot].width = a.in_mt == MT_I128 ? 16 : 8;
      if (prog->out_nullable[a.out_idx]) rp.use_vbits = 1;
    }
    rp.agg_val[k] = slot;
  }
  const int ncols_moved = 2 + rp.has_k1 + rp.nvals + rp.use_vbits;
  if (ncols_moved > PT_MAXC) return nullptr;
  // shared-memory budget of the aggregation kernel: table of C slots + two stage buffers
  const int slot_bytes = 8 + (rp.has_k1 ? 8 : 0) + plan.limbs * 8 + 4 + plan.nvalids * 4 + 2;   // + the claimed-slot log
  int sbytes = RG_CHUNK * 8 + 16 + (rp.has_k1 ? RG_CHUNK * 8 + 16 : 0) + (rp.use_vbits ? RG_CHUNK * 4 + 16 : 0);
  for (int s2 = 0; s2 < rp.nvals; s2++) sbytes += RG_CHUNK * rp.val[s2].width + 16;
  sbytes = (sbytes + 127) & ~127;
  int C = 2048;
  while (C >= 1024 && C * slot_bytes + 2 * sbytes + 512 > 200 * 1024) C >>= 1;
  if (C < 1024) return nullptr;
  const int agg_smem = C * slot_bytes + 2 * sbytes + 512;

  // 1. materialise the (filtered, projected) rows
  struct Side { DevBuf h, k0, k1, v[RG_MAX_VALS], vbits; };
  Side A, B;
  auto alloc_side = [&](Side& sd) {
    sd.h = DevBuf((size_t)n * 4 + 64); sd.k0 = DevBuf((size_t)n * 8 + 64);
    if (rp.has_k1) sd.k1 = DevBuf((size_t)n * 8 + 64);
    for (int s2 = 0; s2 < rp.nvals; s2++) sd.v[s2] = DevBuf((size_t)n * rp.val[s2].width + 64);
    if (rp.use_vbits) sd.vbits = DevBuf((size_t)n * 4 + 64);
  };
  auto rows_of = [&](Side& sd) {
    RGRows r; memset(&r, 0, sizeof(r));
    r.h = sd.h.as<uint32_t>(); r.k0 = sd.k0.as<uint64_t>(); r.k1 = sd.k1.as<uint64_t>(); r.vbits = sd.vbits.as<uint32_t>();
    for (int s2 = 0; s2 < rp.nvals; s2++) r.v[s2] = sd.v[s2].as<char>();
    return r;
  };
  alloc_side(A);
  DevBuf counter(16);
  CUDA_CHECK(cudaMemsetAsync(counter.p, 0, 16, stream()));
  {
    const int vm_smem = prog->hdr.smem_bytes;
    if (vm_smem > 32 * 1024) CUDA_CHECK(cudaFuncSetAttribute(radix_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, vm_smem));
    KernelTimer kt("radix_rows_kernel");
    radix_rows_kernel<<<vm_grid(n, vm_smem, prog->hdr.tile_rows), VM_NT, vm_smem, stream()>>>(prog->d_hdr.as<VMProgramHeader>(), prog->d_code.as<VMInstr>(), in, plan, rp,
                                                                                                rows_of(A), n, counter.as<unsigned long long>());
    CUDA_CHECK(cudaGetLastError());
    count_launch();
  }
  int64_t m = n;
  if (plan.has_pred) { unsigned long long hm = 0; d2h(&hm, counter.p, 1); sync(); m = (int64_t)hm; }
  if (m == 0) return nullptr;
  // 2. radix partition by key hash so that a partition's groups fit the shared-memory table at load <= ~0.4
  int64_t P = 1;
  while (P * (int64_t)(C * 2 / 5) < m && P < (1 << 20)) P <<= 1;
  int lgP = 0; while ((1LL << lgP) < P) lgP++;
  Side* cur = &A; Side* oth = &B;
  if (P > 1) {
    alloc_side(B);
    DevBuf pid((size_t)m * 4);
    // LSD passes of at most 8 bits each (the <= 256-way scatter is the fast one), stable, so the final order is by h & (P - 1)
    for (int shift = 0; shift < lgP;) {
      const int bits = std::min(8, lgP - shift);
      rg_digit_kernel<<<grid_for(m, 256), 256, 0, stream()>>>(cur->h.as<uint32_t>(), m, shift, (1u << bits) - 1u, pid.as<int32_t>());
      count_launch();
      ScatterCols sc; memset(&sc, 0, sizeof(sc));
      auto add = [&](DevBuf& i, DevBuf& o, int w) { sc.width[sc.n] = w; sc.in[sc.n] = i.p; sc.out[sc.n] = o.p; sc.n++; };
      add(cur->h, oth->h, 4); add(cur->k0, oth->k0, 8);
      if (rp.has_k1) add(cur->k1, oth->k1, 8);
      for (int s2 = 0; s2 < rp.nvals; s2++) add(cur->v[s2], oth->v[s2], rp.val[s2].width);
      if (rp.use_vbits) add(cur->vbits, oth->vbits, 4);
      partition_scatter_arrays(pid.as<int32_t>(), m, 1 << bits, sc);
      std::swap(cur, oth);
      shift += bits;
    }
  }
  DevBuf off((size_t)(P + 1) * 4);
  rg_offsets_kernel<<<grid_for(m, 256), 256, 0, stream()>>>(cur->h.as<uint32_t>(), m, (uint32_t)(P - 1), off.as<int32_t>());
  count_launch();
  // 3. aggregate every partition in shared memory
  DevBuf gk0((size_t)m * 8), gk1(rp.has_k1 ? (size_t)m * 8 : 8), gacc((size_t)m * plan.limbs * 8), gnv((size_t)m * plan.nvalids * 4), ovf(4);
  CUDA_CHECK(cudaMemsetAsync(ovf.p, 0, 4, stream()));
  RGAgg ap; memset(&ap, 0, sizeof(ap));
  ap.rows = rows_of(*cur); ap.off = off.as<int32_t>(); ap.P = (int32_t)P; ap.C = C; ap.m = m;
  ap.gk0 = gk0.as<uint64_t>(); ap.gk1 = gk1.as<uint64_t>(); ap.gacc = gacc.as<uint64_t>(); ap.gnvalid = gnv.as<uint32_t>();
  ap.gcount = counter.as<unsigned long long>() + 1; ap.overflow = ovf.as<int32_t>();
  {
    CUDA_CHECK(cudaFuncSetAttribute(radix_agg_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, agg_smem));
    KernelTimer kt("radix_agg_kernel");
    radix_agg_kernel<<<(int)std::min<int64_t>(P, sm_count()), RG_NT, agg_smem, stream()>>>(plan, rp, ap);
    CUDA_CHECK(cudaGetLastError());
    count_launch();
  }
  unsigned long long hg = 0; int32_t hovf = 0;
  d2h(&hg, counter.as<unsigned long long>() + 1, 1);
  d2h(&hovf, ovf.p, 1);
  sync();
  if (hovf) return nullptr;   // pathological skew: the global-table regime takes over
  const int64_t ngroups = (int64_t)hg;
  // 4. unpack keys, finalise aggregates
  ColsGuard outs;
  RGKeyOut ko; memset(&ko, 0, sizeof(ko));
  for (int k = 0; k < nkeys; k++) {
    const Column* kc = t->cols[key_table_cols[k]];
    Column* c = new_column(kc->dtype, kc->scale, ngroups, false);
    outs.v.push_back(c);
    ko.data[k] = c->data.p; ko.width[k] = dtype_width(kc->dtype);
  }
  AggOut ao;
  make_agg_outputs(plan, prog, specs, naggs, ngroups, outs, ao);
  if (ngroups) {
    radix_finalize_kernel<<<grid_for(ngroups, 256), 256, 0, stream()>>>(plan, rp, ngroups, gk0.as<uint64_t>(), gk1.as<uint64_t>(), gacc.as<uint64_t>(), gnv.as<uint32_t>(), ao, ko);
    CUDA_CHECK(cudaGetLastError());
    count_launch();
  }
  sync();   // the scratch arrays are freed on return
  return new_table(outs.release());
}

// core: program outputs -> (keys, aggregates).  Key outputs must be plain input columns.
Table* scan_aggregate(const Program* prog, bool has_pred, const Table* t, const int* key_outs, int nkeys,
                      const b2_agg_spec* specs, int naggs) {
  check_program_inputs(prog, t);
  B2_CHECK(naggs <= AG_MAX_AGGS, "too many aggregates");
  B2_CHECK(nkeys <= MAX_KEYS, "too many group-by keys");
  if (has_pred) B2_CHECK(prog->hdr.nouts >= 1 && prog->out_dtype[0] == B2_BOOL8, "fused predicate must be output 0 and BOOL8");
  const int base = has_pred ? 1 : 0;
  const int64_t n = t->rows;
  AggPlan plan; memset(&plan, 0, sizeof(plan));
  plan.nkeys = nkeys; plan.naggs = naggs; plan.has_pred = has_pred;
  std::vector<int> key_table_cols;
  for (int k = 0; k < nkeys; k++) {
    int o = key_outs[k] + base;
    B2_CHECK(o >= 0 && o < prog->hdr.nouts, "key output index out of range");
    const VMOperand& op = prog->hdr.outs[o];
    if (op.kind != OK_COL) throw Error(B2_ERR_UNSUPPORTED, "group-by keys must be plain columns of the input (project computed keys first)");
    key_table_cols.push_back(op.idx);
  }
  plan.keys = key_cols_of(t, key_table_cols.data(), nkeys);
  {
    // packed-key budget: fixed-width columns take their width, short strings share what is left of 8 bytes
    int fixed_bytes = 0, nstr = 0; bool ok = nkeys > 0;
    for (int k = 0; k < nkeys; k++) {
      if (plan.keys.c[k].dtype == B2_STRING) nstr++;
      else if (plan.keys.c[k].width == 16) ok = false;
      else fixed_bytes += plan.keys.c[k].width;
    }
    ok = ok && fixed_bytes + 2 * nstr <= 8;
    for (int k = 0; k < nkeys && ok; k++)
      plan.keys.c[k].pack = plan.keys.c[k].dtype == B2_STRING ? (8 - fixed_bytes) / nstr : plan.keys.c[k].width;
    plan.fast_keys = ok;
  }
  int limbs = 0, nvalids = 0;
  for (int k = 0; k < naggs; k++) {
    AggD& a = plan.aggs[k];
    a.kind = specs[k].kind;
    a.out_idx = -1; a.in_mt = MT_I64; a.is_float = 0;
    bool in_nullable = false;
    int in_dtype = B2_INT64;
    if (a.kind != B2_AGG_COUNT_ALL) {
      int o = specs[k].column + base;
      B2_CHECK(o >= 0 && o < prog->hdr.nouts, "aggregate input index out of range");
      a.out_idx = o; a.in_mt = prog->hdr.out_mt[o]; in_nullable = prog->out_nullable[o]; in_dtype = prog->out_dtype[o];
      if (in_dtype == B2_STRING) throw Error(B2_ERR_UNSUPPORTED, "aggregates over strings");
    }
    a.is_float = (a.in_mt == MT_F32 || a.in_mt == MT_F64);
    switch (a.kind) {
      case B2_AGG_SUM:
        if (a.is_float) a.nlimbs = 1;
        else if (is_decimal(in_dtype)) {
          a.nlimbs = a.in_mt == MT_I128 ? 3 : 2;
          B2_CHECK(specs[k].out_dtype == B2_DECIMAL128 || specs[k].out_dtype == B2_DECIMAL64, "decimal sum needs a decimal result type");
          B2_CHECK(specs[k].out_precision >= 1 && specs[k].out_precision <= 38, "decimal sum needs out_precision");
        } else {
          B2_CHECK(specs[k].out_dtype == B2_INT64, "integral sum result type is INT64");
          a.nlimbs = 1;
        }
        break;
      case B2_AGG_COUNT: case B2_AGG_COUNT_ALL: a.nlimbs = 1; break;
      case B2_AGG_MIN: case B2_AGG_MAX:
        if (a.in_mt == MT_I128) throw Error(B2_ERR_UNSUPPORTED, "min/max over DECIMAL128");
        a.nlimbs = 1; break;
      default: throw Error(B2_ERR_UNSUPPORTED, "aggregate kind " + std::to_string(a.kind));
    }
    a.limb_off = limbs; limbs += a.nlimbs;
    a.track_valid = (a.kind == B2_AGG_SUM || a.kind == B2_AGG_MIN || a.kind == B2_AGG_MAX) && (in_nullable || nkeys == 0 || has_pred);
    if (a.track_valid) a.valid_off = nvalids++;
  }
  plan.limbs = std::max(limbs, 1); plan.nvalids = std::max(nvalids, 1);
  VMInputs in; fill_inputs(in, t);
  const int vm_smem = prog->hdr.smem_bytes;

  DevBuf gkeys, gknull;
  auto alloc_table = [&](int64_t cap, DevBuf& slots, DevBuf& acc, DevBuf& nv, DevBuf& ovf, GTable& gt) {
    slots = DevBuf((size_t)cap * 4); acc = DevBuf((size_t)cap * plan.limbs * 8); nv = DevBuf((size_t)cap * plan.nvalids * 4);
    ovf = DevBuf(4);
    gt.keys = nullptr; gt.knull = nullptr;
    if (plan.fast_keys) { gkeys = DevBuf((size_t)cap * 8); gknull = DevBuf((size_t)cap * 4); gt.keys = gkeys.as<uint64_t>(); gt.knull = gknull.as<uint32_t>(); }
    gt.slots = slots.as<int32_t>(); gt.acc = acc.as<uint64_t>(); gt.nvalid = nv.as<uint32_t>(); gt.mask = (uint32_t)(cap - 1);
    gt.overflow = ovf.as<int32_t>();
    CUDA_CHECK(cudaMemsetAsync(ovf.p, 0, 4, stream()));
    init_table_kernel<<<grid_for(cap, 256), 256, 0, stream()>>>(gt, plan, cap);
    count_launch();
  };

  DevBuf slots, acc, nv, ovf;
  GTable gt;
  int64_t cap = 0;
  bool done = false;
  // cardinality probe: on large keyed inputs run the shared-memory regime over a 256 K-row prefix first;
  // if even that overflows the per-CTA tables the whole input goes straight to the global regime
  bool try_smem = true;
  if (nkeys > 0 && n > (1 << 20)) {
    DevBuf ps, pa, pn, po; GTable pg;
    const int64_t pn_rows = 1 << 18;
    int per_slot = 4 + plan.limbs * 8 + plan.nvalids * 4 + 16;
    int nslots = 128;
    while (nslots * 2 <= SMEM_SLOTS_MAX && nslots * 2 * per_slot <= 24 * 1024) nslots *= 2;
    plan.smem_slots = nslots;
    int table_bytes = nslots * 4 + nslots * plan.limbs * 8 + nslots * plan.nvalids * 4 + 8 + nslots * 12 + nslots * 4 + 8 + 2 * 2 * prog->hdr.tile_rows + 16;
    int smem = ((vm_smem + 15) & ~15) + table_bytes;
    if (smem <= 160 * 1024) {
      int grid = vm_grid(pn_rows, smem, prog->hdr.tile_rows);
      int64_t pcap = 1;
      while (pcap < (int64_t)grid * nslots * 2) pcap <<= 1;
      alloc_table(pcap, ps, pa, pn, po, pg);
      if (smem > 32 * 1024) CUDA_CHECK(cudaFuncSetAttribute(aggregate_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      aggregate_kernel<true><<<grid, VM_NT, smem, stream()>>>(prog->d_hdr.as<VMProgramHeader>(), prog->d_code.as<VMInstr>(), in, plan, pg, pn_rows,
                                                                (vm_smem + 15) & ~15);
      CUDA_CHECK(cudaGetLastError());
      count_launch();
      int32_t h = 0;
      d2h(&h, po.p, 1);
      sync();
      try_smem = h == 0;
    }
    if (!try_smem) {   // many groups: radix-partitioned shared-memory aggregation (falls through when not applicable)
      if (Table* r = radix_groupby(prog, t, plan, specs, key_table_cols, in)) return r;
    }
  }
  // regime 1: shared-memory tables (always right for reductions; optimistic for group-by)
  if (try_smem) {
    // table sized for <= ~24 KB: more slots = shorter probe chains and more groups before the global regime
    int per_slot = 4 + plan.limbs * 8 + plan.nvalids * 4 + 16;
    int nslots = 128;
    while (nslots * 2 <= SMEM_SLOTS_MAX && nslots * 2 * per_slot <= 24 * 1024) nslots *= 2;
    if (nkeys == 0) nslots = 8;   // a reduction uses slot 0 only; the freed shared memory buys a 4th CTA per SM
    plan.smem_slots = nslots;
    int table_bytes = nslots * 4 + nslots * plan.limbs * 8 + nslots * plan.nvalids * 4 + 8;
    if (nkeys == 0) table_bytes += plan.limbs * VM_NT * 8 + plan.nvalids * VM_NT * 4;
    else table_bytes += nslots * 12 + nslots * 4 + 8 + 2 * 2 * prog->hdr.tile_rows + 16;
    int smem = ((vm_smem + 15) & ~15) + table_bytes;
    if (smem <= 160 * 1024) {
      int grid = n > 0 ? vm_grid(n, smem, prog->hdr.tile_rows) : 1;
      cap = 1;
      while (cap < (int64_t)grid * nslots * 2) cap <<= 1;
      if (nkeys == 0) cap = 1;
      alloc_table(cap, slots, acc, nv, ovf, gt);
      if (n > 0 || nkeys == 0) {
        if (smem > 32 * 1024) CUDA_CHECK(cudaFuncSetAttribute(aggregate_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        KernelTimer kt_aggregate_smem_kernel("aggregate_smem_kernel");
        aggregate_kernel<true><<<grid, VM_NT, smem, stream()>>>(prog->d_hdr.as<VMProgramHeader>(), prog->d_code.as<VMInstr>(), in, plan, gt, n,
                                                                  (vm_smem + 15) & ~15);
        CUDA_CHECK(cudaGetLastError());
        count_launch();
      }
      int32_t h_ovf = 0;
      if (nkeys > 0) { d2h(&h_ovf, ovf.p, 1); sync(); }
      done = h_ovf == 0;
    }
  }
  if (!done) {  // regime 2: global table sized for the worst case (every row its own group)
    cap = 1024;
    while (cap < n * 2) cap <<= 1;
    alloc_table(cap, slots, acc, nv, ovf, gt);
    if (vm_smem > 32 * 1024) CUDA_CHECK(cudaFuncSetAttribute(aggregate_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, vm_smem));
    KernelTimer kt_aggregate_global_kernel("aggregate_global_kernel");
    aggregate_kernel<false><<<vm_grid(n, vm_smem, prog->hdr.tile_rows), VM_NT, vm_smem, stream()>>>(prog->d_hdr.as<VMProgramHeader>(), prog->d_code.as<VMInstr>(), in,
                                                                                plan, gt, n, (vm_smem + 15) & ~15);
    CUDA_CHECK(cudaGetLastError());
    count_launch();
  }
  // compact occupied slots
  DevBuf pos((size_t)(cap + 1) * 4);
  occupied_flags_kernel<<<grid_for(cap, 256), 256, 0, stream()>>>(gt.slots, cap, pos.as<int32_t>());
  count_launch();
  DevBuf sums = exclusive_scan<int32_t, int32_t>(pos.as<int32_t>(), pos.as<int32_t>(), cap, true);
  int32_t ngroups = 0;
  d2h(&ngroups, pos.as<int32_t>() + cap, 1);
  sync();
  ColsGuard outs;
  AggOut ao;
  make_agg_outputs(plan, prog, specs, naggs, ngroups, outs, ao);
  DevBuf rep((size_t)std::max(ngroups, 1) * 4);
  finalize_kernel<<<grid_for(cap, 256), 256, 0, stream()>>>(gt, plan, cap, pos.as<int32_t>(), ao, rep.as<int32_t>());
  CUDA_CHECK(cudaGetLastError());
  count_launch();
  std::vector<Column*> result;
  if (nkeys > 0) {
    Table* kt = gather_table(t, rep.as<int32_t>(), ngroups, false, &key_table_cols);
    for (auto*& c : kt->cols) {
      if ((c->dtype == B2_FLOAT32 || c->dtype == B2_FLOAT64) && ngroups > 0) {
        KeyCol k; memset(&k, 0, sizeof(k));
        k.data = c->data.p; k.dtype = c->dtype; k.width = dtype_width(c->dtype);
        normalize_float_key_kernel<<<grid_for(ngroups, 256), 256, 0, stream()>>>(k, ngroups);
        CUDA_CHECK(cudaGetLastError());
        count_launch();
      }
      result.push_back(c); c = nullptr;
    }
    kt->cols.clear();
    delete kt;
  }
  for (auto* c : outs.release()) result.push_back(c);
  return new_table(std::move(result));
}

// identity program over selected columns of a table (used by the unfused b2_reduce / b2_groupby)
Program* make_passthrough_program(const Table* t, const std::vector<int>& cols) {
  std::unique_ptr<Program> p(new Program());
  memset(&p->hdr, 0, sizeof(p->hdr));
  B2_CHECK((int)cols.size() <= VM_MAX_OUTS, "too many columns");
  p->hdr.nouts = (int)cols.size();
  p->col_dtype.assign(t->cols.size() > VM_MAX_COLS ? VM_MAX_COLS : t->cols.size(), -1);
  int maxc = 0;
  for (size_t i = 0; i < cols.size(); i++) {
    int c = cols[i];
    B2_CHECK(c >= 0 && c < (int)t->cols.size() && c < VM_MAX_COLS, "column index out of range");
    const Column* col = t->cols[c];
    VMOperand& o = p->hdr.outs[i];
    memset(&o, 0, sizeof(o));
    o.kind = OK_COL; o.idx = c; o.nullable = col->nullable();
    p->hdr.out_mt[i] = col->dtype == B2_STRING ? MT_I8 : (uint8_t)mt_of_dtype(col->dtype);
    p->out_dtype.push_back(col->dtype); p->out_scale.push_back(col->scale); p->out_precision.push_back(0);
    p->out_nullable.push_back(col->nullable());
    p->col_dtype[c] = col->dtype;
    maxc = std::max(maxc, c + 1);
  }
  p->hdr.ncols = maxc;
  set_tile_geometry(p->hdr, 0);
  p->col_dtype.resize(maxc);
  p->d_hdr = DevBuf(sizeof(VMProgramHeader));
  h2d(p->d_hdr.p, &p->hdr, 1);
  p->d_code = DevBuf(sizeof(VMInstr));
  sync();
  return p.release();
}

}  // namespace b2

using namespace b2;
extern "C" {

int b2_scan_aggregate(b2_handle program, int32_t has_predicate, b2_handle table, const int32_t* key_cols, int32_t nkeys,
                      const b2_agg_spec* aggs, int32_t naggs, b2_handle* out_table) {
  B2_TRY
  *out_table = to_handle(scan_aggregate(program_from(program), has_predicate != 0, table_from(table), key_cols, nkeys, aggs, naggs));
  B2_CATCH
}

static Table* unfused(const Table* t, const int32_t* key_cols, int nkeys, const b2_agg_spec* aggs, int naggs) {
  std::vector<int> cols;
  std::vector<int> key_outs;
  for (int k = 0; k < nkeys; k++) { key_outs.push_back((int)cols.size()); cols.push_back(key_cols[k]); }
  std::vector<b2_agg_spec> specs(aggs, aggs + naggs);
  for (auto& s : specs) {
    if (s.kind == B2_AGG_COUNT_ALL) continue;
    int c = s.column;
    s.column = (int)cols.size();
    cols.push_back(c);
  }
  if (cols.empty()) cols.push_back(0);
  std::unique_ptr<Program> p(make_passthrough_program(t, cols));
  return scan_aggregate(p.get(), false, t, key_outs.data(), nkeys, specs.data(), naggs);
}

int b2_reduce(b2_handle table, const b2_agg_spec* aggs, int32_t naggs, b2_handle* out_table) {
  B2_TRY
  *out_table = to_handle(unfused(table_from(table), nullptr, 0, aggs, naggs));
  B2_CATCH
}

int b2_groupby(b2_handle table, const int32_t* key_cols, int32_t nkeys, const b2_agg_spec* aggs, int32_t naggs, b2_handle* out_table) {
  B2_TRY
  *out_table = to_handle(unfused(table_from(table), key_cols, nkeys, aggs, naggs));
  B2_CATCH
}

__global__ void count_occupied_kernel(const int32_t* slots, int64_t cap, unsigned long long* out) {
  unsigned long long acc = 0;
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < cap; s += (int64_t)gridDim.x * blockDim.x) acc += slots[s] != SLOT_EMPTY;
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

int b2_distinct_count(b2_handle table, const int32_t* key_cols, int32_t nkeys, int64_t* out) {
  B2_TRY
  // Table.distinctCount: group-by with no aggregates; the row count of the result
  Table* t = table_from(table);
  std::unique_ptr<Table, void (*)(Table*)> r(unfused(t, key_cols, nkeys, nullptr, 0), table_release);
  // a key-only group-by yields exactly the distinct rows; with zero keys every row is one group
  *out = nkeys == 0 ? (t->rows > 0 ? 1 : 0) : r->rows;
  B2_CATCH
}

}  // extern "C"
