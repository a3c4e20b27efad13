// omg_sp.cuh -- "sparse" variant of the interior-point kernel (included by omg_b200.cu).
//
// Same algorithm as ipm_body (oracle/ipm_ref.py; reference call site problem.py:113), with
// the linear algebra and the table streams re-designed for instance-level parallelism:
//
//   * KKT factorisation K = L D L^T on a SPARSE symbolic structure computed once per problem
//     (constrained minimum-degree ordering; all instances of a batch share it): config 2 needs
//     4.0 k stored entries instead of 8.9 k for the envelope of the time-ordered band -> the
//     factor fits 4 blocks per SM -- and the sequential chain shrinks from 200 pivots to 8
//     supernode levels + one dense root of 36 columns.
//       - SUPERNODES: paths of the elimination tree of up to SP_SNW columns with the structure
//         of their last column (few explicit zeros), one level step each:
//         GATHER, left-looking, one thread per stored entry: one record per (entry, source
//         supernode) -- byte offsets of the two rows in the supernode's first column + its table
//         entry -- contributes  v -= sum_t A_it * rd_t * A_jt  over the supernode's columns
//         (unscaled columns A = L D, rd = 1/d: the pivot signs come with d);
//         PANEL: one task per panel row; every task factorises the w x w diagonal block for
//         itself (identical arithmetic) and finishes its row -- no block barrier inside;
//       - the dense root (the final chain of the elimination tree, <= 40 columns): right-looking
//         by panels of four columns with the trailing triangle held in REGISTERS (static entry
//         ownership), two barriers per four pivots;
//       - early rejection of an attempt at the first negative pivot among variables that no
//         equality row touches (the inertia count could not come out right any more);
//       - the right-hand side rides along as row N, so only the backward sweep remains
//         (root: one warp, shuffle broadcast; the rest: level by level, 8 lanes per column, the
//         supernode's own triangle solved inside its warp with shuffles).
//   * every table stream is laid out per THREAD ("thread streams"): a thread owns whole
//     outputs (slots, rows, H positions, columns), balanced by record count; record k of its
//     chunk t sits at ((t*8+k)*NT + tid) -> every warp load is one coalesced line, there are
//     no descriptor loads, 8 independent loads are in flight per thread, and term records
//     take 16 bytes instead of 32;
//   * K is assembled in the block's L2-resident scratch (structural entries only) and STAGED
//     into shared memory by a TMA bulk load (cp.async.bulk + mbarrier, SASS UBLKCP) over the
//     region the Jacobian values occupied during the assembly -- factor and Jacobian share
//     their shared memory in time, which is what lets a fourth block fit on an SM; the same
//     load serves the inertia-correction retries;
//   * m-vectors that are only streamed (one thread per row, coalesced) live in the L2-resident
//     scratch; shared memory holds what is gathered at random: L, the Jacobian values, x, the
//     parameter tape, Sigma, y.
#pragma once

#define SP_MAXROOT 40
#define SP_SNW 4                // columns of a supernode (elimination-tree path)
#define SP_SNZ 8                // explicit zeros a supernode may add
#define SP_SNZ_TOTAL 400        // ... and all of them together
#define SP_RCH 1               // root: row chunks per thread (40 columns -> 125 chunks of 8)
#define SP_RCW 8               // root: columns per chunk
#define SP_MAXCOL 62           // |struct| of a column (pair delta is 6 bits)
#define SP_MAXL 8191           // stored entries incl. zero slot (13 bits)
#define SP_MAXN 2046

struct __align__(16) PT16 { double coef; unsigned short cidx, a, b, c; };   // cidx bit 15: last record of its output

// "thread stream": every thread owns whole outputs; its records are stored consecutively,
// padded to n_chunk chunks of SP_R records; record k of chunk t of thread tid sits at
// ((t * SP_R + k) * NT + tid) -> every warp load is one coalesced line, no descriptor loads,
// SP_R independent loads in flight per thread.  The last record of an output carries an end
// flag and the output index.
#ifndef SP_R
#define SP_R 8
#endif
struct SpStream { int n_chunk; const void* rec; };

struct SpTab {
  int nt;                          // threads per block the streams were laid out for
  int Lsz, zslot, R0, nr, n_lev, root0, n_rootent;
  int neg_lev;                     // levels < neg_lev hold only variables no equality row touches: a negative
                                   //   pivot there already decides the inertia test (see SP_CHECK)
  // factorisation levels (+ the gather into the root as level n_lev): slices of 32 entries
  const int* lev_ptr;              // [n_lev+2] slice ranges
  const uint4* fdesc;              // per slice lane: {entry word, pair offset (uint4 units), n4, 0}
                                   //   entry word: lidx | col<<13 | isdiag<<24 | eq-pivot<<25 (0xffffffff idle)
  const uint4* fpair;              // 2 pairs per uint4, [slice][k2][lane]; pair = {a8 | b8<<16, k8}: byte offsets into LK / rd
  const unsigned* root_ch;         // [SP_RCH * nt] row chunk of a thread: i | k0<<6 | cnt<<12 | eq-pivot<<16
                                   //   (root-local row i (nr = rhs), columns k0 .. k0+cnt-1; 0: none)
  const uint4* sntab; int n_sn;    // per supernode (+ a dummy): {d1 | d2<<16, d3 | r0<<16, r1 | r2<<16, r3}: byte distance from a
                                   //   row's entry in the first column to column t, byte offset of 1/d_t in rd
  // panel step of the supernodes with 2..SP_SNW columns: per level, rounds of nt tasks
  const int* ptask_ptr;            // [n_lev+1] round ranges per level
  const uint4* ptask;              // {c0 | w<<11 | q<<14 | eq-pivots<<17 | valid<<31, cb0 | cb1<<16, cb2 | cb3<<16, r}:
                                   //   q = 0: row r of the rows below the block (the last one is the rhs row);
                                   //   q >= 1: row q of the diagonal block.  cb: byte offset of a column's diagonal entry
  const int* ksign;                // [N] +1 / -1 by permuted index
  // backward sweep: per level, rounds of NT/8 columns; one 32-byte record per lane
  const int* brnd_ptr;             // [n_lev+1] round ranges per level
  const uint4* bdesc;              // [round][NT][3]: {j8 | valid<<16 | nq<<17, rhs8, e0, e1}, {e2..e5}, {e6, e7, -, -};
                                   //   e = LK byte offset | uu byte offset << 16 of entry sub + 8 q (zero slot if none)
  const int* diagidx; const int* rhsidx;     // [N] L index of the diagonal / rhs entry of a column
  const int* pos_var; const int* pos_eq;     // permutation of this structure
  const int* jdst;                 // [nnz_j] L index of the border entry of an equality-row slot
  const uint2* border; int n_border;   // equality rows: {slot | row<<16, L index}; slot 0xffff = rhs entry
  const unsigned short* vdiag;     // [N] L index of the diagonal of permuted column j | eq-row<<15
  SpStream J, G, W, H, C, R;
};

struct SpSmem {   // offsets in doubles
  int LK, jval, xe, xt, dx, gf, rd, diag0, V, sig, y, red, filt, rt8, rki, lptr, sntab, total;
  // scratch (global) offsets in doubles
  int Kc, g, s, zU, dsc, sU, ds, dy, dzU, gt, st, wv, zL, sL, dzL, beq, jt, yg, sigg, gtotal;
};

// ---- TMA bulk copies (1-D) ---------------------------------------------------------
#ifndef OMG_CPU_EMU
__device__ __forceinline__ unsigned sp_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sp_mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(sp_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void sp_mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(sp_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void sp_mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n .reg .pred p;\n WAIT_%=:\n"
      " mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      " @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}\n"
      :: "r"(sp_smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void sp_bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               :: "r"(sp_smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(sp_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void sp_bulk_s2g(void* dst_gmem, const void* src_smem, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               :: "l"(dst_gmem), "r"(sp_smem_u32(src_smem)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void sp_bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void sp_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void sp_fence_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void sp_prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" :: "l"(p)); }
#else
static inline void sp_prefetch_l1(const void*) {}
static inline void sp_mbar_init(unsigned long long* bar, unsigned) { *bar = 0; }
static inline void sp_mbar_expect_tx(unsigned long long*, unsigned) {}
static inline void sp_mbar_wait(unsigned long long*, unsigned) { __syncthreads(); }   // every thread waits: the copy (thread 0) is done
static inline void sp_bulk_g2s(void* d, const void* s, unsigned bytes, unsigned long long*) { memcpy(d, s, bytes); }
static inline void sp_bulk_s2g(void* d, const void* s, unsigned bytes) { memcpy(d, s, bytes); }
static inline void sp_bulk_wait_all() {}
static inline void sp_bulk_wait_read() {}
static inline void sp_fence_async() {}
#endif

#ifndef OMG_CPU_EMU
__device__ __forceinline__ double sp_rcp(double x) { return __drcp_rn(x); }   // correctly rounded, = 1.0 / x
#else
static inline double sp_rcp(double x) { return 1.0 / x; }
#endif

// term streams: SP_R independent 16-byte loads per chunk, then the sums in stream order.
//   VAL(r) -> value of record r (uint4);  BODY uses o_ (the record's uint4) and acc_
#define SP_STREAM16(ST, VAL, BODY)                                                           \
  {                                                                                          \
    const uint4* rp_ = reinterpret_cast<const uint4*>((ST).rec) + tid;                       \
    double acc_ = 0.0;                                                                       \
    for (int t_ = 0; t_ < (ST).n_chunk; ++t_, rp_ += SP_R * NT) {                            \
      uint4 rr_[SP_R];                                                                       \
      _Pragma("unroll")                                                                      \
      for (int k_ = 0; k_ < SP_R; ++k_) rr_[k_] = __ldg(rp_ + k_ * NT);                      \
      _Pragma("unroll")                                                                      \
      for (int k_ = 0; k_ < SP_R; ++k_) {                                                    \
        const uint4 o_ = rr_[k_];                                                            \
        acc_ += (VAL);                                                                     \
        if (o_.z & 0x8000u) { BODY acc_ = 0.0; }                                             \
      }                                                                                      \
    }                                                                                        \
  }
// 8-byte index streams; end flag = bit 16 of .y (bit 30 for H)
#define SP_STREAM8(ST, ENDBIT, VAL, BODY)                                                    \
  {                                                                                          \
    const uint2* rp_ = reinterpret_cast<const uint2*>((ST).rec) + tid;                       \
    double acc_ = 0.0;                                                                       \
    for (int t_ = 0; t_ < (ST).n_chunk; ++t_, rp_ += SP_R * NT) {                            \
      uint2 rr_[SP_R];                                                                       \
      _Pragma("unroll")                                                                      \
      for (int k_ = 0; k_ < SP_R; ++k_) rr_[k_] = __ldg(rp_ + k_ * NT);                      \
      _Pragma("unroll")                                                                      \
      for (int k_ = 0; k_ < SP_R; ++k_) {                                                    \
        const uint2 o_ = rr_[k_];                                                            \
        acc_ += (VAL);                                                                     \
        if (o_.y & (ENDBIT)) { BODY acc_ = 0.0; }                                            \
      }                                                                                      \
    }                                                                                        \
  }
#define SP_COEF(r) __hiloint2double((int)(r).y, (int)(r).x)
#define SP_VJ(X) (SP_COEF(o_) * V[o_.z & 0x7fffu] * (X)[o_.z >> 16])                       // J: a = x0, b = slot, c = row
#define SP_VG(X) (SP_COEF(o_) * V[o_.z & 0x7fffu] * (X)[o_.z >> 16] * (X)[o_.w & 0xffffu])   // G: a, b = x0, x1, c = row
#define SP_VC(JV, YV) ((JV)[o_.x & 0xffffu] * (YV)[o_.x >> 16])                             // C / R: slot | index<<16

// objective terms (few, off the hot path): ONE out-of-line copy instead of an unrolled inline
// expansion at every call site -- the kernel's code is larger than the instruction cache
#ifndef OMG_CPU_EMU
__device__ __noinline__
#else
static
#endif
double sp_eval_range(const PTerm* t, int lo, int hi, const double* V, const double* xe) {
  double acc = 0.0;
  int aux;
#pragma unroll 1
  for (int k = lo; k < hi; ++k) acc += term_value(t + k, V, xe, &aux);
  return acc;
}

// ---------------------------------------------------------------------------------------
// factorisation K = L D L^T in LK (unscaled columns A = L D), rd = 1/d.  ctl->fail on a bad
// pivot or wrong inertia (mode 0: IPOPT's count test; mode 1: sign by position).
// flags[3]: per-level pivot reports (negative count | bad<<16 | eq-bad<<24), rotating so that
// a level's report is read after its barrier while the next level already writes its own.
// Early rejection (mode 0): while every eliminated column is a variable v that no equality row
// touches (levels < P.neg_lev), a negative pivot means v^T H v < 0 for a v with J_eq v = 0 --
// the reduced Hessian is not positive definite, the inertia cannot be (n, n_eq, 0), and the
// count at the end of the factorisation would say the same (more than n_eq negatives).
// ---------------------------------------------------------------------------------------
#define SP_PIVOT(j, v, isneg_)                                                                 \
  {                                                                                           \
    const bool neg_ = (v) < 0.0;                                                              \
    const double d_ = fabs(v);                                                                \
    bool bad_;                                                                                \
    if (mode) bad_ = (neg_ != (isneg_)) || !(d_ > ((isneg_) ? 0.0 : PIV_TOL * fmax(rd[j], 1e-300))) || !(d_ < 1e300); \
    else bad_ = !(d_ > PIV_TOL * fmax(rd[j], 1e-300)) || !(d_ < 1e300);                       \
    rd[j] = sp_rcp(v);                      /* rd[j] held |K_jj| until now */                 \
    const int rep_ = (neg_ ? 1 : 0) + (bad_ ? (1 << 16) : 0) + ((bad_ && (isneg_)) ? (1 << 24) : 0); \
    if (rep_) atomicAdd(&flags[slot_], rep_);                                                 \
  }
#define SP_CHECK()                                                                            \
  {                                                                                           \
    const int rep_ = flags[slot_];                                                            \
    if (tid == 0) flags[(slot_ == 0) ? 2 : slot_ - 1] = 0;                                    \
    slot_ = (slot_ == 2) ? 0 : slot_ + 1;                                                     \
    nneg += rep_ & 0xffff;                                                                    \
    if ((rep_ >> 16) || (mode == 0 && (nneg > T.n_eq || (nneg > 0 && lv < P.neg_lev)))) {    \
      if (tid == 0) { ctl->fail = 1; ctl->eq_fail = (rep_ >> 24) ? 1 : 0; }                   \
      __syncthreads();                                                                        \
      return;                                                                                 \
    }                                                                                         \
  }
// pair record (8 bytes): byte offsets a8 | b8<<16 into LK, k8 into rd -- no index arithmetic
#define SP_LDB(base, off) (*reinterpret_cast<const double*>(reinterpret_cast<const char*>(base) + (off)))
// (record: byte offsets of the two rows' entries in the source supernode's first column, byte
// offset of the supernode's table entry; up to four columns contribute)
#define SP_PAIR(lo, hi)                                                                        \
  {                                                                                           \
    const uint4 st_ = *reinterpret_cast<const uint4*>(sntb + (hi));                           \
    const char* pa_ = reinterpret_cast<const char*>(LK) + ((lo) & 0xffffu);                   \
    const char* pb_ = reinterpret_cast<const char*>(LK) + ((lo) >> 16);                       \
    v0 -= SP_LDB(pa_, 0) * SP_LDB(rd, st_.y >> 16) * SP_LDB(pb_, 0);                          \
    v1 -= SP_LDB(pa_, st_.x & 0xffffu) * SP_LDB(rd, st_.z & 0xffffu) * SP_LDB(pb_, st_.x & 0xffffu); \
    v0 -= SP_LDB(pa_, st_.x >> 16) * SP_LDB(rd, st_.z >> 16) * SP_LDB(pb_, st_.x >> 16);      \
    v1 -= SP_LDB(pa_, st_.y & 0xffffu) * SP_LDB(rd, st_.w) * SP_LDB(pb_, st_.y & 0xffffu);    \
  }
#define SP_PAIR4(pc) { SP_PAIR((pc).x, (pc).y) SP_PAIR((pc).z, (pc).w) }
// descriptor of slice sl (idle if the level has no slice for this warp) / its first 16 pairs
#define SP_FDESC(d, sl, s_end) { (d) = make_uint4(0xffffffffu, 0u, 0u, 0u); if ((sl) < (s_end)) (d) = __ldg(P.fdesc + (sl) * 32 + lane); }
#define SP_NPF 2                 // uint4 words (2 pairs each) of every entry fetched one level ahead
#define SP_FPAIRS(p, d) { const uint4* q_ = P.fpair + (d).y;                                   \
    _Pragma("unroll") for (int w_ = 0; w_ < SP_NPF; ++w_) if ((d).z > (unsigned)w_) (p)[w_] = __ldg(q_ + 32 * w_); }

__device__ __forceinline__ void sp_factor(const DevTab& T, const SpTab& P, const SpSmem& S, Ctl* ctl,
                                          int* flags, const int mode, double* pc) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double* LK = sm + S.LK; double* rd = sm + S.rd;
  long long t0_ = clock64();
#define SP_FT(k) do { if (pc && tid == 0) { const long long t_ = clock64(); pc[k] += (double)(t_ - t0_); t0_ = t_; } } while (0)
  const int* lptr = reinterpret_cast<const int*>(sm + S.lptr);
  const int* tptr = lptr + (2 * P.n_lev + 3);
  const char* sntb = reinterpret_cast<const char*>(sm + S.sntab);
  if (tid < 3) flags[tid] = 0;
  int slot_ = 0, nneg = 0;
  // ownership of the root (static): every thread holds up to SP_RCH chunks of SP_RCW
  // consecutive columns of ONE row in registers
  unsigned rch[SP_RCH];
#pragma unroll
  for (int q = 0; q < SP_RCH; ++q) rch[q] = __ldg(P.root_ch + q * NT + tid);
  // ---- levels of the elimination tree (+ the gather into the root as level n_lev) ----
  // A level is worked off in steps of NWARP slices (step k of level lv: slice lptr[lv] + k NWARP +
  // warp).  Software pipeline over ALL steps, across the level barriers (descriptors and pair
  // records do not depend on the numerics): descriptor two steps ahead, the first pair words of
  // every entry one step ahead.
  int lv = 0, b0 = lptr[0], lv1, b1, lv2, b2;
#define SP_NEXT(lvn, bn, lvc, bc)                                                              \
  { lvn = lvc; bn = bc + NWARP;                                                               \
    if (lvc <= P.n_lev && bn >= lptr[lvc + 1]) { lvn = lvc + 1; bn = (lvn <= P.n_lev) ? lptr[lvn] : 0; } }
  SP_NEXT(lv1, b1, lv, b0)
  SP_NEXT(lv2, b2, lv1, b1)
  uint4 dA, dB, pA[SP_NPF], pB[SP_NPF];
  SP_FDESC(dA, b0 + warp, lptr[1])
  SP_FDESC(dB, b1 + warp, (lv1 <= P.n_lev) ? lptr[lv1 + 1] : 0)
  SP_FPAIRS(pA, dA)
  __syncthreads();
  while (lv <= P.n_lev) {
    uint4 dC;
    SP_FPAIRS(pB, dB)                                       // next step
    {   // the rest of that slice's pair block: one 128-byte line per lane into L1
      const int nl = ((int)dB.z - SP_NPF) * 4;
      if (lane < nl) sp_prefetch_l1(P.fpair + (dB.y - lane) + (SP_NPF * 4 + lane) * 8);
    }
    SP_FDESC(dC, b2 + warp, (lv2 <= P.n_lev) ? lptr[lv2 + 1] : 0)
    uint4 tk0 = make_uint4(0u, 0u, 0u, 0u);                 // first panel task of this level, fetched early
    if (lv1 != lv && lv < P.n_lev && tptr[lv] < tptr[lv + 1]) tk0 = __ldg(P.ptask + (size_t)tptr[lv] * NT + tid);
    {
      const uint4 d = dA;
      const unsigned e = d.x;
      const int li = (e == 0xffffffffu) ? P.zslot : (int)(e & 0x1fffu);
      const int n4 = (int)d.z;
      double v0 = LK[li], v1 = 0.0;
      uint4 r[4];
      if (n4 > SP_NPF) {                                   // the rest of a long list: four loads in flight
        const uint4* q_ = P.fpair + d.y + SP_NPF * 32;
#pragma unroll
        for (int t = 0; t < 4; ++t) if (SP_NPF + t < n4) r[t] = __ldg(q_ + t * 32);
      }
#pragma unroll
      for (int w = 0; w < SP_NPF; ++w) if (n4 > w) SP_PAIR4(pA[w])
      if (n4 > SP_NPF) {
#pragma unroll
        for (int t = 0; t < 4; ++t) if (SP_NPF + t < n4) SP_PAIR4(r[t])
      }
      for (int k = SP_NPF + 4; k < n4; k += 4) {
        const uint4* q_ = P.fpair + d.y + k * 32;
#pragma unroll
        for (int t = 0; t < 4; ++t) if (k + t < n4) r[t] = __ldg(q_ + t * 32);
#pragma unroll
        for (int t = 0; t < 4; ++t) if (k + t < n4) SP_PAIR4(r[t])
      }
      const double v = v0 + v1;
      if (e != 0xffffffffu) {
        LK[li] = v;
        if (e & (1u << 24)) { const int j = (e >> 13) & 0x7ffu; SP_PIVOT(j, v, (e & (1u << 25)) != 0u) }
      }
    }
    if (lv1 != lv) {                                        // the level's last step
    __syncthreads();
    SP_CHECK()
    SP_FT(8);                                               // gathers (levels and root)
    if (lv < P.n_lev && tptr[lv] < tptr[lv + 1]) {
      // ---- panel step of this level's supernodes (2..SP_SNW columns).  After the gather the
      // panel holds its pre-final entries; every task factorises the w x w diagonal block for
      // itself (identical arithmetic in all of them) and finishes ONE row by forward
      // substitution.  Rows below the block are stored in place (nobody else reads them); the
      // rows of the block itself -- read by every task -- after the closing barrier.
      double pv1 = 0.0, pv2 = 0.0, pv3 = 0.0;
      unsigned po1 = 0xffffffffu, po2 = 0xffffffffu, po3 = 0xffffffffu;
      for (int tr = tptr[lv]; tr < tptr[lv + 1]; ++tr) {
        const uint4 tk = (tr == tptr[lv]) ? tk0 : __ldg(P.ptask + (size_t)tr * NT + tid);
        if (tk.x & 0x80000000u) {
          const int w = (tk.x >> 11) & 7, q = (tk.x >> 14) & 7;
          const unsigned cb0 = tk.y & 0xffffu, cb1 = tk.y >> 16, cb2 = tk.z & 0xffffu, cb3 = tk.z >> 16;
          const double d0 = SP_LDB(LK, cb0), a10 = SP_LDB(LK, cb0 + 8), g11 = SP_LDB(LK, cb1);
          const double a20 = (w > 2) ? SP_LDB(LK, cb0 + 16) : 0.0, g21 = (w > 2) ? SP_LDB(LK, cb1 + 8) : 0.0,
                       g22 = (w > 2) ? SP_LDB(LK, cb2) : 1.0;
          const double a30 = (w > 3) ? SP_LDB(LK, cb0 + 24) : 0.0, g31 = (w > 3) ? SP_LDB(LK, cb1 + 16) : 0.0,
                       g32 = (w > 3) ? SP_LDB(LK, cb2 + 8) : 0.0, g33 = (w > 3) ? SP_LDB(LK, cb3) : 1.0;
          double x0 = 0.0, x1 = 0.0, x2 = 0.0, x3 = 0.0;
          unsigned o1 = 0u, o2 = 0u, o3 = 0u;
          if (q == 0) {                                          // a row below the block: offsets, loads first
            const unsigned r8 = (tk.w + (unsigned)w) * 8u;       // entry of column t: cb_t + 8 (w - t + r)
            o1 = cb1 + r8 - 8u; o2 = cb2 + r8 - 16u; o3 = cb3 + r8 - 24u;
            x0 = SP_LDB(LK, cb0 + r8); x1 = SP_LDB(LK, o1);
            if (w > 2) x2 = SP_LDB(LK, o2);
            if (w > 3) x3 = SP_LDB(LK, o3);
          }
          const double r0 = sp_rcp(d0);
          const double l10 = a10 * r0, l20 = a20 * r0, l30 = a30 * r0;
          const double d1 = g11 - l10 * a10;
          const double r1 = sp_rcp(d1);
          const double a21 = g21 - l20 * a10, a31 = g31 - l30 * a10;
          const double l21 = a21 * r1, l31 = a31 * r1;
          const double d2 = g22 - l20 * a20 - l21 * a21;
          const double r2 = sp_rcp(d2);
          const double a32 = g32 - l30 * a20 - l31 * a21;
          const double l32 = a32 * r2;
          const double d3 = g33 - l30 * a30 - l31 * a31 - l32 * a32;
          if (q == 0) {
            x1 -= (x0 * r0) * a10;
            x2 -= (x0 * r0) * a20 + (x1 * r1) * a21;
            x3 -= (x0 * r0) * a30 + (x1 * r1) * a31 + (x2 * r2) * a32;
            *reinterpret_cast<double*>(reinterpret_cast<char*>(LK) + o1) = x1;
            if (w > 2) *reinterpret_cast<double*>(reinterpret_cast<char*>(LK) + o2) = x2;
            if (w > 3) *reinterpret_cast<double*>(reinterpret_cast<char*>(LK) + o3) = x3;
          } else {                                               // row q of the block: pivots, stores deferred
            const int c0 = (int)(tk.x & 0x7ffu);
            const unsigned eqb = (tk.x >> 17) & 15u;
            if (q == 1) {
              { const int jc = c0; SP_PIVOT(jc, d0, (eqb & 1u) != 0u) }
              { const int jc = c0 + 1; SP_PIVOT(jc, d1, (eqb & 2u) != 0u) }
              pv1 = d1; po1 = cb1;
            } else if (q == 2) {
              { const int jc = c0 + 2; SP_PIVOT(jc, d2, (eqb & 4u) != 0u) }
              pv1 = a21; po1 = cb1 + 8; pv2 = d2; po2 = cb2;
            } else {
              { const int jc = c0 + 3; SP_PIVOT(jc, d3, (eqb & 8u) != 0u) }
              pv1 = a31; po1 = cb1 + 16; pv2 = a32; po2 = cb2 + 8; pv3 = d3; po3 = cb3;
            }
          }
        }
      }
      __syncthreads();
      SP_CHECK()
      if (po1 != 0xffffffffu) *reinterpret_cast<double*>(reinterpret_cast<char*>(LK) + po1) = pv1;
      if (po2 != 0xffffffffu) *reinterpret_cast<double*>(reinterpret_cast<char*>(LK) + po2) = pv2;
      if (po3 != 0xffffffffu) *reinterpret_cast<double*>(reinterpret_cast<char*>(LK) + po3) = pv3;
    }
    SP_FT(15);                                              // panel steps
    }
    dA = dB; dB = dC;
#pragma unroll
    for (int w = 0; w < SP_NPF; ++w) pA[w] = pB[w];
    lv = lv1; b0 = b1; lv1 = lv2; b1 = b2;
    { int lvn_, bn_; SP_NEXT(lvn_, bn_, lv1, b1) lv2 = lvn_; b2 = bn_; }
  }
#undef SP_NEXT
  // ---- dense root: right-looking by PANELS of four columns, trailing entries in registers ----
  // entry (row i, column k) lives at R[off(k) + i - k], off(k) = k (nr + 1) - k (k - 1) / 2.
  // Panel p0, two barriers for four pivots:
  //   1. the owners publish the columns p0..p0+3 as they stand after the earlier panels (the
  //      updates of the panel's own columns are still missing)                      -- barrier
  //   2. every owner of a panel row factorises the 4 x 4 diagonal block for itself (10 loads, a
  //      few dozen flops, identical in all of them), finishes its own row by forward
  //      substitution and stores it (rows below the block in place; the block's own rows after
  //      the barrier, they are still being read); the four diagonal owners report the pivots
  //                                                                                  -- barrier
  //   3. rank-4 update of the registers:  val[j] -= sum_t (x_it / d_t) x_{k0+j,t}.
  const int nr = P.nr;
  if (nr > 0) {
    static_assert(SP_RCH == 1 && SP_RCW == 8, "panelised root: one chunk of 8 columns per thread");
    double* R = LK + P.root0;
    const int i = rch[0] & 63u, k0 = (rch[0] >> 6) & 63u, cnt = (rch[0] >> 12) & 15u;
    const bool eqp = (rch[0] & 0x10000u) != 0u;
    double val[SP_RCW];
#pragma unroll
    for (int j = 0; j < SP_RCW; ++j) {
      const int k = k0 + j;
      val[j] = (j < cnt) ? R[k * (nr + 1) - (k * (k - 1)) / 2 + i - k] : 0.0;
    }
#define SP_ROFF(c) ((c) * (nr + 1) - ((c) * ((c) - 1)) / 2 - (c))      /* R[SP_ROFF(c) + row] */
    for (int p0 = 0; p0 < nr; p0 += 4) {
      const int pw = (nr - p0 < 4) ? nr - p0 : 4;
      const int half = p0 - k0;                              // 0 / 4: the panel is inside this chunk
      const bool mine = cnt > 0 && (half == 0 || half == 4) && i >= p0;
      const int u = i - p0;
      double* C0 = R + SP_ROFF(p0);
      double* C1 = R + SP_ROFF(p0 + 1);
      double* C2 = R + SP_ROFF(p0 + 2);
      double* C3 = R + SP_ROFF(p0 + 3);
      double x0 = 0.0, x1 = 0.0, x2 = 0.0, x3 = 0.0;        // this row's panel entries
      if (mine) {
        x0 = (half == 0) ? val[0] : val[4]; x1 = (half == 0) ? val[1] : val[5];
        x2 = (half == 0) ? val[2] : val[6]; x3 = (half == 0) ? val[3] : val[7];
        if (u < pw) {                                        // rows of the diagonal block: published
          C0[i] = x0;
          if (u >= 1) C1[i] = x1;
          if (u >= 2) C2[i] = x2;
          if (u >= 3) C3[i] = x3;
        }
      }
      __syncthreads();
      if (mine) {
        // diagonal block (missing columns of a short last panel: identity)
        const double d0 = C0[p0];
        const double a10 = (pw > 1) ? C0[p0 + 1] : 0.0, g11 = (pw > 1) ? C1[p0 + 1] : 1.0;
        const double a20 = (pw > 2) ? C0[p0 + 2] : 0.0, g21 = (pw > 2) ? C1[p0 + 2] : 0.0, g22 = (pw > 2) ? C2[p0 + 2] : 1.0;
        const double a30 = (pw > 3) ? C0[p0 + 3] : 0.0, g31 = (pw > 3) ? C1[p0 + 3] : 0.0, g32 = (pw > 3) ? C2[p0 + 3] : 0.0,
                     g33 = (pw > 3) ? C3[p0 + 3] : 1.0;
        const double r0 = sp_rcp(d0);
        const double l10 = a10 * r0, l20 = a20 * r0, l30 = a30 * r0;
        const double d1 = g11 - l10 * a10;
        const double r1 = sp_rcp(d1);
        const double a21 = g21 - l20 * a10, a31 = g31 - l30 * a10;
        const double l21 = a21 * r1, l31 = a31 * r1;
        const double d2 = g22 - l20 * a20 - l21 * a21;
        const double r2 = sp_rcp(d2);
        const double a32 = g32 - l30 * a20 - l31 * a21;
        const double l32 = a32 * r2;
        const double d3 = g33 - l30 * a30 - l31 * a31 - l32 * a32;
        if (u < pw) {                                        // a row of the block: entries and pivot
          double dv = d0;
          x0 = d0;
          if (u == 1) { x0 = a10; x1 = d1; dv = d1; }
          if (u == 2) { x0 = a20; x1 = a21; x2 = d2; dv = d2; }
          if (u == 3) { x0 = a30; x1 = a31; x2 = a32; x3 = d3; dv = d3; }
          const int jc = P.R0 + i;
          SP_PIVOT(jc, dv, eqp)
        } else {                                             // a row below: forward substitution
          x1 -= (x0 * r0) * a10;
          x2 -= (x0 * r0) * a20 + (x1 * r1) * a21;
          x3 -= (x0 * r0) * a30 + (x1 * r1) * a31 + (x2 * r2) * a32;
          C0[i] = x0;
          if (pw > 1) C1[i] = x1;
          if (pw > 2) C2[i] = x2;
          if (pw > 3) C3[i] = x3;
        }
      }
      __syncthreads();
      SP_CHECK()
      if (mine && u < pw) {                                  // the block's own rows, finished
        C0[i] = x0;
        if (u >= 1) C1[i] = x1;
        if (u >= 2) C2[i] = x2;
        if (u >= 3) C3[i] = x3;
      }
      if (cnt > 0 && i > p0 + 3 && k0 + cnt - 1 > p0 + 3) { // entries right of the panel
        if (!mine) { x0 = C0[i]; x1 = C1[i]; x2 = C2[i]; x3 = C3[i]; }   // (pw == 4 here)
        const double y0 = x0 * rd[P.R0 + p0], y1 = x1 * rd[P.R0 + p0 + 1],
                     y2 = x2 * rd[P.R0 + p0 + 2], y3 = x3 * rd[P.R0 + p0 + 3];
#pragma unroll
        for (int j = 0; j < SP_RCW; ++j) {
          const int k = k0 + j;                               // row k of the panel columns
          if (j < cnt && k > p0 + 3) val[j] -= y0 * C0[k] + y1 * C1[k] + y2 * C2[k] + y3 * C3[k];
        }
      }
    }
#undef SP_ROFF
  }
  __syncthreads();
  SP_FT(9);
  if (mode == 0 && nneg != T.n_eq) {   // Sylvester: wrong inertia
    if (tid == 0) { ctl->fail = 1; ctl->eq_fail = (nneg < T.n_eq) ? 1 : 0; }
    __syncthreads();
  }
}

// backward sweep: u = L^-T D^-1 z, z = the rhs entries of LK; result in uu[0..N)
__device__ __forceinline__ void sp_back_solve(const DevTab& T, const SpTab& P, const SpSmem& S, double* uu, double* pc) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  long long t0_ = clock64();
  const double* LK = sm + S.LK; const double* rd = sm + S.rd;
  const int* bptr = reinterpret_cast<const int*>(sm + S.lptr) + (P.n_lev + 2);
  const int nr = P.nr, R0 = P.R0;
  // descriptors of the first round of the top level, fetched while warp 0 does the root; after
  // that every round fetches the next one's before it starts (they do not depend on the numerics)
  uint4 na = make_uint4(0u, 0u, 0u, 0u), nb = na, nc = na;
  if (P.n_lev > 0) {
    const size_t o_ = ((size_t)bptr[P.n_lev - 1] * NT + tid) * 3;
    na = __ldg(P.bdesc + o_); nb = __ldg(P.bdesc + o_ + 1); nc = __ldg(P.bdesc + o_ + 2);
  }
  if (tid == NT - 1) uu[T.N] = 0.0;      // what the absent entries of the level records point at
  if (warp == 0 && nr > 0) {
    // root, one warp: lane l holds rows l and l+32 (root-local); four columns per trip so that
    // the operand loads run ahead of the dependent chain  w -> u_c -> broadcast -> w
    const double* R = LK + P.root0;
    const int i0 = lane, i1 = lane + 32;
    // offset of column c in R: c*(nr+1) - c*(c-1)/2
    const int o0 = i0 * (nr + 1) - (i0 * (i0 - 1)) / 2, o1 = i1 * (nr + 1) - (i1 * (i1 - 1)) / 2;
    double w0 = (i0 < nr) ? R[o0 + (nr - i0)] : 0.0;
    double w1 = (i1 < nr) ? R[o1 + (nr - i1)] : 0.0;
    for (int c = nr - 1; c >= 0; c -= 4) {
      double a0[4], a1[4], rdv[4];
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int ct = c - t;
        a0[t] = (i0 < ct) ? R[o0 + (ct - i0)] : 0.0;
        a1[t] = (i1 < ct && i1 < nr) ? R[o1 + (ct - i1)] : 0.0;
        rdv[t] = (ct >= 0) ? rd[R0 + ct] : 0.0;
      }
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int ct = c - t;
        if (ct >= 0) {
          const double mine = ((ct < 32) ? w0 : w1) * rdv[t];
          const double uc = __shfl_sync(FULL, mine, ct & 31);
          w0 -= a0[t] * uc;
          w1 -= a1[t] * uc;
          if (lane == (ct & 31)) uu[R0 + ct] = uc;
        }
      }
    }
  }
  __syncthreads();
  SP_FT(14);
  // the other columns, level by level from the top, 8 lanes per column; the records hold BYTE
  // offsets (entry of L, matching component of u), absent entries point at the zero slot
  const int sub = lane & 7;
#define SP_BENT(e) acc += SP_LDB(LK, (e) & 0xffffu) * SP_LDB(uu, (e) >> 16)
  for (int lv = P.n_lev - 1; lv >= 0; --lv) {
    const int r0 = bptr[lv], r1 = bptr[lv + 1];
    for (int r = r0; r < r1; ++r) {
      const uint4 da = na, db = nb, dc = nc;
      {
        const int rn = (r + 1 < r1) ? r + 1 : ((lv > 0) ? bptr[lv - 1] : -1);
        if (rn >= 0) { const size_t o_ = ((size_t)rn * NT + tid) * 3; na = __ldg(P.bdesc + o_); nb = __ldg(P.bdesc + o_ + 1); nc = __ldg(P.bdesc + o_ + 2); }
      }
      const int nq = (da.x >> 17) & 15u;                 // rounds of 8 entries this level needs (uniform)
      double acc = 0.0, acc2 = 0.0;
      { SP_BENT(da.z); }
      if (nq > 1) { acc2 += SP_LDB(LK, da.w & 0xffffu) * SP_LDB(uu, da.w >> 16); }
      if (nq > 2) { SP_BENT(db.x); acc2 += SP_LDB(LK, db.y & 0xffffu) * SP_LDB(uu, db.y >> 16); }
      if (nq > 4) { SP_BENT(db.z); acc2 += SP_LDB(LK, db.w & 0xffffu) * SP_LDB(uu, db.w >> 16); }
      if (nq > 6) { SP_BENT(dc.x); acc2 += SP_LDB(LK, dc.y & 0xffffu) * SP_LDB(uu, dc.y >> 16); }
      // the supernode's own triangle: rt = columns of the supernode solved before this one
      const int rt = (int)((dc.w >> 3) & 7u) - 1 - (int)(dc.w & 7u);
      const unsigned cb = dc.z;
      const double e0 = (rt > 0) ? SP_LDB(LK, cb + 8u * (unsigned)rt) : 0.0;
      const double e1 = (rt > 1) ? SP_LDB(LK, cb + 8u * (unsigned)(rt - 1)) : 0.0;
      const double e2 = (rt > 2) ? SP_LDB(LK, cb + 8u * (unsigned)(rt - 2)) : 0.0;
      const unsigned j8 = da.x & 0xffffu;
      const double rdj = SP_LDB(rd, j8);
      acc += acc2;
      acc += __shfl_xor_sync(FULL, acc, 1);
      acc += __shfl_xor_sync(FULL, acc, 2);
      acc += __shfl_xor_sync(FULL, acc, 4);
      double vj = SP_LDB(LK, da.y & 0xffffu) - acc;
      double uj = vj * rdj;                              // final where rt <= 0
      const int grp8 = lane & 24;
#pragma unroll
      for (int st = 0; st < SP_SNW - 1; ++st) {
        const int src = (rt > st) ? grp8 + 8 * (rt - st) : lane;     // lane group of the column solved at step st
        const double got = __shfl_sync(FULL, uj, src);
        if (rt > st) {
          vj -= ((st == 0) ? e0 : (st == 1) ? e1 : e2) * got;
          if (rt == st + 1) uj = vj * rdj;
        }
      }
      if ((da.x & 0x10000u) && sub == 0)
        *reinterpret_cast<double*>(reinterpret_cast<char*>(uu) + j8) = uj;
    }
    __syncthreads();
  }
#undef SP_BENT
}

// ---------------------------------------------------------------------------------------
// the solver kernel (no intermediates, term degree <= 3)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void ipm_body_sp(const DevTab& T, const SpTab& P, const omg_options& O,
                                            const Batch& A, const SpSmem& S) {
  __shared__ Ctl ctl;
  __shared__ int fflags[3];
  __shared__ unsigned long long kbar;
  __shared__ double phase_cyc[NPHASE];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = T.n, m = T.m, N = T.N;
  double* LK = sm + S.LK; double* jval = sm + S.jval;
  double* xe = sm + S.xe; double* xt = sm + S.xt; double* dx = sm + S.dx;
  double* rd = sm + S.rd; double* diag0 = sm + S.diag0; double* V = sm + S.V;
  // shared: sg2 = Sigma * dsc^2 and yd = y * dsc (what the gathers need with the UNSCALED
  // Jacobian values kept in jval), grad f; y, Sigma, dsc themselves are only streamed
  double* sg2 = sm + S.sig; double* yd = sm + S.y; double* gf = sm + S.gf;
  double* red = sm + S.red; double* filt = sm + S.filt;
  unsigned char* rt = reinterpret_cast<unsigned char*>(sm + S.rt8);
  double* D = A.dscr + (size_t)blockIdx.x * A.dscr_stride;
  double* Kg = D + S.Kc;
#define SP_GV(name, off) double* __restrict__ name = D + (off)
  SP_GV(g, S.g); SP_GV(s, S.s); SP_GV(zU, S.zU); SP_GV(dsc, S.dsc); SP_GV(sU, S.sU); SP_GV(ds, S.ds);
  SP_GV(dy, S.dy); SP_GV(dzU, S.dzU); SP_GV(gt, S.gt); SP_GV(st, S.st); SP_GV(wv, S.wv); SP_GV(zL, S.zL);
  SP_GV(sL, S.sL); SP_GV(dzL, S.dzL); SP_GV(beq, S.beq); SP_GV(jt, S.jt); SP_GV(y, S.yg); SP_GV(sig, S.sigg);
#undef SP_GV
  int* I = A.iscr + (size_t)blockIdx.x * A.iscr_stride;
  int* eqidx = I; int* eqrow = eqidx + m;
  unsigned kphase = 0;
  {  // once per block
    int* lp = reinterpret_cast<int*>(sm + S.lptr);
    for (int e = tid; e < P.n_lev + 2; e += NT) lp[e] = P.lev_ptr[e];
    for (int e = tid; e < P.n_lev + 1; e += NT) lp[P.n_lev + 2 + e] = P.brnd_ptr[e];
    for (int e = tid; e < P.n_lev + 1; e += NT) lp[2 * P.n_lev + 3 + e] = P.ptask_ptr[e];
    for (int e = tid; e < P.n_sn; e += NT) reinterpret_cast<uint4*>(sm + S.sntab)[e] = P.sntab[e];
    if (tid == 0) { sp_mbar_init(&kbar, 1); sp_fence_async(); }
    if (tid == 0) { sg2[m] = 0.0; yd[m] = 0.0; wv[m] = 0.0; }
    for (int i = tid; i <= N; i += NT) rd[i] = 0.0;
    for (int i = tid; i < P.Lsz; i += NT) Kg[i] = 0.0;      // fill positions stay zero for good
  }
  __syncthreads();

  for (;;) {
    if (tid == 0) ctl.inst = atomicAdd(A.counter, 1);
    __syncthreads();
    const int inst = ctl.inst;
    if (inst >= A.B) return;
    const double* x0 = A.x0 + (size_t)inst * n;
    const double* par = A.p + (size_t)inst * T.n_par;
    const double* lbg = A.lbg + (A.bounds_shared ? 0 : (size_t)inst * m);
    const double* ubg = A.ubg + (A.bounds_shared ? 0 : (size_t)inst * m);
    const bool tracing = (O.trace != 0) && inst == 0 && A.trace != nullptr;
    long long phase_t0 = clock64();
    if (tracing && tid == 0) for (int k = 0; k < NPHASE; ++k) phase_cyc[k] = 0.0;

    // ---- S1: parameter tape ---------------------------------------------------------
    for (int i = tid; i < 1 + T.n_par; i += NT) V[i] = (i == 0) ? 1.0 : par[i - 1];
    __syncthreads();
    for (int l = 0; l < T.n_levels; ++l) {
      for (int e = T.level_ptr[l] + tid; e < T.level_ptr[l + 1]; e += NT) {
        double acc = 0.0;
        for (int t = T.tape_ptr[e]; t < T.tape_ptr[e + 1]; ++t) {
          const int4 f = __ldg(reinterpret_cast<const int4*>(T.tape_fac) + t);
          acc += T.tape_coef[t] * V[f.x] * V[f.y] * V[f.z] * V[f.w];
        }
        switch (T.tape_func[e]) {
          case 1: acc = 1.0 / acc; break;
          case 2: acc = (acc >= 0.0) ? 1.0 : 0.0; break;
          case 3: acc = (acc > 0.0) ? 1.0 : 0.0; break;
          case 4: acc = sin(acc); break;
          case 5: acc = cos(acc); break;
          case 6: acc = sqrt(acc); break;
          default: break;
        }
        V[1 + T.n_par + e] = acc;
      }
      __syncthreads();
    }
    // ---- S2: x ------------------------------------------------------------------------
    for (int i = tid; i <= n; i += NT) { xe[i] = (i < n) ? x0[i] : 1.0; xt[i] = 1.0; }
    __syncthreads();

    // ---- S3: scaling, row classification, starting point --------------------------------
    double fmaxv = 0.0;
    for (int j = tid; j < n; j += NT)
      fmaxv = fmax(fmaxv, fabs(sp_eval_range(T.DFt, T.dfptr[j], T.dfptr[j + 1], V, xe)));
    {
      double r1[1] = {fmaxv}; const int o1[1] = {OP_MAX};
      block_reduce<1>(r1, o1, red);
      fmaxv = r1[0];
    }
    const double smg = O.scaling_max_gradient;
    const double fsc = (fmaxv > smg) ? fmax(smg / fmaxv, 1e-8) : 1.0;
    // unscaled Jacobian -> jval, g -> gt
    SP_STREAM16(P.J, SP_VJ(xe), jval[o_.w & 0xffffu] = acc_;)
    SP_STREAM16(P.G, SP_VG(xe), gt[o_.w >> 16] = acc_;)
    __syncthreads();
    for (int i = tid; i < m; i += NT) {
      const RowRec rr = T.rowrec[i];
      double gm = 0.0;
      for (int k = 0; k < rr.ns; ++k) gm = fmax(gm, fabs(jval[rr.s0 + k]));
      const double d = (gm > smg) ? fmax(smg / gm, 1e-8) : 1.0;
      dsc[i] = d;
      const double lb = lbg[i], ub = ubg[i];
      const bool eq = (lb == ub);
      const bool hL = (lb > -INF_BOUND) && !eq, hU = (ub < INF_BOUND) && !eq;
      rt[i] = (unsigned char)((hL ? 1 : 0) | (hU ? 2 : 0) | (eq ? 4 : 0));
      double l = lb * d, uu = ub * d;
      beq[i] = l;
      if (hL) l -= O.bound_relax_factor * fmax(1.0, fabs(l));
      if (hU) uu += O.bound_relax_factor * fmax(1.0, fabs(uu));
      sL[i] = l; sU[i] = uu;
      const double gi = d * gt[i];
      g[i] = gi;
      double si = gi;
      const double k1 = O.bound_push, k2 = O.bound_frac;
      double pl = k1 * fmax(1.0, fabs(l)), pu = k1 * fmax(1.0, fabs(uu));
      if (hL && hU) { pl = fmin(pl, k2 * (uu - l)); pu = fmin(pu, k2 * (uu - l)); }
      if (hL) si = fmax(si, l + pl);
      if (hU) si = fmin(si, uu - pu);
      s[i] = si;
      double yi = 0.0;
      if (A.lam0) yi = A.lam0[(size_t)inst * m + i] * fsc / d;
      y[i] = yi; yd[i] = yi * d;
      zL[i] = hL ? fmax(O.mult_bound_push, -yi) : 0.0;
      zU[i] = hU ? fmax(O.mult_bound_push, yi) : 0.0;
    }
    __syncthreads();
    if (tid == 0) {
      int ne = 0, nbnd = 0, bad = 0;
      for (int i = 0; i < m; ++i) {
        const int r = rt[i];
        if (r & 4) {
          if (ne < T.n_eq && T.eq_rows[ne] == i) { eqrow[ne] = i; eqidx[i] = ne; } else bad = 1;
          ++ne;
        } else eqidx[i] = -1;
        nbnd += (r & 1) + ((r >> 1) & 1);
      }
      if (ne != T.n_eq) bad = 1;
      ctl.n_eq = bad ? -1 : ne; ctl.n_bounds = nbnd;
      ctl.mu = O.mu_init; ctl.tau = fmax(TAU_MIN, 1.0 - O.mu_init);
      ctl.theta_max = -1.0; ctl.theta_min = -1.0;
      ctl.delta_w_last = 0.0; ctl.nfilt = 0; ctl.status = -1; ctl.iter = 0;
      ctl.fsc = fsc; ctl.alpha = 0.0; ctl.delta_w = 0.0; ctl.n_restart = 0;
      ctl.f = fsc * sp_eval_range(T.Ft, 0, T.n_f, V, xe);
    }
    __syncthreads();
    if (ctl.n_eq < 0) {   // equality pattern differs from the lowered structure
      if (tid == 0) { A.status[inst] = OMG_ERROR_IN_STEP_COMPUTATION; A.iters[inst] = 0; A.f[inst] = 0.0; }
      for (int i = tid; i < n; i += NT) A.x[(size_t)inst * n + i] = x0[i];
      for (int i = tid; i < m; i += NT) A.lam[(size_t)inst * m + i] = 0.0;
      __syncthreads();
      continue;
    }
    const int n_eq = ctl.n_eq;
    const int n_bounds = ctl.n_bounds;

    // =========================== IP iterations ===================================
    for (int iter = 0;; ++iter) {
      TICK(0);
      double rv[NRED];
      const int rop[NRED] = {OP_MAX, OP_MAX, OP_MIN, OP_MAX, OP_MAX, OP_MAX,
                             OP_SUM, OP_SUM, OP_SUM, OP_SUM, OP_MAX, OP_SUM};
      for (int r = 0; r < NRED; ++r) rv[r] = 0.0;
      rv[2] = 1e300;
      // ---- I1: Jacobian values (scaled) + per-row residual terms ---------------------
      SP_STREAM16(P.J, SP_VJ(xe), jval[o_.w & 0xffffu] = acc_;)
#pragma unroll 2
      for (int i = tid; i < m; i += NT) {
        const int r = rt[i];
        const double d = dsc[i];
        const double gi = g[i], si = s[i], yi = y[i];
        const double zl_ = zL[i], zu_ = zU[i], sl_ = sL[i], su_ = sU[i], be_ = beq[i], ub_ = ubg[i], lb_ = lbg[i];
        const double ci = (r & 4) ? gi - be_ : gi - si;
        rv[0] = fmax(rv[0], fabs(ci));
        rv[8] += fabs(ci);
        double zl = 0.0, zu = 0.0;
        if (r & 1) { zl = zl_; const double dl = si - sl_; const double pz = dl * zl;
          rv[1] = fmax(rv[1], pz); rv[2] = fmin(rv[2], pz); rv[9] += log(dl); rv[7] += zl; }
        if (r & 2) { zu = zu_; const double du = su_ - si; const double pz = du * zu;
          rv[1] = fmax(rv[1], pz); rv[2] = fmin(rv[2], pz); rv[9] += log(du); rv[7] += zu; }
        const double gun = gi / d;
        if (r & 6) rv[3] = fmax(rv[3], gun - ub_);
        if (r & 5) rv[3] = fmax(rv[3], lb_ - gun);
        if (!(r & 4)) { const double rs = fabs(-yi - zl + zu);
          rv[4] = fmax(rv[4], rs); rv[5] = fmax(rv[5], rs * d); }
        rv[6] += fabs(yi);
      }
      __syncthreads();
      TICK(1);
      // ---- I2: columns: grad f, dual residual (J^T y through the CSC ELL) --------------
      for (int j = tid; j < n; j += NT)
        gf[j] = ctl.fsc * sp_eval_range(T.DFt, T.dfptr[j], T.dfptr[j + 1], V, xe);
      __syncthreads();
      SP_STREAM8(P.C, 0x10000u, SP_VC(jval, yd), rv[10] = fmax(rv[10], fabs(gf[o_.y & 0xffffu] + acc_));)
      block_reduce<NRED>(rv, rop, red);
      const double cinf = rv[0], maxprod = rv[1], minprod = rv[2], viol = rv[3];
      const double dinf = fmax(rv[10], rv[4]);
      const double dinf_un = fmax(rv[10], rv[5]) / ctl.fsc;
      const double ysum = rv[6], zsum = rv[7], theta = rv[8], logsum = rv[9];
      const double s_d = fmax(S_MAX, (ysum + zsum) / fmax(1.0, (double)(m + n_bounds))) / S_MAX;
      const double s_c = fmax(S_MAX, zsum / fmax(1.0, (double)n_bounds)) / S_MAX;
      double mu = ctl.mu;
      const double cmpl0 = n_bounds ? fmax(fabs(maxprod), fabs(minprod)) : 0.0;
      const double E0 = fmax(fmax(dinf / s_d, cinf), cmpl0 / s_c);
      TICK(2);
      // ---- I3: termination + barrier update (uniform) -----------------------------------
      int status = -1;
      if (!isfinite(E0) || !isfinite(theta)) status = OMG_INVALID_NUMBER_DETECTED;
      else if (E0 <= O.tol && dinf_un <= O.dual_inf_tol && viol <= O.constr_viol_tol &&
               cmpl0 / ctl.fsc <= O.compl_inf_tol) status = OMG_SOLVE_SUCCEEDED;
      else if (iter >= O.max_iter) status = OMG_MAX_ITER_EXCEEDED;
      if (tracing && tid == 0 && iter < TRACE_ROWS - 2) {
        double* tr = A.trace + iter * TRACE_COLS;
        tr[0] = iter; tr[1] = ctl.f / ctl.fsc; tr[2] = cinf; tr[3] = dinf; tr[4] = mu; tr[5] = E0;
        tr[6] = ctl.alpha; tr[7] = ctl.delta_w;
      }
      if (status >= 0) { if (tid == 0) { ctl.status = status; ctl.iter = iter; } break; }
      {
        const double mu_min = fmin(O.tol, O.compl_inf_tol * ctl.fsc) / (KAPPA_EPS + 1.0);
        bool changed = false;
        for (;;) {
          const double cm = n_bounds ? fmax(fabs(maxprod - mu), fabs(minprod - mu)) : 0.0;
          const double Emu = fmax(fmax(dinf / s_d, cinf), cm / s_c);
          if (Emu <= KAPPA_EPS * mu && mu > mu_min) {
            mu = fmax(mu_min, fmin(KAPPA_MU * mu, pow(mu, THETA_MU)));
            changed = true;
          } else break;
        }
        __syncthreads();
        if (tid == 0) {
          ctl.mu = mu; ctl.tau = fmax(TAU_MIN, 1.0 - mu);
          if (changed) ctl.nfilt = 0;
          if (ctl.theta_max < 0.0) {
            ctl.theta_max = THETA_MAX_FACT * fmax(1.0, theta);
            ctl.theta_min = THETA_MIN_FACT * fmax(1.0, theta);
          }
          ctl.theta = theta;
          ctl.phi = ctl.f - mu * logsum;
          ctl.delta_w = 0.0; ctl.delta_c = 0.0; ctl.first_try = 1;
        }
      }
      __syncthreads();
      const double tau = ctl.tau;
      TICK(3);
      // ---- I4: Sigma, w = Sigma r_d + phi_s ----------------------------------------------
#pragma unroll 2
      for (int i = tid; i < m; i += NT) {
        const int r = rt[i];
        double sg = 0.0, ph = 0.0, rdd = 0.0;
        const double si = s[i], gi_ = g[i], sl_ = sL[i], su_ = sU[i], zl_ = zL[i], zu_ = zU[i];
        if (!(r & 4)) {
          rdd = gi_ - si;
          if (r & 1) { const double dl = si - sl_; sg += zl_ / dl; ph -= mu / dl; }
          if (r & 2) { const double du = su_ - si; sg += zu_ / du; ph += mu / du; }
        }
        const double d = dsc[i];
        sig[i] = sg; sg2[i] = sg * d * d;
        wv[i] = d * ((r & 4) ? y[i] : (sg * rdd + ph));
      }
      __syncthreads();
      TICK(4);
      // ---- I7/I8: assemble + factorise, with inertia correction -----------------------
      // K is assembled in the block's L2-resident scratch Kg (structural entries only: the fill
      // positions were zeroed once and are never written), then staged into shared memory by a
      // TMA bulk load over the region the Jacobian values occupied -- the same load serves the
      // inertia-correction retries.
      {
        // H positions: gather J^T Sigma J.  record: s1 | s2<<16, row | (dst | diag<<13 | end<<14)<<16
        SP_STREAM8(P.H, 0x40000000u, jval[o_.x & 0xffffu] * sg2[o_.y & 0xffffu] * jval[o_.x >> 16],
                   Kg[(o_.y >> 16) & 0x1fffu] = acc_;)
        __syncthreads();
        TICK(5);
        // Lagrangian Hessian W (lambda = y*dsc, objective factor fsc)
        // record: a = lambda row (m: objective, m+1: padding), b = x0, c = L index
        {
          const double fsc_ = ctl.fsc;
#define SP_LAM(lr) (((lr) < (unsigned)m) ? yd[lr] : (((lr) == (unsigned)m) ? fsc_ : 0.0))
          SP_STREAM16(P.W, SP_COEF(o_) * V[o_.z & 0x7fffu] * SP_LAM(o_.z >> 16) * xe[o_.w & 0xffffu],
                      Kg[o_.w >> 16] += acc_;)
#undef SP_LAM
        }
        // equality border + right-hand-side entries: one record per border slot
        // (slot | row<<16, L index; slot 0xffff: the rhs entry of the row)
        for (int e = tid; e < P.n_border; e += NT) {
          const uint2 b = __ldg(P.border + e);
          const int i = (int)(b.x >> 16), sl = (int)(b.x & 0xffffu);
          Kg[b.y] = (sl == 0xffff) ? -(g[i] - beq[i]) : dsc[i] * jval[sl];
        }
        SP_STREAM8(P.C, 0x10000u, SP_VC(jval, wv),
                   { Kg[(o_.y >> 17) & 0x1fffu] = -(gf[o_.y & 0xffffu] + acc_); })
        sp_fence_async();                    // Kg reaches L2 (the fence carries MEMBAR.ALL.GPU) and is
        __syncthreads();                     // ordered before the async-proxy read; no L1 invalidation
      }
      for (;;) {
        // stage K (TMA bulk load, mbarrier), then shift the diagonal by (delta_w, -delta_c)
        if (tid == 0) {
          sp_mbar_expect_tx(&kbar, (unsigned)(P.Lsz * 8));
          sp_bulk_g2s(LK, Kg, (unsigned)(P.Lsz * 8), &kbar);
        }
        sp_mbar_wait(&kbar, kphase & 1u);
        ++kphase;
        for (int pj = tid; pj < N; pj += NT) {          // vdiag: L index of the diagonal | eq-row<<15
          const unsigned dd = __ldg(P.vdiag + pj);
          if (dd & 0x8000u) { LK[dd & 0x7fffu] = -ctl.delta_c; diag0[pj] = ctl.delta_c; }
          else { const double v = LK[dd] + ctl.delta_w; LK[dd] = v; diag0[pj] = fabs(v); }
        }
        if (tid == 0) { ctl.fail = 0; ctl.eq_fail = 0; }
        __syncthreads();
        TICK(6);
        sp_factor(T, P, S, &ctl, fflags, O.inertia_mode, tracing ? phase_cyc : nullptr);
        TICK(7);
        if (!ctl.fail) break;
        // the failed attempt wrote LK through the generic proxy; the next staging overwrites it
        // through the async proxy (cp.async.bulk): every writer orders its writes before the
        // barrier that precedes the copy (PTX memory model, proxy fence)
        sp_fence_async();
        if (tid == 0) {
          if (ctl.eq_fail) ctl.delta_c = DELTA_C_VAL * pow(mu, DELTA_C_EXP);
          if (ctl.first_try) {
            ctl.delta_w = (ctl.delta_w_last == 0.0) ? DELTA_W0
                          : fmax(DELTA_W_MIN, KAPPA_W_MINUS * ctl.delta_w_last);
            ctl.first_try = 0;
          } else {
            ctl.delta_w *= (ctl.delta_w_last == 0.0) ? KAPPA_W_PLUS_FIRST : KAPPA_W_PLUS;
          }
        }
        __syncthreads();
        if (ctl.delta_w > DELTA_W_MAX) break;
      }
      if (ctl.fail) {
        if (tid == 0) { ctl.status = OMG_ERROR_IN_STEP_COMPUTATION; ctl.iter = iter; }
        __syncthreads();
        break;
      }
      if (tid == 0 && ctl.delta_w > 0.0) ctl.delta_w_last = ctl.delta_w;
      // ---- I9: solve ------------------------------------------------------------------
      sp_back_solve(T, P, S, xt, tracing ? phase_cyc : nullptr);        // xt is free here: u (permuted) -> xt[0..N)
      for (int j = tid; j < n; j += NT) dx[j] = xt[P.pos_var[j]];
      for (int k = tid; k < n_eq; k += NT) dx[n + k] = xt[P.pos_eq[k]];
      if (tid == 0) dx[n + n_eq] = 0.0;
      __syncthreads();
      TICK(10);
      // ---- I10: ds, dy, dz, fraction to the boundary -----------------------------------
      double sv[4];
      const int sop[4] = {OP_MIN, OP_MIN, OP_SUM, OP_SUM};
      sv[0] = 1.0; sv[1] = 1.0; sv[2] = 0.0; sv[3] = 0.0;
      // J dx through the row ELL -> ds (temporarily)
      // (the Jacobian values were overwritten by the factor: J dx straight from the terms;
      //  record: a = x0, b = column, c = row)
      SP_STREAM16(P.R, SP_COEF(o_) * V[o_.z & 0x7fffu] * xe[o_.z >> 16] * dx[o_.w & 0xffffu], ds[o_.w >> 16] = acc_;)
      __syncthreads();
#pragma unroll 2
      for (int i = tid; i < m; i += NT) {
        const int r = rt[i];
        const double jd = dsc[i] * ds[i];
        const double si = s[i], gi_ = g[i], sl_ = sL[i], su_ = sU[i], zl_ = zL[i], zu_ = zU[i], sg_ = sig[i], yi_ = y[i];
        if (r & 4) {
          ds[i] = 0.0; dy[i] = dx[n + eqidx[i]]; dzL[i] = 0.0; dzU[i] = 0.0;
        } else {
          const double dsi = jd + (gi_ - si);
          double ph = 0.0, a = 0.0, b = 0.0;
          if (r & 1) { const double dl = si - sl_; const double z = zl_; ph -= mu / dl;
            a = mu / dl - z - (z / dl) * dsi;
            if (dsi < 0.0) sv[0] = fmin(sv[0], -tau * dl / dsi);
            if (a < 0.0) sv[1] = fmin(sv[1], -tau * z / a); dzL[i] = a; }
          if (r & 2) { const double du = su_ - si; const double z = zu_; ph += mu / du;
            b = mu / du - z + (z / du) * dsi;
            if (dsi > 0.0) sv[0] = fmin(sv[0], tau * du / dsi);
            if (b < 0.0) sv[1] = fmin(sv[1], -tau * z / b); }
          ds[i] = dsi; dzU[i] = b;
          dy[i] = sg_ * dsi + ph - yi_;
          sv[2] += ph * dsi;
        }
      }
      for (int j = tid; j < n; j += NT) sv[2] += gf[j] * dx[j];
      block_reduce<4>(sv, sop, red);
      const double a_p = sv[0], a_d = sv[1], gphi = sv[2];
      TICK(11);
      // ---- I11: filter line search ----------------------------------------------------
      const double theta0 = ctl.theta, phi0 = ctl.phi;
      double a_min;
      if (gphi < 0.0) {
        a_min = fmin(GAMMA_THETA, GAMMA_PHI * theta0 / (-gphi));
        if (theta0 <= ctl.theta_min)
          a_min = fmin(a_min, DELTA_LS * pow(theta0, S_THETA) / pow(-gphi, S_PHI));
      } else a_min = GAMMA_THETA;
      a_min *= GAMMA_ALPHA;
      double alpha = a_p;
      bool accepted = false, ftype = false;
      double ft = 0.0;
      int n_ls = 0;
      while (alpha >= a_min && n_ls < MAX_LS) {
        ++n_ls;
        for (int j = tid; j < n; j += NT) xt[j] = xe[j] + alpha * dx[j];
        if (tid == 0) xt[n] = 1.0;
        __syncthreads();
        SP_STREAM16(P.G, SP_VG(xt), gt[o_.w >> 16] = acc_;)
        __syncthreads();
        double tv[3];
        const int top[3] = {OP_SUM, OP_SUM, OP_SUM};
        tv[0] = 0.0; tv[1] = 0.0; tv[2] = 0.0;
#pragma unroll 2
        for (int i = tid; i < m; i += NT) {
          const int r = rt[i];
          const double gi = dsc[i] * gt[i];
          const double be_ = beq[i], s_ = s[i], ds_ = ds[i], sl_ = sL[i], su_ = sU[i];
          gt[i] = gi;
          if (r & 4) tv[0] += fabs(gi - be_);
          else {
            const double si = s_ + alpha * ds_;
            st[i] = si;
            tv[0] += fabs(gi - si);
            if (r & 1) tv[1] += log(si - sl_);
            if (r & 2) tv[1] += log(su_ - si);
          }
        }
        for (int t = tid; t < T.n_f; t += NT) tv[2] += sp_eval_range(T.Ft, t, t + 1, V, xt);
        block_reduce<3>(tv, top, red);
        ft = ctl.fsc * tv[2];
        const double tht = tv[0], pht = ft - mu * tv[1];
        bool ok = isfinite(pht) && isfinite(tht) && tht <= ctl.theta_max;
        if (ok) {
          const int nf = ctl.nfilt;
          for (int q = 0; q < nf; ++q)
            if (!(tht < filt[2 * q] || pht < filt[2 * q + 1])) { ok = false; break; }
        }
        ftype = false;
        if (ok) {
          const bool switching = (theta0 <= ctl.theta_min && gphi < 0.0 &&
                                  alpha * pow(-gphi, S_PHI) > DELTA_LS * pow(theta0, S_THETA));
          if (switching) { ok = cmp_le(pht - phi0, ETA_PHI * alpha * gphi, phi0); ftype = ok; }
          else ok = cmp_le(tht, (1.0 - GAMMA_THETA) * theta0, theta0) ||
                    cmp_le(pht - phi0, -GAMMA_PHI * theta0, phi0);
        }
        if (ok) { accepted = true; break; }
        alpha *= 0.5;
      }
      bool soft = false;
      if (!accepted && O.soft_resto) {
        // ---- soft restoration (IPOPT): accept a step along the same direction if it reduces
        // the primal-dual error of the barrier problem
        __syncthreads();
        SP_STREAM16(P.J, SP_VJ(xe), jval[o_.w & 0xffffu] = acc_;)      // (the factor is dead by now)
        __syncthreads();
        double pv[1]; const int pop[1] = {OP_SUM};
        pv[0] = 0.0;
        for (int i = tid; i < m; i += NT) {
          const int r = rt[i];
          if (r & 4) { pv[0] += fabs(g[i] - beq[i]); continue; }
          const double si = s[i];
          double zl = 0.0, zu = 0.0, acc = fabs(g[i] - si);
          if (r & 1) { zl = zL[i]; acc += fabs((si - sL[i]) * zl - mu); }
          if (r & 2) { zu = zU[i]; acc += fabs((sU[i] - si) * zu - mu); }
          pv[0] += acc + fabs(-y[i] - zl + zu);
        }
        SP_STREAM8(P.C, 0x10000u, SP_VC(jval, yd), pv[0] += fabs(gf[o_.y & 0xffffu] + acc_);)
        block_reduce<1>(pv, pop, red);
        const double pd0 = pv[0];
        alpha = a_p;
        for (int n_try = 0; n_try < 12; ++n_try) {
          for (int j = tid; j < n; j += NT) xt[j] = xe[j] + alpha * dx[j];
          if (tid == 0) xt[n] = 1.0;
          __syncthreads();
          const double az = fmin(alpha, a_d);
          pv[0] = 0.0;
          // trial Jacobian -> jt (scratch), trial g -> gt, trial y -> wv
          SP_STREAM16(P.J, SP_VJ(xt), jt[o_.w & 0xffffu] = acc_;)
          SP_STREAM16(P.G, SP_VG(xt), gt[o_.w >> 16] = acc_;)
          __syncthreads();
          for (int i = tid; i < m; i += NT) {
            const int r = rt[i];
            const double gi = dsc[i] * gt[i];
            gt[i] = gi;
            const double yt = y[i] + alpha * dy[i];
            wv[i] = yt * dsc[i];
            if (r & 4) { pv[0] += fabs(gi - beq[i]); continue; }
            const double si = s[i] + alpha * ds[i];
            st[i] = si;
            double zl = 0.0, zu = 0.0, acc = fabs(gi - si);
            if (r & 1) { zl = zL[i] + az * dzL[i]; acc += fabs((si - sL[i]) * zl - mu); }
            if (r & 2) { zu = zU[i] + az * dzU[i]; acc += fabs((sU[i] - si) * zu - mu); }
            pv[0] += acc + fabs(-yt - zl + zu);
          }
          __syncthreads();
          SP_STREAM8(P.C, 0x10000u, SP_VC(jt, wv),
                     { const int c_ = o_.y & 0xffffu;
                       pv[0] += fabs(ctl.fsc * sp_eval_range(T.DFt, T.dfptr[c_], T.dfptr[c_ + 1], V, xt) + acc_); })
          block_reduce<1>(pv, pop, red);
          if (isfinite(pv[0]) && pv[0] <= SOFT_RESTO_FACTOR * pd0) {
            double fv[1]; fv[0] = 0.0;
            for (int t = tid; t < T.n_f; t += NT) fv[0] += sp_eval_range(T.Ft, t, t + 1, V, xt);
            block_reduce<1>(fv, pop, red);
            ft = ctl.fsc * fv[0];
            accepted = true; soft = true; ftype = true;
            break;
          }
          alpha *= 0.5;
        }
      }
      if (!accepted) {
        if (ctl.n_restart < O.max_restarts) {
          __syncthreads();
          const double mu_r = O.restart_mu;
          for (int i = tid; i < m; i += NT) {
            const int r = rt[i];
            double si = g[i];
            if (r & 1) si = fmax(si, sL[i] + O.restart_push * fmax(1.0, fabs(sL[i])));
            if (r & 2) si = fmin(si, sU[i] - O.restart_push * fmax(1.0, fabs(sU[i])));
            s[i] = si; y[i] = 0.0; yd[i] = 0.0;
            if (r & 1) zL[i] = mu_r / (si - sL[i]);
            if (r & 2) zU[i] = mu_r / (sU[i] - si);
          }
          if (tid == 0) {
            ctl.n_restart += 1; ctl.mu = mu_r; ctl.tau = fmax(TAU_MIN, 1.0 - mu_r);
            ctl.nfilt = 0; ctl.theta_max = -1.0; ctl.delta_w_last = 0.0;
          }
          __syncthreads();
          continue;
        }
        if (tid == 0) { ctl.status = OMG_RESTORATION_FAILED; ctl.iter = iter; }
        __syncthreads();
        break;
      }
      __syncthreads();
      if (tid == 0) {
        if (soft) ctl.nfilt = 0;
        if (!ftype) {
          const double th = (1.0 - GAMMA_THETA) * theta0, ph = phi0 - GAMMA_PHI * theta0;
          int nf = 0;
          for (int q = 0; q < ctl.nfilt; ++q)
            if (!(filt[2 * q] >= th && filt[2 * q + 1] >= ph)) {
              filt[2 * nf] = filt[2 * q]; filt[2 * nf + 1] = filt[2 * q + 1]; ++nf; }
          if (nf >= MAXF) {
            for (int q = 1; q < nf; ++q) { filt[2 * (q - 1)] = filt[2 * q]; filt[2 * (q - 1) + 1] = filt[2 * q + 1]; }
            --nf;
          }
          filt[2 * nf] = th; filt[2 * nf + 1] = ph; ++nf;
          ctl.nfilt = nf;
        }
        ctl.f = ft; ctl.alpha = alpha;
      }
      TICK(12);
      // ---- I12: accept ----------------------------------------------------------------------
      for (int j = tid; j <= n; j += NT) xe[j] = (j < n) ? xt[j] : 1.0;
#pragma unroll 2
      for (int i = tid; i < m; i += NT) {
        const int r = rt[i];
        const double gt_ = gt[i], y_ = y[i], dy_ = dy[i], d_ = dsc[i], st_ = st[i], sl_ = sL[i], su_ = sU[i],
                     zl_ = zL[i], zu_ = zU[i], dzl_ = dzL[i], dzu_ = dzU[i];
        g[i] = gt_;
        { const double yn = y_ + alpha * dy_; y[i] = yn; yd[i] = yn * d_; }
        if (!(r & 4)) {
          const double si = st_;
          s[i] = si;
          if (r & 1) { const double dl = si - sl_; double z = zl_ + a_d * dzl_;
            z = fmin(fmax(z, mu / (KAPPA_SIGMA * dl)), KAPPA_SIGMA * mu / dl); zL[i] = z; }
          if (r & 2) { const double du = su_ - si; double z = zu_ + a_d * dzu_;
            z = fmin(fmax(z, mu / (KAPPA_SIGMA * du)), KAPPA_SIGMA * mu / du); zU[i] = z; }
        }
      }
      __syncthreads();
    }  // iterations

    // ---- write results -------------------------------------------------------------------
    __syncthreads();
    for (int i = tid; i < n; i += NT) A.x[(size_t)inst * n + i] = xe[i];
    for (int i = tid; i < m; i += NT) A.lam[(size_t)inst * m + i] = y[i] * dsc[i] / ctl.fsc;
    if (tracing && tid == 0) {
      TICK(13);
      double* tr = A.trace + (TRACE_ROWS - 2) * TRACE_COLS;
      for (int k = 0; k < NPHASE; ++k) tr[k] = phase_cyc[k];
    }
    if (tid == 0) {
      A.f[inst] = ctl.f / ctl.fsc;
      A.status[inst] = ctl.status;
      A.iters[inst] = ctl.iter;
    }
    __syncthreads();
  }
}
