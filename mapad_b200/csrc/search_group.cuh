// search_group.cuh — K2: the search kernel.  One read per lane GROUP (G consecutive lanes of a warp; G = 1 .. 32 is a
// compile-time choice), persistent groups pulling reads from a global queue (longest reads first), and one flat loop in
// which every iteration pops and expands ONE frame of the group's current read.  A read is never restarted: its state
// grows in 256 KiB chunks taken from a pool in HBM until the reference's own limits (STACK_LIMIT / EDIT_TREE_LIMIT,
// /root/reference/src/map/mapping.rs:52-54) are reached.
//
// Per-read state and where it lives:
//   * min-max heap of (score, node) pairs — 64-byte FAMILY lines: the line owned by the node at 1-based position h of
//     an odd (max) level holds the two children 2h, 2h+1 and the four grandchildren 4h .. 4h+3 of h, i.e. exactly the six
//     entries one trickle-down step of MinMaxHeap::pop_max looks at.  The first TOPL lines (positions 1 .. 63 for
//     TOPL = 11) sit in shared memory, the rest in pooled chunks.  The logical array — and therefore every tie — is
//     that of min_max_heap::MinMaxHeap (SURVEY Appendix A4/A9); only the physical placement differs.
//   * edit tree = frame storage: one 32-byte node (one sector) per accepted child, both layouts (wide: 40-bit
//     interval fields), bump-allocated, slab free list through `parent` (backtrack_tree.rs:34-53)
//   * hits: std BinaryHeap emulation in a small per-group array
// The sequential semantics are those of search_core.cuh::search_step (mapping.rs:932-1383): all lanes of a group run
// the same decisions on the same data; the lanes share the memory work (see the cooperative sections below).
#pragma once
#include "search_core.cuh"
#include "simt.cuh"

namespace mapad {

#ifndef MAPAD_GCHUNK_SHIFT
#define MAPAD_GCHUNK_SHIFT 18u  // 256 KiB chunks; the emulation tests also build a 4 KiB variant to stress the chunk tables
#endif
#define MAPAD_GCHUNK_BYTES (1u << MAPAD_GCHUNK_SHIFT)
#define MAPAD_GPOOL_EMPTY 0xffffffffu

// Free chunk ids live in MAPAD_GPOOL_SHARDS independent Treiber stacks (heads 128 bytes apart; the 32-bit tag in the upper
// half of a head defeats ABA).  A group works on the shard its slot number selects and scans the others only when that one
// is empty, so that the thousands of groups of all launches in flight do not hammer one atomic (measured: with a single
// stack the compare-and-swap loop accounted for 37 % of the stall samples of a saturated launch, profiles/r2_*).
#define MAPAD_GPOOL_SHARDS 256u
#define MAPAD_GPOOL_HEAD_STRIDE 16u  // in 8-byte words
struct GChunkPool {
  uint8_t* base;
  uint32_t n_chunks;
  unsigned long long* heads;  // MAPAD_GPOOL_SHARDS x MAPAD_GPOOL_HEAD_STRIDE words; word 8 of shard 0: the pressure deadline
  uint32_t* next;
};
// Admission control.  A group that finds the whole pool empty while its read needs a chunk publishes "pressure until
// now + 2 ms" (and keeps renewing it while it waits); groups about to START a read hold back while pressure is on.
// Reads in flight then finish and free memory instead of competing with newcomers that would only be handed back later
// (measured on hg19-scale chunks without it: 5 % of the reads were deferred and re-run, profiles/r2_summary.md).
#define MAPAD_PRESSURE_HOLD_NS 2000000ull
MAPAD_DEV unsigned long long dev_now_ns() {
#if defined(__CUDA_ARCH__)
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
#else
  static unsigned long long fake = 0;
  fake += 1000;
  return fake;
#endif
}
MAPAD_DEV volatile unsigned long long* gpool_pressure(const GChunkPool& p) { return reinterpret_cast<volatile unsigned long long*>(p.heads + 8); }

MAPAD_DEV uint32_t gpool_pop(const GChunkPool& p, uint32_t shard) {
  unsigned long long* head = p.heads + (size_t)shard * MAPAD_GPOOL_HEAD_STRIDE;
#if defined(__CUDA_ARCH__)
  unsigned long long old = *reinterpret_cast<volatile unsigned long long*>(head);
  while (true) {
    const uint32_t idx = (uint32_t)old;
    if (idx == MAPAD_GPOOL_EMPTY) return idx;
    const uint32_t nxt = reinterpret_cast<volatile uint32_t*>(p.next)[idx];
    const unsigned long long neu = (((old >> 32) + 1ull) << 32) | nxt;
    const unsigned long long seen = atomicCAS(head, old, neu);
    if (seen == old) return idx;
    old = seen;
  }
#else
  const uint32_t idx = (uint32_t)*head;
  if (idx == MAPAD_GPOOL_EMPTY) return idx;
  *head = p.next[idx];
  return idx;
#endif
}
MAPAD_DEV uint32_t gpool_acquire(const GChunkPool& p, uint32_t hint) {
  for (uint32_t k = 0; k < MAPAD_GPOOL_SHARDS; ++k) {
    const uint32_t got = gpool_pop(p, (hint + k) & (MAPAD_GPOOL_SHARDS - 1u));
    if (got != MAPAD_GPOOL_EMPTY) return got;
  }
  return MAPAD_GPOOL_EMPTY;
}
MAPAD_DEV void gpool_release(const GChunkPool& p, uint32_t idx, uint32_t hint) {
  unsigned long long* head = p.heads + (size_t)(hint & (MAPAD_GPOOL_SHARDS - 1u)) * MAPAD_GPOOL_HEAD_STRIDE;
#if defined(__CUDA_ARCH__)
  unsigned long long old = *reinterpret_cast<volatile unsigned long long*>(head);
  while (true) {
    reinterpret_cast<volatile uint32_t*>(p.next)[idx] = (uint32_t)old;
    __threadfence();
    const unsigned long long neu = (((old >> 32) + 1ull) << 32) | idx;
    const unsigned long long seen = atomicCAS(head, old, neu);
    if (seen == old) return;
    old = seen;
  }
#else
  p.next[idx] = (uint32_t)*head;
  *head = idx;
#endif
}
// host-side helper shared with the emulation harness: chunk i starts in shard i % SHARDS
inline void gpool_init_host(uint32_t n_chunks, unsigned long long* heads, uint32_t* next) {
  for (uint32_t s = 0; s < MAPAD_GPOOL_SHARDS; ++s) heads[(size_t)s * MAPAD_GPOOL_HEAD_STRIDE] = s < n_chunks ? s : MAPAD_GPOOL_EMPTY;
  heads[8] = 0ull;  // pressure deadline
  for (uint32_t i = 0; i < n_chunks; ++i) next[i] = i + MAPAD_GPOOL_SHARDS < n_chunks ? i + MAPAD_GPOOL_SHARDS : MAPAD_GPOOL_EMPTY;
}

// Back-off while waiting for the pool (device: __nanosleep; emulation: let the other groups run).
#if !defined(__CUDA_ARCH__)
extern "C" void mapad_simt_emu_yield(void);
#endif
template <int G>
MAPAD_DEV void dev_backoff() {
#if defined(__CUDA_ARCH__)
  __nanosleep(2000);
#else
  if (G > 1) mapad_simt_emu_yield();
#endif
}

// ---- family layout of the min-max heap ----------------------------------------------------------
// 1-based position x -> (line, slot).  Positions 1..3 live in line 0 (slots 0..2).  A position on an even level >= 2
// is a CHILD of its owner x >> 1 (slots 0, 1), one on an odd level >= 3 a GRANDCHILD of its owner x >> 2 (slots 2..5).
// Owners are the positions of odd levels; the owner o of level lo gets line  o - C(lo),  C(lo) = (2^(lo+1) - 1) / 3.
struct HLoc { uint32_t line, slot; };
MAPAD_HD int clz32(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return __clz((int)x);
#else
  return __builtin_clz(x);
#endif
}
MAPAD_DEV int ffs32(uint32_t x) {  // 1-based index of the lowest set bit, 0 if none
#if defined(__CUDA_ARCH__)
  return __ffs((int)x);
#else
  return __builtin_ffs((int)x);
#endif
}
// Straight-line code on purpose: the lanes of a group call this with different positions (the ancestor chain of a push), and a
// branch per special case made them diverge (heap_loc + line_ptr: 24 % of all warp instructions at 13 of 32 active threads,
// profiles/r2_g32_wide_50Mbp_hotspots.txt).
MAPAD_HD HLoc heap_loc(uint32_t x) {
  const bool small = x < 4u;
  const int lvl = 31 - clz32(x);
  const uint32_t odd = (uint32_t)lvl & 1u;
  const uint32_t owner = x >> (1u + odd);
  const uint32_t slot = odd ? 2u + (x & 3u) : (x & 1u);
  const int lo = lvl - 1 - (int)odd;                              // < 0 only for x < 4
  const uint32_t c = 0x55555555u & ((2u << (lo < 0 ? 0 : lo)) - 1u);
  return HLoc{small ? 0u : owner - c, small ? x - 1u : slot};
}
// number of lines that positions 1..n occupy
MAPAD_HD uint32_t heap_lines_for(uint32_t n) {
  if (n < 4u) return 1u;
  const int lvl = 31 - clz32(n);
  // the last position of the deepest even level <= lvl decides
  const uint32_t x = (lvl & 1) ? ((1u << lvl) - 1u) : n;
  return heap_loc(x).line + 1u;
}

struct alignas(16) ulonglong2_compat { unsigned long long a, b; };
MAPAD_DEV float u32_as_f32(uint32_t u) {
#if defined(__CUDA_ARCH__)
  return __uint_as_float(u);
#else
  union { uint32_t u; float f; } c; c.u = u; return c.f;
#endif
}

template <bool WIDE> struct GNodeOf { using type = NodeT<false>; };
template <> struct GNodeOf<true> { using type = NodeW32; };

#define MAPAD_POOL_TIMEOUT_FLAG 4u   // Cursors::overflow bit: a group found no base chunks within the start-up patience
#define MAPAD_PATIENCE_MAX 10000000u // back-off rounds of 2 us: 20 s
// Everything one launch needs (passed by value as the kernel parameter).
template <bool WIDE>
struct GroupLaunch {
  DevIndex ix;
  DevParams P;
  ReadBatch rb;
  const float* bound_table;
  const PenRow* delta;
  const float* dcomp;
  GChunkPool pool;
  uint32_t* tables;        // n_groups x (nt + ht)
  uint32_t nt, ht;
  HitTmp* hit_base;        // n_groups x MAPAD_MAX_HITS
  uint32_t max_nodes, max_heap;
  const uint32_t* work_list;  // read ids in processing order (longest first), or nullptr
  uint32_t n_work;
  uint32_t* deferred_list;
  Cursors* cur;
  ReadMid* mid;
  mapad_hit* hit_pool;
  uint32_t hit_cap;
  mapad_edit_op* op_pool;
  uint32_t op_cap;
  uint32_t iter_budget;    // profiling aid: stop every group after this many expansions (0 = off)
  uint32_t flags_or;       // ORed into ReadMid::flags (bit 1: the read went through a retry launch)
  uint32_t patient;        // 1: never hand a read back, wait for the pool (last-resort launches)
  uint32_t prefetch;       // latency hiding for deep heaps (bit 0: next family lines of a trickle-down, bit 1: the two
                           // occ blocks of the popped frame while its heap is being repaired); see MAPAD_TRICKLE_PREFETCH
};


// Workspace of one group (search_core.cuh's workspace concept).  Every lane of the group holds the same copy and makes
// the same calls; pool operations are done once, by lane 0, and broadcast.
template <bool WIDE, int G, int TOPL>
struct GroupWorkspace {
  using Node = typename GNodeOf<WIDE>::type;
  static constexpr uint32_t NPC_SHIFT = MAPAD_GCHUNK_SHIFT - 5u;  // nodes per chunk (32 B each)
  static constexpr uint32_t LPC_SHIFT = MAPAD_GCHUNK_SHIFT - 6u;  // heap lines per chunk (64 B each)
  // launch-wide constants are read through `a` (kernel parameter space) instead of being copied into registers
  const GroupLaunch<WIDE>* a;
  uint32_t slot;         // this group's number: selects its chunk table, hit array and home shard of the pool
  uint32_t frames;       // frames popped so far by the current read (also sets the patience when the pool is dry)
  uint32_t n_node_chunks, n_heap_chunks;
  uint32_t heap_hi;      // logical heap indices below this are known to be backed by memory
  Node* node0;           // chunk 0 of each kind is owned for good: no table lookup for small searches
  HeapEnt* heap0;
  HeapEnt* top;          // shared memory: TOPL lines of 8 entries
  int gl;                // lane in group

  // chunk table of this group: [0, nt) node chunks, [nt, nt + ht) heap chunks
  MAPAD_DEV uint32_t* table() const { return a->tables + (size_t)slot * (a->nt + a->ht); }
  MAPAD_DEV HitTmp* hits() const { return a->hit_base + (size_t)slot * MAPAD_MAX_HITS; }
  MAPAD_DEV uint32_t shard() const { return (slot * 2654435761u) >> 24; }  // spreads neighbouring groups over the 256 shards
  // How long (in 2 us back-off rounds) the group waits for a chunk when the pool is dry: one round per frame already
  // popped, at least 0.4 ms — young reads step aside first.  (Ten rounds per frame were measured: reads then sleep on their
  // memory for seconds and the GPU idles.)
  MAPAD_DEV uint32_t patience() const {
    if (a->patient || frames >= MAPAD_PATIENCE_MAX) return MAPAD_PATIENCE_MAX;
    uint32_t p = frames < 200u ? 200u : frames;
#if !defined(__CUDA_ARCH__)
    if (G == 1) p = 0;               // the emulation runs per-thread groups one after the other: nobody to wait for
    else if (p > 2000u) p = 2000u;   // keep the emulated waits short
#endif
    return p;
  }

  MAPAD_DEV Node& node(uint32_t id) const {
    if (id < (1u << NPC_SHIFT)) return node0[id];
    const uint32_t c = table()[id >> NPC_SHIFT];
    return reinterpret_cast<Node*>(a->pool.base + ((size_t)c << MAPAD_GCHUNK_SHIFT))[id & ((1u << NPC_SHIFT) - 1u)];
  }
  // The pooled storage is addressed by the plain line number (lines < TOPL are unused there).  Selects instead of branches
  // (see heap_loc); only the chunk-table lookup of lines beyond chunk 0 is conditional.
  MAPAD_DEV HeapEnt* line_ptr(uint32_t line) const {
    static_assert((uint32_t)TOPL <= (1u << LPC_SHIFT), "the shared-memory lines are a prefix of chunk 0's line numbers");
    const bool in_top = line < (uint32_t)TOPL;
    const bool in0 = line < (1u << LPC_SHIFT);
    uint32_t c = 0u;
    if (!in0) c = table()[a->nt + (line >> LPC_SHIFT)];
    uint8_t* chunk = in0 ? reinterpret_cast<uint8_t*>(heap0) : a->pool.base + ((size_t)c << MAPAD_GCHUNK_SHIFT);
    uint8_t* base = in_top ? reinterpret_cast<uint8_t*>(top) : chunk;
    const uint32_t idx = in0 ? line : (line & ((1u << LPC_SHIFT) - 1u));
    return reinterpret_cast<HeapEnt*>(base + ((size_t)idx << 6));
  }
  MAPAD_DEV Node* node_ptr(uint32_t id) const {
    const bool in0 = id < (1u << NPC_SHIFT);
    uint32_t c = 0u;
    if (!in0) c = table()[id >> NPC_SHIFT];
    uint8_t* chunk = in0 ? reinterpret_cast<uint8_t*>(node0) : a->pool.base + ((size_t)c << MAPAD_GCHUNK_SHIFT);
    return reinterpret_cast<Node*>(chunk) + (in0 ? id : (id & ((1u << NPC_SHIFT) - 1u)));
  }
  MAPAD_DEV HeapEnt* slot_ptr(uint32_t i0) const {  // 0-based logical index
    const HLoc l = heap_loc(i0 + 1u);
    return line_ptr(l.line) + l.slot;
  }
  // The pool is shared by every group of every launch on the device.  When it is dry the group waits for chunks that
  // finishing reads give back — the longer, the more work its own read has already absorbed (patience is set by the caller
  // in proportion to the frames popped so far), so that young reads step aside first (they are handed back and re-run).
  MAPAD_DEV uint32_t acquire_chunk() const {
    uint32_t got = MAPAD_GPOOL_EMPTY;
    if (gl == 0) {
      got = gpool_acquire(a->pool, shard());
      if (got == MAPAD_GPOOL_EMPTY) {
        const uint32_t rounds = patience();
        for (uint32_t w = 0; got == MAPAD_GPOOL_EMPTY && w < rounds; ++w) {
          *gpool_pressure(a->pool) = dev_now_ns() + MAPAD_PRESSURE_HOLD_NS;  // newcomers hold back while this group waits
          dev_backoff<G>();
          got = gpool_acquire(a->pool, shard());
        }
      }
    }
    return Grp<G>::shfl(got, 0);
  }
  // Group start: both base chunks or none, and no pressure while waiting.  Launches of several handles share the pool and
  // each may start up to n_chunks / 4 groups, so two launches can hold every chunk as base chunks; the others' groups then
  // wait until those launches exit.  Groups that each held one chunk while waiting for a second could together hold the
  // rest of the pool, and pressure published by a group that runs no read would hold back the groups that own the pool
  // (they wait before every next read) — either way nobody returns a chunk until the 20 s patience runs out (MAPAD_ELIMIT).
  MAPAD_DEV bool acquire_base(uint32_t& c_nodes, uint32_t& c_heap) const {
    uint32_t n = MAPAD_GPOOL_EMPTY, h = MAPAD_GPOOL_EMPTY;
    if (gl == 0) {
      for (uint32_t w = 0; w < MAPAD_PATIENCE_MAX; ++w) {
        n = gpool_acquire(a->pool, shard());
        if (n != MAPAD_GPOOL_EMPTY) {
          h = gpool_acquire(a->pool, shard());
          if (h != MAPAD_GPOOL_EMPTY) break;
          gpool_release(a->pool, n, shard());
          n = MAPAD_GPOOL_EMPTY;
        }
        dev_backoff<G>();
      }
    }
    c_nodes = Grp<G>::shfl(n, 0);
    c_heap = Grp<G>::shfl(h, 0);
    return c_heap != MAPAD_GPOOL_EMPTY;
  }
  MAPAD_DEV bool ensure_node(uint32_t id) {
    if (id >= a->max_nodes) return false;
    const uint32_t c = id >> NPC_SHIFT;
    if (c < n_node_chunks) return true;
    if (c >= a->nt) return false;
    const uint32_t got = acquire_chunk();
    if (got == MAPAD_GPOOL_EMPTY) return false;
    table()[c] = got;
    n_node_chunks = c + 1;
    return true;
  }
  MAPAD_DEV bool ensure_heap(uint32_t n0) {  // room for logical index n0
    if (n0 < heap_hi) return true;           // backed before (the heap shrinks and regrows around its high-water mark)
    if (n0 >= a->max_heap) return false;
    const HLoc l = heap_loc(n0 + 1u);
    if (l.line < (uint32_t)TOPL) { heap_hi = n0 + 1u; return true; }
    const uint32_t c = l.line >> LPC_SHIFT;
    if (c < n_heap_chunks) { heap_hi = n0 + 1u; return true; }
    if (c >= a->ht) return false;
    const uint32_t got = acquire_chunk();
    if (got == MAPAD_GPOOL_EMPTY) return false;
    table()[a->nt + c] = got;
    n_heap_chunks = c + 1;
    heap_hi = n0 + 1u;
    return true;
  }
  MAPAD_DEV uint32_t min_cap() const { return a->max_nodes; }
  MAPAD_DEV void release_base() const {  // group exit: the two base chunks go back to the pool
    if (gl == 0) { gpool_release(a->pool, table()[0], shard()); gpool_release(a->pool, table()[a->nt], shard()); }
  }
  MAPAD_DEV void release_extra() {  // keep chunk 0 of each kind
    if (gl == 0) {
      uint32_t* t = table();
      for (uint32_t c = n_node_chunks; c > 1; --c) gpool_release(a->pool, t[c - 1], shard());
      for (uint32_t c = n_heap_chunks; c > 1; --c) gpool_release(a->pool, t[a->nt + c - 1], shard());
    }
    n_node_chunks = 1;
    n_heap_chunks = 1;
    heap_hi = 0;
  }
  struct Store {
    const GroupWorkspace* w;
    MAPAD_DEV HeapEnt get(uint32_t i) const { return *w->slot_ptr(i); }
    MAPAD_DEV void set(uint32_t i, HeapEnt e) const { *w->slot_ptr(i) = e; }
  };
  MAPAD_DEV Store heap() const { return Store{this}; }
};

// FmdExtIterator for a lane group (dev_index.cuh::extend_all, fmd_index.rs:117-182): the two occ blocks hold 8 (narrow) or
// 16 (wide) words of 2-bit codes; with G >= 8 lanes 0..3 of every 8 count the words of the block of row lower - 1, lanes
// 4..7 those of the block of row lower + size - 1, and three xor-shuffles give every lane both totals (G = 4: two lanes
// per block, two shuffles).
template <bool WIDE, int G>
MAPAD_DEV void extend_all_group(const DevIndex& ix, const BiIv& in, BiIv out[4], int gl) {
  if (G < 4) { extend_all<WIDE>(ix, in, out); return; }
  constexpr int LPB = G >= 8 ? 4 : 2;          // lanes per block
  constexpr int NW = WIDE ? 8 : 4;             // code words per block
  constexpr int WPL = NW / LPB;                // words per lane
  const int role = gl & (2 * LPB - 1), blk = role / LPB, q = role % LPB;
  const bool have_lo = in.lower != 0;
  const uint64_t r_lo = have_lo ? in.lower - 1 : 0, r_hi = in.lower + in.size - 1;
  const uint64_t r = blk ? r_hi : r_lo;
  // this lane's code words
  uint32_t nC = 0, nG = 0, nT = 0;
  {
    const uint8_t* p = WIDE ? ix.occ() + (r >> 7) * 64 + 32 : ix.occ() + (r >> 6) * 32 + 16;
    const int npos = WIDE ? (int)(r & 127) + 1 : (int)(r & 63) + 1;
    const uint32_t* wp = reinterpret_cast<const uint32_t*>(p) + q * WPL;
#pragma unroll
    for (int k = 0; k < WPL; ++k) {
#if defined(__CUDA_ARCH__)
      const uint32_t w = __ldg(wp + k);
#else
      const uint32_t w = wp[k];
#endif
      count_word(w, npos - 16 * (q * WPL + k), nC, nG, nT);
    }
  }
  uint32_t packed = nC | (nG << 10) | (nT << 20);  // each count <= 128
#if defined(__CUDA_ARCH__)
  packed += Grp<G>::shfl_xor(packed, 1);
  if (LPB == 4) packed += Grp<G>::shfl_xor(packed, 2);
  const uint32_t other = Grp<G>::shfl_xor(packed, LPB);
#else
  packed += Grp<G>::shfl_xor_self(packed, 1, gl);
  if (LPB == 4) packed += Grp<G>::shfl_xor_self(packed, 2, gl);
  const uint32_t other = Grp<G>::shfl_xor_self(packed, LPB, gl);
#endif
  const uint32_t p_lo = blk ? other : packed, p_hi = blk ? packed : other;
  // per block: base counts + partial counts + the '$' / 'X' corrections of occ_finish
  uint64_t lo[4] = {0, 0, 0, 0}, hi[4];
  uint64_t s_lo = 0;
#pragma unroll
  for (int b = 0; b < 2; ++b) {
    if (b == 0 && !have_lo) continue;
    const uint64_t rr = b ? r_hi : r_lo;
    const uint32_t pk = b ? p_hi : p_lo;
    uint64_t* c = b ? hi : lo;
    const uint32_t cC = pk & 1023u, cG = (pk >> 10) & 1023u, cT = pk >> 20;
    uint64_t bstart;
    int npos;
    bool flagged;
    if (!WIDE) {
      const U4 cn = load16(ix.occ() + (rr >> 6) * 32);
      bstart = (rr >> 6) << 6; npos = (int)(rr & 63) + 1;
      flagged = (cn.x >> 31) != 0;
      c[0] = cn.x & 0x7fffffffu; c[1] = cn.y; c[2] = cn.z; c[3] = cn.w;
    } else {
      const uint8_t* p = ix.occ() + (rr >> 7) * 64;
      const U4 c0 = load16(p), c1 = load16(p + 16);
      bstart = (rr >> 7) << 7; npos = (int)(rr & 127) + 1;
      const uint64_t a0 = (uint64_t)c0.x | ((uint64_t)c0.y << 32);
      flagged = (a0 >> 63) != 0;
      c[0] = a0 & 0x7fffffffffffffffull;
      c[1] = (uint64_t)c0.z | ((uint64_t)c0.w << 32);
      c[2] = (uint64_t)c1.x | ((uint64_t)c1.y << 32);
      c[3] = (uint64_t)c1.z | ((uint64_t)c1.w << 32);
    }
    uint32_t nA = (uint32_t)npos - cC - cG - cT;
    const uint64_t s0 = ix.m.sentinel_rows[0], s1 = ix.m.sentinel_rows[1];
    nA -= (uint32_t)(s0 >= bstart && s0 <= rr);
    nA -= (uint32_t)(s1 >= bstart && s1 <= rr);
    if (flagged) {
      const uint64_t upto = x_rows_upto(ix, rr);
      const uint64_t before = bstart == 0 ? 0 : x_rows_upto(ix, bstart - 1);
      nA -= (uint32_t)(upto - before);
    }
    c[0] += nA; c[1] += cC; c[2] += cG; c[3] += cT;
  }
  if (have_lo) s_lo = sentinels_upto(ix, r_lo);
  uint64_t l = in.lower_rev + (sentinels_upto(ix, r_hi) - s_lo);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c = 3 - k;
    const uint64_t sz = hi[c] - lo[c];
    out[k].lower = ix.m.less[c + 1] + lo[c];
    out[k].lower_rev = l;
    out[k].size = sz;
    l += sz;
  }
}

// ---------------------------------------------------------------------------------------------
// One read's search, executed by the G lanes of a group.  Memory discipline: the sequential state that lives in
// registers (heap length, slab cursors, best hit) is computed identically by every lane; heap entries, tree nodes and
// hits in memory are WRITTEN BY LANE 0 ONLY and read by all lanes, with a group barrier between a read phase and the
// write phase that follows it (and between a write phase and the next read phase).  For G = 1 the barriers vanish and
// this is a plain per-thread search.
// ---------------------------------------------------------------------------------------------
// Speculative prefetch of the heap lines the NEXT trickle-down step may need (it depends on which grandchild wins): with
// at least four lanes per read, lane b asks for the family line of grandchild b while the current step is being decided,
// so a descent through the pooled (HBM / L2) levels costs one memory latency per TWO steps.  Costs up to 4x the line
// traffic of those levels and ~25 instructions per step.  Run-time switch GroupLaunch::prefetch (host: MAPAD_TRICKLE_PREFETCH):
// on small references the kernel is issue-bound and the extra address arithmetic costs more than it hides (-6 % on cfg3,
// profiles/r2_summary.md); reads with heaps of 1e5 - 2e6 entries (hg19 scale) are bound by exactly these dependent
// round trips.  Only descents of heaps that reach into pooled memory (n >= 8 * TOPL) prefetch at all.
MAPAD_DEV void prefetch_line(const void* p) {
#if defined(__CUDA_ARCH__)
  asm volatile("prefetch.L1 [%0];" ::"l"(p));
#else
  (void)p;
#endif
}

struct HeapLine6 { HeapEnt x[6]; };
MAPAD_DEV HeapLine6 load_line6(const HeapEnt* ln) {  // three aligned 16-byte loads
  HeapLine6 r;
  const ulonglong2_compat* q = reinterpret_cast<const ulonglong2_compat*>(ln);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const ulonglong2_compat v = q[k];
    r.x[2 * k].score = u32_as_f32((uint32_t)v.a); r.x[2 * k].node = (uint32_t)(v.a >> 32);
    r.x[2 * k + 1].score = u32_as_f32((uint32_t)v.b); r.x[2 * k + 1].node = (uint32_t)(v.b >> 32);
  }
  return r;
}

template <bool WIDE, int G, int TOPL>
struct GroupSearch {
  using WS = GroupWorkspace<WIDE, G, TOPL>;
  using Node = typename WS::Node;
  WS ws;
  uint32_t heap_n, node_hi, free_head, tree_len, n_hits;
  float best_score;    // hits[0] of the BinaryHeap (its maximum) while n_hits > 0
  uint64_t best_size;
  uint32_t limit_hit;
  bool overflow;

  MAPAD_DEV void wr(HeapEnt* p, HeapEnt e) const { if (ws.gl == 0) *p = e; }
  MAPAD_DEV HeapEnt rd(uint32_t x1) const { const HLoc l = heap_loc(x1); return ws.line_ptr(l.line)[l.slot]; }
  MAPAD_DEV HeapEnt* ptr(uint32_t x1) const { const HLoc l = heap_loc(x1); return ws.line_ptr(l.line) + l.slot; }

  // Requests the two occ blocks the expansion of node `nd` will read (extend_all_group: rows lower - 1 and lower + size - 1
  // of the interval the extension starts from); even lanes ask for the first, odd lanes for the second.
  MAPAD_DEV void prefetch_occ(const Node& nd, int L) const {
    Frame f;
    node_load(nd, 0u, f);
    const bool forward = f.start <= L - f.start - f.len;
    const uint64_t lower = forward ? f.iv.lower_rev : f.iv.lower;
    const uint64_t r = (ws.gl & 1) ? lower + f.iv.size - 1u : (lower ? lower - 1u : 0u);
    const DevIndex& ix = ws.a->ix;
    prefetch_line(WIDE ? ix.occ() + (r >> 7) * 64 : ix.occ() + (r >> 6) * 32);
  }

  // MinMaxHeap::trickle_down_max from 1-based position h (2 or 3: the top of the max levels) with `e` in the hole;
  // n = number of elements.  One family line per step.
  // `occ_node` (optional): the node of the frame being popped; its two occ blocks are requested after the first round trip
  // of the descent, so that their latency overlaps the remaining steps (the node was requested before the descent began).
  MAPAD_DEV void trickle_max(uint32_t h, HeapEnt e, uint32_t n, const Node* occ_node, int L) {
    HeapEnt* hpos = ws.top + (h - 1u);
    uint32_t c_lo = 1u;  // C(level of h)
    bool synced = false;
    const uint32_t pf = n >= 8u * (uint32_t)TOPL ? ws.a->prefetch : 0u;
    bool occ_pending = (pf & 2u) != 0u && occ_node != nullptr;
    while (2u * h <= n) {
      const uint32_t line = h - c_lo;
      HeapEnt* ln = ws.line_ptr(line);
      const HeapLine6 f = load_line6(ln);
      if ((pf & 1u) && G >= 4 && ws.gl < 4) {
        const uint32_t g = 4u * h + (uint32_t)ws.gl;             // grandchild gl of h; its family line is needed if it has children
        const uint32_t gline = g - ((c_lo << 2) | 1u);
        if (2u * g <= n && gline >= (uint32_t)TOPL) prefetch_line(ws.line_ptr(gline));
      }
      Grp<G>::sync();  // every lane holds the line (and everything read before) — lane 0 may write now
      synced = true;
      if (occ_pending && line >= (uint32_t)TOPL) { prefetch_occ(*occ_node, L); occ_pending = false; }
      int best = -1;
      float bk = e.score;
      if (4u * h + 3u <= n) {  // all six candidates exist (every step but the last one or two of a descent)
#pragma unroll
        for (int c = 0; c < 6; ++c)
          if (f.x[c].score > bk) { best = c; bk = f.x[c].score; }
      } else {
#pragma unroll
        for (int c = 0; c < 6; ++c) {
          const uint32_t idx = c < 2 ? 2u * h + (uint32_t)c : 4u * h + (uint32_t)(c - 2);
          if (idx <= n && f.x[c].score > bk) { best = c; bk = f.x[c].score; }
        }
      }
      if (best < 0) break;
      // select chains instead of f.x[best]: a dynamically indexed register array goes through local memory (6 local stores
      // + 2 local loads per step = 245 L1 / 266 L2 write sectors per popped frame in profiles/r2_g32_wide_50Mbp_raw.csv)
      HeapEnt be = f.x[0];
#pragma unroll
      for (int c = 1; c < 6; ++c) if (best == c) be = f.x[c];
      wr(hpos, be);
      hpos = ln + best;
      if (best < 2) break;  // moved to a child: done
      const int pc = (best - 2) >> 1;  // the grandchild's parent is one of the two children in the same line
      const HeapEnt pe = pc ? f.x[1] : f.x[0];
      if (pe.score > e.score) { wr(ln + pc, e); e = pe; }
      h = 4u * h + (uint32_t)(best - 2);
      c_lo = (c_lo << 2) | 1u;
    }
    if (!synced) Grp<G>::sync();
    wr(hpos, e);
  }

  // MinMaxHeap::trickle_down_min from the root (pop_min, used by the limit recovery of mapping.rs:1358-1380): the node at a
  // min level looks at its two children and four grandchildren, which the family layout spreads over three lines (the
  // children sit in the line the node itself lives in); all six are fetched in one round trip by every lane.
  MAPAD_DEV void trickle_min(HeapEnt e, uint32_t n) {
    // h: 1-based position on a min level with `e` in the hole.  Its children 2h, 2h+1 are the entries c0, c1 stored at
    // cp[0], cp[1]; its grandchildren 4h .. 4h+3 are slots 0, 1 of the family lines of 2h and 2h+1 (two consecutive lines),
    // whose slots 2 .. 5 hold the children of those grandchildren, i.e. the c0, c1 of the next step: two line loads per step.
    uint32_t h = 1u;
    HeapEnt* hpos = ws.top;
    HeapEnt* cp = ws.top + 1;
    HeapEnt c0 = ws.top[1], c1 = ws.top[2];
    uint32_t c_lo = 1u;  // C(level of the children of h)
    bool synced = false;
    const uint32_t pf = n >= 8u * (uint32_t)TOPL ? ws.a->prefetch : 0u;
    while (2u * h <= n) {
      const uint32_t la = 2u * h - c_lo;
      HeapEnt* pa = ws.line_ptr(la);
      // la is odd and TOPL is odd: the next line is adjacent in memory unless it starts a new chunk
      HeapEnt* pb = (la + 1u == (uint32_t)TOPL || ((la + 1u) & ((1u << WS::LPC_SHIFT) - 1u)) == 0u) ? ws.line_ptr(la + 1u) : pa + 8;
      HeapLine6 fa, fb;
#pragma unroll
      for (int c = 0; c < 6; ++c) { fa.x[c] = e; fb.x[c] = e; }
      if (4u * h <= n) fa = load_line6(pa);
      if (4u * h + 2u <= n) fb = load_line6(pb);
      if ((pf & 1u) && G >= 8 && ws.gl < 8) {
        // the next step (at grandchild g) reads the family lines of 2g and 2g+1: eight candidates, one per lane
        const uint32_t g = 4u * h + ((uint32_t)ws.gl >> 1);
        const uint32_t gline = 2u * g - ((c_lo << 2) | 1u) + ((uint32_t)ws.gl & 1u);
        if (4u * g + 2u * ((uint32_t)ws.gl & 1u) <= n && gline >= (uint32_t)TOPL) prefetch_line(ws.line_ptr(gline));
      }
      Grp<G>::sync();
      synced = true;
      const HeapEnt x[6] = {c0, c1, fa.x[0], fa.x[1], fb.x[0], fb.x[1]};
      int best = -1;
      float bk = e.score;
      if (4u * h + 3u <= n) {
#pragma unroll
        for (int c = 0; c < 6; ++c)
          if (x[c].score < bk) { best = c; bk = x[c].score; }
      } else {
#pragma unroll
        for (int c = 0; c < 6; ++c) {
          const uint32_t idx = c < 2 ? 2u * h + (uint32_t)c : 4u * h + (uint32_t)(c - 2);
          if (idx <= n && x[c].score < bk) { best = c; bk = x[c].score; }
        }
      }
      if (best < 0) break;
      HeapEnt be = x[0];
#pragma unroll
      for (int c = 1; c < 6; ++c) if (best == c) be = x[c];
      wr(hpos, be);
      if (best < 2) { hpos = cp + best; break; }
      const int gb = best - 2;                     // which grandchild
      const HeapEnt pe = gb < 2 ? c0 : c1;          // its parent is one of the two children
      HeapEnt* ppos = cp + (gb >> 1);
      HeapEnt* gp = gb < 2 ? pa : pb;               // line of the chosen grandchild: slot gb & 1
      hpos = gp + (gb & 1);
      if (pe.score < e.score) { wr(ppos, e); e = pe; }
      // the children of the chosen grandchild: slots 2 + 2 (gb & 1), 3 + 2 (gb & 1) of the same line
      const HeapLine6& f = gb < 2 ? fa : fb;
      c0 = (gb & 1) ? f.x[4] : f.x[2];
      c1 = (gb & 1) ? f.x[5] : f.x[3];
      cp = gp + 2 + 2 * (gb & 1);
      h = 4u * h + (uint32_t)gb;
      c_lo = (c_lo << 2) | 1u;
    }
    if (!synced) Grp<G>::sync();
    wr(hpos, e);
  }

  // MinMaxHeap::push of `e` + Tree::add_node of `nd` (the two writes of an accepted child).
  // The positions a new element can visit depend only on its position x: the parent p = x / 2, then the grandparent chain
  // of x (the element stays on its level) or of p (it was swapped with the parent).  Cooperative version: every lane reads
  // the parent, lanes [0, G/2) fetch the chain of x and lanes [G/2, G) the chain of p in the same round trip, a vote finds
  // where the climb stops, and the lanes whose ancestors move one chain level down write them in parallel.  Deeper chains
  // (more than G/2 levels) continue with all G lanes on the chosen chain.
  MAPAD_DEV void push(HeapEnt e, const NodeWords& nd) {
    const uint32_t x = heap_n + 1u;
    heap_n = x;
    Grp<G>::sync();  // writes of the previous phase are visible
    if (x == 1u) {
      if (ws.gl == 0) { node_put(ws.node_ptr(e.node), nd); ws.top[0] = e; }
      return;
    }
    const uint32_t p = x >> 1;
    const bool min_level = ((31 - clz32(x)) & 1) == 0;
    if (G == 1) {  // sequential: count the steps first, then move the ancestors down
      const HeapEnt pe = rd(p);
      const bool moved = min_level ? (e.score > pe.score) : (e.score < pe.score);
      const bool climb_max = min_level == moved;
      uint32_t t = 0, c = moved ? p : x;
      while (c >= 4u) {
        const HeapEnt ae = rd(c >> 2);
        if (climb_max ? (e.score > ae.score) : (e.score < ae.score)) { t += 1; c >>= 2; } else break;
      }
      node_put(ws.node_ptr(e.node), nd);
      uint32_t cur = x;
      if (moved) { *ptr(x) = pe; cur = p; }
      for (uint32_t k = 0; k < t; ++k) { *ptr(cur) = *ptr(cur >> 2); cur >>= 2; }
      *ptr(cur) = e;
      return;
    }
    constexpr int H = G > 1 ? G / 2 : 1;
    const int gl = ws.gl;
    const bool in_b = gl >= H;
    const uint32_t lvl = (uint32_t)(in_b ? gl - H : gl) + 1u;          // chain level of this lane in round 1
    const uint32_t anc = lvl < 16u ? (in_b ? p : x) >> (2u * lvl) : 0u;  // 1-based position of that grandparent, 0 = none
    HeapEnt v = e;
    if (anc) v = rd(anc);
    const HeapEnt pe = rd(p);
    const bool moved = min_level ? (e.score > pe.score) : (e.score < pe.score);
    const bool climb_max = min_level == moved;
    const bool wins = anc != 0u && (climb_max ? (e.score > v.score) : (e.score < v.score));
    const uint32_t ball = Grp<G>::ballot(wins);  // also: every lane has finished reading
    const uint32_t half = moved ? (ball >> H) : (ball & ((1u << H) - 1u));
    const uint32_t t1 = (uint32_t)ffs32(~half) - 1u;                     // leading run of winning levels (<= H)
    const uint32_t cur0 = moved ? p : x;
    if (anc != 0u && in_b == moved && lvl <= t1) *ptr(cur0 >> (2u * (lvl - 1u))) = v;
    uint32_t total = t1, base = (uint32_t)H;
    while (total == base && base < 16u && (cur0 >> (2u * base)) >= 4u) {  // every fetched level won and the chain goes on
      const uint32_t l2 = base + (uint32_t)gl + 1u;
      const uint32_t a2 = l2 < 16u ? cur0 >> (2u * l2) : 0u;
      HeapEnt v2 = e;
      if (a2) v2 = rd(a2);
      const bool w2 = a2 != 0u && (climb_max ? (e.score > v2.score) : (e.score < v2.score));
      const uint32_t b2 = Grp<G>::ballot(w2);
      const uint32_t t2 = b2 == 0xffffffffu ? 32u : (uint32_t)ffs32(~b2) - 1u;
      if (a2 != 0u && (uint32_t)gl < t2) *ptr(cur0 >> (2u * (l2 - 1u))) = v2;
      total += t2;
      base += (uint32_t)G;
    }
    if (gl == 0) {
      node_put(ws.node_ptr(e.node), nd);
      if (moved) *ptr(x) = pe;
      *ptr(cur0 >> (2u * total)) = e;
    }
  }

  MAPAD_DEV void begin(const DevIndex& ix, int start_pos) {
    heap_n = 0; node_hi = 1; free_head = MAPAD_NO_NODE; tree_len = 1; n_hits = 0; best_score = 0.0f; best_size = 0;
    ws.frames = 0; limit_hit = 0; overflow = false;
    Frame root;
    root.iv = BiIv{0, 0, ix.m.n};
    root.start = start_pos; root.len = 0; root.gap_f = GAP_CLOSED; root.gap_b = GAP_CLOSED; root.ngaps = 0;
    root.score = 0.0f; root.node = 0;
    // tree.clear(): root = NodeId(0)
    push(HeapEnt{0.0f, 0}, node_words(static_cast<const Node*>(nullptr), root, 0, pack_op(0, MAPAD_ED_MATCH, 0)));
    Grp<G>::sync();  // the root is visible to every lane before the first step reads it
  }

  // check_and_push_stack_frame (mapping.rs:932-987)
  MAPAD_DEV void check_and_push(const Frame& f, uint32_t parent_node, uint32_t op, int L, const BoundCtx& bc, const DevParams& P) {
    if (n_hits > 0 && bound_reject_iterative(bc, f.score, best_score)) return;
    if (f.ngaps > P.max_num_gaps_open) return;
    uint32_t id;
    if (free_head != MAPAD_NO_NODE) {  // slab: most recently vacated key first
      id = free_head;
      free_head = ws.node(id).parent;
    } else {
      id = node_hi;
      if (!ws.ensure_node(id)) { overflow = true; return; }
      node_hi += 1;
    }
    tree_len += 1;
    const NodeWords nd = node_words(static_cast<const Node*>(nullptr), f, parent_node, op);
    if (f.len == L) {  // a hit: std BinaryHeap::push
      Grp<G>::sync();
      if (ws.gl == 0) {
        node_put(ws.node_ptr(id), nd);
        if (n_hits < MAPAD_MAX_HITS) {
          HitTmp h;
          h.score = f.score; h.node = id; h.lower = f.iv.lower; h.lower_rev = f.iv.lower_rev; h.size = f.iv.size;
          uint32_t nh = n_hits;
          bh_push(ws.hits(), nh, h);
        }
      }
      if (n_hits < MAPAD_MAX_HITS) n_hits += 1;
      Grp<G>::sync();
      best_score = ws.hits()[0].score;
      best_size = ws.hits()[0].size;
      return;
    }
    if (!ws.ensure_heap(heap_n)) { overflow = true; return; }
    push(HeapEnt{f.score, id}, nd);
  }

  // One pop-and-expand step of k_mismatch_search (mapping.rs:1058-1380); same decisions as search_core.cuh::search_step.
  MAPAD_DEV int step(const DevIndex& ix, const DevParams& P, const SearchJob& job) {
    const int L = job.L;
    const BoundCtx& bc = job.bc;
    const float open_ext = job.open_ext;
    const uint32_t n = heap_n;
    if (n == 0) return STEP_DONE;
    // ---- MinMaxHeap::pop_max ----
    uint32_t m = 1;
    if (n == 2) m = 2;
    else if (n >= 3) m = ws.top[1].score > ws.top[2].score ? 2u : 3u;
    const HeapEnt topent = ws.top[m - 1u];
    ws.frames += 1;
    const Node pn = ws.node(topent.node);  // issued before the heap is repaired: both latencies overlap
    const uint32_t n1 = n - 1u;
    if (m <= n1) {
      const HeapEnt last = rd(n);
      trickle_max(m, last, n1, &pn, job.L);
    }
    heap_n = n1;
    Frame sf;
    node_load(pn, topent.node, sf);
    sf.score = topent.score;
    int j, d_k, d_l;
    bool forward;
    if (sf.start <= L - sf.start - sf.len) {  // mapping.rs:1077-1097
      j = sf.start + sf.len; forward = true; d_k = sf.start; d_l = sf.start + sf.len;
    } else {
      j = sf.start - 1; forward = false; d_k = sf.start - 1; d_l = sf.start + sf.len - 1;
    }
    const PenRow row = job.delta[j];
    const int side_gap = forward ? sf.gap_f : sf.gap_b;
    const float insertion_score = fadd(side_gap == GAP_INS ? P.gap_extend : open_ext, sf.score);
    const float deletion_score = fadd(side_gap == GAP_DEL ? P.gap_extend : open_ext, sf.score);
    const int num_gaps_open = side_gap == GAP_CLOSED ? sf.ngaps + 1 : sf.ngaps;
    const float lower_bound = d_get(job.dcomp, L, job.start_pos, d_k, d_l);
    if (n_hits > 0) {  // mapping.rs:1201-1208
      if (bound_reject_iterative(bc, fadd(sf.score, lower_bound), best_score)) return STEP_DONE;
    }
    const int child_start = forward ? sf.start : sf.start - 1;
    // candidates in the reference's order (insertion; then for T,G,C,A: deletion, match/mismatch) as 4-bit codes
    uint64_t codes = 0;
    int n_cand = 0;
    {  // insertion (mapping.rs:1213-1242)
      const int dist = j < L - j - 1 ? j : L - j - 1;
      if (!bound_reject(bc, fadd(insertion_score, lower_bound)) && dist >= P.gap_dist_ends) { n_cand = 1; }
    }
    BiIv ext[4];
    {
      const BiIv in = forward ? BiIv{sf.iv.lower_rev, sf.iv.lower, sf.iv.size} : sf.iv;
      extend_all_group<WIDE, G>(ix, in, ext, ws.gl);
    }
    const bool del_ok = !bound_reject(bc, fadd(deletion_score, lower_bound));
    const int dist5 = forward ? j : j + 1;
    const int dist3 = L - dist5;
    const bool del_dist_ok = (dist5 < dist3 ? dist5 : dist3) >= P.gap_dist_ends;
    const uint8_t read_base = job.seq[j];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (ext[k].size < 1) continue;
      const int pen_idx = forward ? k : 3 - k;  // rank = 4 - k; forward: 4 - rank, backward: rank - 1
      if (del_ok && del_dist_ok) { codes |= (uint64_t)(4 | k) << (4 * n_cand); n_cand += 1; }
      const float mm_score = fadd(row.d[pen_idx], sf.score);
      if (!bound_reject(bc, fadd(mm_score, lower_bound))) { codes |= (uint64_t)(8 | k) << (4 * n_cand); n_cand += 1; }
    }
    for (int i = 0; i < n_cand && !overflow; ++i) {
      const uint32_t code = (uint32_t)(codes >> (4 * i)) & 15u;
      const uint32_t type = code >> 2, k = code & 3u;
      Frame ch = sf;
      uint32_t op;
      if (type == 0) {
        ch.start = child_start; ch.len = sf.len + 1;
        if (forward) ch.gap_f = GAP_INS; else ch.gap_b = GAP_INS;
        ch.score = insertion_score; ch.ngaps = num_gaps_open;
        op = pack_op(j, MAPAD_ED_INSERTION, 0);
      } else {
        BiIv ip = k == 0 ? ext[0] : (k == 1 ? ext[1] : (k == 2 ? ext[2] : ext[3]));
        const int rank = 4 - (int)k;
        uint8_t c;
        if (forward) { ip = BiIv{ip.lower_rev, ip.lower, ip.size}; c = complement_base(rank_base(rank)); }
        else c = rank_base(rank);
        ch.iv = ip;
        if (type == 1) {
          if (forward) ch.gap_f = GAP_DEL; else ch.gap_b = GAP_DEL;
          ch.score = deletion_score; ch.ngaps = num_gaps_open;
          op = pack_op(j, MAPAD_ED_DELETION, c);
        } else {
          const int pen_idx = forward ? (int)k : 3 - (int)k;
          const float pen = pen_idx == 0 ? row.d[0] : (pen_idx == 1 ? row.d[1] : (pen_idx == 2 ? row.d[2] : row.d[3]));
          ch.start = child_start; ch.len = sf.len + 1;
          if (forward) ch.gap_f = GAP_CLOSED; else ch.gap_b = GAP_CLOSED;
          ch.score = fadd(pen, sf.score);
          op = c == read_base ? pack_op(j, MAPAD_ED_MATCH, 0) : pack_op(j, MAPAD_ED_MISMATCH, c);
        }
      }
      check_and_push(ch, sf.node, op, L, bc, P);
    }
    if (overflow) return STEP_OVERFLOW;
    // early exits (mapping.rs:1348-1355)
    if (n_hits > 9 || (n_hits > 0 && best_size > 1)) return STEP_DONE;
    // limits (mapping.rs:1358-1380): evict the worst frames (MinMaxHeap::pop_min) and their tree nodes
    if (heap_n > P.stack_limit || tree_len > P.edit_tree_limit) {
      limit_hit += 1;
      if (P.stack_limit_abort) return STEP_DONE;
      const long long e1 = (long long)heap_n - (long long)P.stack_limit;
      const long long e2 = (long long)tree_len - (long long)P.edit_tree_limit;
      const long long excess = e1 > e2 ? e1 : e2;
      for (long long e = 0; e < excess && heap_n > 0; ++e) {  // MinMaxHeap::pop_min + Tree::remove, every lane in step
        Grp<G>::sync();
        const HeapEnt mn = ws.top[0];
        const uint32_t n1 = heap_n - 1u;
        if (n1 > 0u) {
          const HeapEnt last = rd(heap_n);
          trickle_min(last, n1);
        }
        heap_n = n1;
        if (mn.node != 0u) {  // Tree::remove (backtrack_tree.rs:49-53): the vacated key heads the slab's free list
          Grp<G>::sync();
          if (ws.gl == 0) ws.node(mn.node).parent = free_head;
          free_head = mn.node;
          tree_len -= 1;
        }
      }
    }
    Grp<G>::sync();  // end of step: all writes are visible to the next step's reads
    return STEP_CONTINUE;
  }
};

// The loop of one lane of group `slot` (all G lanes of the group call it with the same arguments but their own `gl`).
template <bool WIDE, int G, int TOPL>
MAPAD_DEV void group_search_lane(const GroupLaunch<WIDE>& a, uint32_t slot, int gl, HeapEnt* smem_top) {
  using GS = GroupSearch<WIDE, G, TOPL>;
  GS gs;
  auto& ws = gs.ws;
  ws.a = &a;
  ws.slot = slot;
  ws.gl = gl;
  // every group takes its two base chunks (nodes, heap) from the device-wide pool when it starts and returns them when it exits
  uint32_t c_nodes, c_heap;
  if (!ws.acquire_base(c_nodes, c_heap)) {
    if (gl == 0) dev_atomic_or(&a.cur->overflow, MAPAD_POOL_TIMEOUT_FLAG);
    return;
  }
  if (gl == 0) { ws.table()[0] = c_nodes; ws.table()[a.nt] = c_heap; }
  Grp<G>::sync();
  ws.n_node_chunks = 1;
  ws.n_heap_chunks = 1;
  ws.heap_hi = 0;
  ws.node0 = reinterpret_cast<typename GS::Node*>(a.pool.base + ((size_t)c_nodes << MAPAD_GCHUNK_SHIFT));
  ws.heap0 = reinterpret_cast<HeapEnt*>(a.pool.base + ((size_t)c_heap << MAPAD_GCHUNK_SHIFT));
  ws.top = smem_top;
  ws.frames = 0;
  uint32_t busy_iters = 0;
  bool have = false;
  uint32_t r = 0;
  int split = 0;
  SearchJob job;
  while (true) {
    if (!have) {
      uint32_t w = 0;
      if (gl == 0) {
        // admission control: do not start a read while groups in flight are waiting for memory (bounded: 30 s)
        for (uint32_t k = 0; k < 15000000u && *gpool_pressure(a.pool) > dev_now_ns(); ++k) dev_backoff<G>();
        w = dev_atomic_add(&a.cur->queue_head, 1u);
      }
      w = Grp<G>::shfl(w, 0);
      if (w >= a.n_work) break;
      r = a.work_list ? a.work_list[w] : w;
      const uint64_t o = a.rb.offsets[r];
      const int L = (int)(a.rb.offsets[r + 1] - o);
      if (L <= 0) {
        if (gl == 0) {
          ReadMid m;
          m.n_hits = 0; m.hit_off = 0; m.frames_popped = 0; m.flags = 0;
          a.mid[r] = m;
        }
        continue;
      }
      split = alignment_start(a.P, a.rb, r, L);
      job = make_job(a.P, a.bound_table, a.rb.seq + o, L, split, a.delta + o, a.dcomp + o);
      gs.begin(a.ix, split);
      have = true;
    }
    const int rc = gs.step(a.ix, a.P, job);
    busy_iters += 1;
    if (a.iter_budget && busy_iters >= a.iter_budget) { ws.release_extra(); break; }
    if (rc == STEP_CONTINUE) continue;
    have = false;
    Grp<G>::sync();
    if (rc == STEP_OVERFLOW) {  // the pool ran dry: the host re-runs the read with fewer groups in flight
      ws.release_extra();
      if (gl == 0) a.deferred_list[dev_atomic_add(&a.cur->n_deferred, 1u)] = r;
      continue;
    }
    // ---- emit: lane l traces hits l, l + G, ... back to the root (extract_edit_operations, record.rs:465-500) ----
    const uint32_t nh = gs.n_hits;
    uint32_t hit_off = 0;
    if (nh) {
      if (gl == 0) hit_off = dev_atomic_add(&a.cur->hit_cursor, nh);
      hit_off = Grp<G>::shfl(hit_off, 0);
      for (uint32_t h = (uint32_t)gl; h < nh; h += (uint32_t)G) {
        const HitTmp ht = ws.hits()[h];
        uint32_t n_left;
        const uint32_t total = path_length<WIDE>(ws, ht.node, split, n_left);
        const uint32_t op_off = dev_atomic_add(&a.cur->op_cursor, total);
        if ((uint64_t)op_off + total <= a.op_cap) path_write<WIDE>(ws, ht.node, split, total, n_left, a.op_pool + op_off);
        else dev_atomic_or(&a.cur->overflow, 1u);
        if ((uint64_t)hit_off + h < a.hit_cap) {
          mapad_hit mh;
          mh.lower = ht.lower; mh.lower_rev = ht.lower_rev; mh.size = ht.size;
          mh.alignment_score = ht.score; mh.edit_off = op_off; mh.edit_len = total; mh.reserved = 0;
          a.hit_pool[hit_off + h] = mh;
        } else {
          dev_atomic_or(&a.cur->overflow, 1u);
        }
      }
    }
    if (gl == 0) {
      ReadMid m;
      m.hit_off = hit_off;
      m.frames_popped = ws.frames;
      m.flags = (gs.limit_hit ? 1u : 0u) | a.flags_or;
      m.n_hits = nh;
      a.mid[r] = m;
    }
    Grp<G>::sync();  // the tree is no longer read: its chunks may go back to the pool
    ws.release_extra();
  }
  Grp<G>::sync();
  ws.release_base();
}

#if defined(__CUDACC__)
// One warp per block: a block's registers and shared memory stay allocated until its LAST group has finished, and the
// heaviest reads run for seconds after the queue is empty — with 128-thread blocks every such read would pin a quarter of
// an SM's resident capacity while the launches of the next chunks wait for block slots.
#ifndef MAPAD_GROUP_BLOCK
#define MAPAD_GROUP_BLOCK 32
#endif
#ifndef MAPAD_GROUP_MIN_BLOCKS
#define MAPAD_GROUP_MIN_BLOCKS 16
#endif
// MINB = resident blocks (warps) per SM the register allocation is sized for: 16 -> up to 128 registers, 20 -> 96, 24 -> 80.
template <bool WIDE, int G, int TOPL, int MINB = MAPAD_GROUP_MIN_BLOCKS>
__global__ void __launch_bounds__(MAPAD_GROUP_BLOCK, MINB) k_search_group(const __grid_constant__ GroupLaunch<WIDE> a) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const uint32_t group_in_block = threadIdx.x / G;
  const uint32_t slot = blockIdx.x * (MAPAD_GROUP_BLOCK / G) + group_in_block;
  HeapEnt* top = reinterpret_cast<HeapEnt*>(smem_raw) + (size_t)group_in_block * TOPL * 8;
  group_search_lane<WIDE, G, TOPL>(a, slot, (int)(threadIdx.x % G), top);
}

__global__ void k_gpool_init(GChunkPool p) {  // chunk i starts in shard i % SHARDS
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < p.n_chunks) p.next[i] = i + MAPAD_GPOOL_SHARDS < p.n_chunks ? i + MAPAD_GPOOL_SHARDS : MAPAD_GPOOL_EMPTY;
  if (i < MAPAD_GPOOL_SHARDS) p.heads[(size_t)i * MAPAD_GPOOL_HEAD_STRIDE] = i < p.n_chunks ? (unsigned long long)i : (unsigned long long)MAPAD_GPOOL_EMPTY;
  if (i == 0) p.heads[8] = 0ull;  // pressure deadline
}
#endif

}  // namespace mapad
