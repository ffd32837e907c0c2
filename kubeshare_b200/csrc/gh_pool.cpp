// gh_pool.cpp -- the shared credit pool: one file-backed MAP_SHARED region per GPU that replaces the
// hook -> gem-pmgr -> gem-schd TCP round trips (reference hook.cpp:300-328, 425-446) for co-resident
// clients.  The token policy that runs inside it, bit-exact with the reference, is gh_policy.h.
//
// What is new: there is no daemon, NO LOCK and no context switch in the decision path.
//
// LOCK-FREE BY CONSTRUCTION.  All policy state (token holder, deadline, per-client quota/mailbox/pod token, ledger)
// lives in a versioned STATE BLOCK.  The region holds NBLK such blocks; the 64-bit word `cur` = (sequence << 8 |
// block index) names the current one.  Every mutation is a transaction:
//     claim a free block (one CAS)  ->  copy the current block into it, validate `cur` did not move  ->  run the
//     SERIAL policy code on the private copy  ->  publish with ONE compare-and-swap on `cur`  ->  free the old block.
// A failed CAS means somebody else's transaction went through (system-wide progress: lock-free); the loser
// re-copies and retries.  A process that is SIGKILLed anywhere -- before, between or after those steps -- never
// blocks anybody: at worst it leaks a claimed block, which is recognised (owner dead, or its publication attempt
// provably resolved) and recycled.  Readers (exporters, gem-poolctl, the hot gpu_mem path)
// never write anything: they copy / peek and validate against `cur`, so a Prometheus scrape cannot delay a token
// hand-over.  Because transactions run the unchanged serial code on a consistent snapshot, the ledger arithmetic
// stays bit-exact with the reference.
// Clients that must wait (throttled, or another client holds the token) futex-wait on their slot's wake word;
// short waits spin.  The region is plain memory: its first pages (header, per-slot counters) are cuMemHostRegister'ed
// by the hook so the device sees the same counters ("shared-pinned").
#ifndef _GNU_SOURCE
#define _GNU_SOURCE
#endif
#include <errno.h>
#include <fcntl.h>
#include <limits.h>
#include <linux/futex.h>
#include <math.h>
#include <sched.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <vector>

#include "gh_internal.h"

#ifdef GEMHOOK_FAULT_INJECTION
// tests/native/pool_kill.cpp: die (SIGKILL) at the n-th pass through a named point of the transaction protocol;
// tests/native/pool_ownership.cpp: stop there (SIGSTOP) instead
#include <signal.h>
extern "C" int gemhook_fault_point;  // 0 = off
extern "C" long gemhook_fault_countdown;
extern "C" int gemhook_fault_signal;
int gemhook_fault_signal = SIGKILL;
#define GH_FAULT(pt)                                                                                \
  do {                                                                                              \
    if (gemhook_fault_point == (pt) && --gemhook_fault_countdown <= 0) raise(gemhook_fault_signal); \
  } while (0)
#else
#define GH_FAULT(pt) do { } while (0)
#endif
enum { FP_AFTER_CLAIM = 1, FP_MID_POLICY = 2, FP_BEFORE_CAS = 3, FP_AFTER_CAS = 4 };

#define GH_NO_TSAN __attribute__((no_sanitize("thread")))

namespace {

const uint64_t POOL_MAGIC = 0x324c4f4f504d4547ULL;  // "GEMPOOL2"
const uint32_t POOL_VERSION = 4;
const uint32_t MAX_ATTACH = 256;
const uint32_t NBLK = 16;

// ---- unversioned shared words ---------------------------------------------------------------------------------
struct alignas(64) SlotShared {  // hot counters other parties (and the device) read; one cache line per slot
  std::atomic<uint64_t> mem_used;
  std::atomic<uint64_t> mem_limit_mirror;  // copy of the slot's mem_limit for the device-side mirror (informational)
  std::atomic<uint64_t> gpu_ns, launches;
  std::atomic<uint32_t> wake;  // futex word: bumped whenever something happens that this slot's waiters care about
  uint32_t _pad[7];
};
static_assert(sizeof(SlotShared) == 64, "shared slot layout");

struct alignas(64) Header {
  uint64_t magic;
  uint32_t version, nslots_max;
  double base_quota, min_quota, window;
  std::atomic<int64_t> start_ns;
  std::atomic<uint32_t> ready;
  uint32_t _pad0;
  std::atomic<uint64_t> boot_id;  // CLOCK_MONOTONIC restarts at boot: a pool file that survived a reboot is re-initialised
  alignas(64) std::atomic<uint64_t> cur;  // (sequence << 8) | index of the current state block
  alignas(64) std::atomic<uint64_t> quota_stamp;  // mtime/size stamp of the quota file last loaded
  std::atomic<uint64_t> commits, conflicts, recycled;
};

// one entry per attached handle; byte 0 of each entry is covered by an OFD lock held by the owner for its
// lifetime -- the kernel drops it when the process dies, in any container, which is how a dead client's
// bytes, token and claimed state blocks are found and reclaimed (the reference reclaims on socket close,
// pod-manager.cpp:533-545)
struct Attach {
  std::atomic<uint32_t> in_use;  // FREE, INIT, LIVE or REAPING (gemhook_pool::take_attachment)
  std::atomic<int32_t> slot;  // -1: observer (a tool or a test that only needs a liveness byte for its transactions)
  std::atomic<uint64_t> bytes;
  std::atomic<uint64_t> burst_bits;  // client_burst_map entry (pod-manager.cpp:98), a double
  uint32_t pid;
  std::atomic<uint32_t> epoch;  // bumped each time the entry is taken: an owner tag names one owner, not one index
};
static_assert(sizeof(Attach) == 32, "attach layout");
enum : uint32_t { FREE = 0, INIT = 1, LIVE = 2, REAPING = 3 };

}  // namespace

#include "gh_policy.h"

namespace {

// block control word: 0 = FREE, else 1 << 63 | owner tag << 40 | publication sequence (40 bits, 0 = not publishing);
// owner tag = attachment index (9 bits, NO_OWNER: the block was published by the pool's initialisation) << 14 | the
// entry's epoch (14 bits)
const int PUB_BITS = 40, EPOCH_BITS = 14, OWNER_BITS = 9;
const uint64_t PUB_MASK = (1ull << PUB_BITS) - 1;
const uint32_t EPOCH_MASK = (1u << EPOCH_BITS) - 1, NO_OWNER = (1u << OWNER_BITS) - 1;
static_assert(1 + OWNER_BITS + EPOCH_BITS + PUB_BITS == 64 && MAX_ATTACH < NO_OWNER, "control word layout");
inline uint64_t ctl_make(uint32_t tag, uint64_t pub) { return (1ull << 63) | (uint64_t)tag << PUB_BITS | (pub & PUB_MASK); }
inline uint32_t ctl_tag(uint64_t w) { return (uint32_t)(w >> PUB_BITS) & ((1u << (OWNER_BITS + EPOCH_BITS)) - 1); }
inline uint64_t ctl_pub(uint64_t w) { return w & PUB_MASK; }
const uint32_t NO_OWNER_TAG = NO_OWNER << EPOCH_BITS;
// the sequence a transaction that copied `seen` publishes; one whose low PUB_BITS are 0 is skipped, so a publishing
// word never reads as merely claimed
inline uint64_t next_seq(uint64_t seen) { return ((seen >> 8) + 1) & PUB_MASK ? (seen >> 8) + 1 : (seen >> 8) + 2; }
// `cur` carries sequence >= pub, modulo 2^PUB_BITS (serial-number arithmetic).  While the publication of pub can still
// succeed, cur is pub - 1 (pub - 2 past a skipped sequence), which reads as "not yet"; every cur in [pub, pub + 2^39)
// reads as "resolved".  A word outlives its publication by 2^39 commits only if its owner stalls that long; at worst
// the block then stays claimed until the owner is found dead.
inline bool pub_resolved(uint64_t pub, uint64_t cur_seq) { return pub && ((cur_seq - pub) & PUB_MASK) < (1ull << (PUB_BITS - 1)); }

struct Region {
  Header h;
  SlotShared shared[GEMHOOK_MAX_SLOTS];
  Attach attach[MAX_ATTACH];
  alignas(64) std::atomic<uint64_t> bctl[NBLK];
  alignas(4096) State blocks[NBLK];
};

uint64_t boot_id_hash() {
  uint64_t h = 1469598103934665603ULL;
  FILE* f = fopen("/proc/sys/kernel/random/boot_id", "r");
  if (f) {
    int c;
    while ((c = fgetc(f)) != EOF) h = (h ^ (uint64_t)(unsigned char)c) * 1099511628211ULL;
    fclose(f);
  }
  return h > 1 ? h : 2;
}

long futex(std::atomic<uint32_t>* addr, int op, uint32_t val, const struct timespec* ts) {
  return syscall(SYS_futex, (uint32_t*)addr, op, val, ts, nullptr, 0);
}

bool attach_move(Attach& a, uint32_t from, uint32_t to) { return a.in_use.compare_exchange_strong(from, to, std::memory_order_acq_rel); }

}  // namespace

// ---- ownership of the shared entries ----------------------------------------------------------------------------
// STATE BLOCKS.  Block b's control word bctl[b] moves
//     FREE (0) --claim--> CLAIMED(o) --publish--> PUBLISHING(o, P) --CAS on `cur` won--> current --retire--> FREE
//     PUBLISHING --unpublish (CAS on `cur` lost)--> CLAIMED --abort--> FREE;  CLAIMED / PUBLISHING --recycle--> FREE
// o = the owner's tag (attachment index, that entry's epoch), P = the sequence `cur` carries if the block becomes current.
// claim: anyone, from FREE.  publish, unpublish, abort: the owner, from the word it wrote.  retire: the committer that
// replaced the block, only from a word that still names the replaced publication (any other word: a recycler freed the
// block first and it is somebody else's now).  recycle: anyone, from the very word it judged never_current.  Each edge is
// one CAS from the word observed, and a new claim writes another tag or epoch, so a stale party frees nothing it did not judge.
// A block that is not current can never become current when (liveness read before `cur`)
//  * its owner is dead: the entry's OFD byte is unlocked, or the entry was re-taken since (its epoch moved on) -- a dead
//    owner cannot publish any more, so a block that is not current now never will be;
//  * or its publication is resolved: `cur` already carries sequence >= P on another block, so the CAS expecting P - 1
//    has failed or will fail.  A live owner learns from its own next control-word CAS that the block is gone.
//
// ATTACHMENT ENTRIES.  attach[i].in_use moves FREE -> INIT -> LIVE (take), LIVE -> FREE (close), LIVE -> REAPING -> FREE
// (reap), each move by the holder of the entry's OFD byte: the taker locks it first and bumps the epoch, the owner stores
// FREE before it unlocks the byte at close, a reaper can lock it only once the owner is gone.  So an entry that reads
// LIVE with its byte unlocked belongs to a dead process; the CASes keep a party that looked earlier from moving it later.
struct gemhook_pool {
  Region* r = nullptr;
  int fd = -1;
  bool anonymous = false;
  int attach_idx = -1;     // this handle's client attachment (set by gemhook_pool_attach)
  int liveness_idx = -1;   // attachment whose OFD byte vouches for this handle's transactions (client or observer)
  std::atomic<uint32_t> rr{0};

  // the OFD lock on byte 0 of attachment entry idx.  F_OFD_SETLK takes (F_WRLCK) or drops (F_UNLCK) it: true on
  // success; F_OFD_GETLK: true if another open file description holds it, or if the kernel cannot tell.  A private
  // pool has no file and one process: always true.
  bool attach_byte(int idx, int cmd, short type) const {
    if (fd < 0) return true;
    struct flock fl;
    memset(&fl, 0, sizeof(fl));
    fl.l_type = type;
    fl.l_whence = SEEK_SET;
    fl.l_start = (off_t)(offsetof(Region, attach) + (size_t)idx * sizeof(Attach));
    fl.l_len = 1;
    if (fcntl(fd, cmd, &fl) != 0) return cmd == F_OFD_GETLK;
    return cmd == F_OFD_SETLK || fl.l_type != F_UNLCK;
  }
  bool entry_alive(int idx) const { return idx == liveness_idx || idx == attach_idx || attach_byte(idx, F_OFD_GETLK, F_WRLCK); }
  bool owner_alive(uint32_t tag) const {
    uint32_t idx = tag >> EPOCH_BITS;
    if (idx >= MAX_ATTACH) return true;
    return (r->attach[idx].epoch.load(std::memory_order_acquire) & EPOCH_MASK) == (tag & EPOCH_MASK) && entry_alive((int)idx);
  }
  uint32_t owner_tag() const {
    if (liveness_idx < 0) return NO_OWNER_TAG;
    return (uint32_t)liveness_idx << EPOCH_BITS | (r->attach[liveness_idx].epoch.load(std::memory_order_relaxed) & EPOCH_MASK);
  }

  // FREE -> INIT -> LIVE.  The byte is locked before the entry leaves FREE, and INIT keeps readers off the fields until
  // they are set (a reaper once took an entry being set up for a dead one: two live clients then shared it)
  int take_attachment(int slot) {
    for (uint32_t i = 0; i < MAX_ATTACH; i++) {
      Attach& a = r->attach[i];
      if (a.in_use.load(std::memory_order_acquire) != FREE || !attach_byte((int)i, F_OFD_SETLK, F_WRLCK)) continue;
      if (attach_move(a, FREE, INIT)) {
        a.epoch.fetch_add(1);
        a.slot.store(slot);
        a.bytes.store(0);
        a.burst_bits.store(0);
        a.pid = (uint32_t)getpid();
        a.in_use.store(LIVE, std::memory_order_release);
        return (int)i;
      }
      attach_byte((int)i, F_OFD_SETLK, F_UNLCK);  // LIVE with its byte free: a dead owner's, left to the reapers
    }
    return -1;
  }

  int64_t now_us() const { return (gh_now_ns() - r->h.start_ns.load(std::memory_order_relaxed)) / 1000; }
  double now_ms() const { return (double)now_us() / 1e3; }  // scheduler.cpp:107-109

  // ---- state blocks ---------------------------------------------------------------------------------------
  // copy the live part of a state block (header fields, nslots slots, ledger_len spans); the source may be
  // overwritten underneath us (then `cur` has moved and the caller discards the copy), so lengths are clamped
  // (word-wise relaxed atomic loads, not memcpy: this is the reader side of a sequence-validated copy -- the loads
  //  may race with a writer that has recycled the source block, which the C++ memory model only tolerates for atomics;
  //  ThreadSanitizer intercepts memcpy even inside a no_sanitize function)
  GH_NO_TSAN static void raw_copy(void* dst, const void* src, size_t bytes) {
    uint64_t* d = (uint64_t*)dst;
    const uint64_t* s = (const uint64_t*)src;
    for (size_t i = 0, n = bytes / 8; i < n; i++) d[i] = __atomic_load_n(s + i, __ATOMIC_RELAXED);
  }
  GH_NO_TSAN static void copy_state(State* dst, const State* src) {
    static_assert(offsetof(State, slots) % 8 == 0 && sizeof(PSlot) % 8 == 0 && sizeof(Span) % 8 == 0, "word copy");
    raw_copy(dst, src, offsetof(State, slots));
    uint32_t ns = dst->nslots, ll = dst->ledger_len;
    if (ns > GEMHOOK_MAX_SLOTS) ns = GEMHOOK_MAX_SLOTS;
    if (ll > LEDGER_CAP) ll = LEDGER_CAP;
    dst->nslots = ns;
    dst->ledger_len = ll;
    raw_copy(dst->slots, src->slots, sizeof(PSlot) * ns);
    raw_copy(dst->ledger, src->ledger, sizeof(Span) * ll);
  }

  // recycle, step 1: a pure judgement of word w (!= 0) on block b -- can the block never become current?
  bool never_current(uint32_t b, uint64_t w) const {
    bool dead = !owner_alive(ctl_tag(w));
    uint64_t c = r->h.cur.load(std::memory_order_acquire);
    return (c & 0xff) != b && (dead || pub_resolved(ctl_pub(w), c >> 8));
  }
  // recycle, step 2: free the block if it still holds the word that was judged
  bool recycle(uint32_t b, uint64_t w) {
    if (!r->bctl[b].compare_exchange_strong(w, 0, std::memory_order_acq_rel)) return false;
    r->h.recycled.fetch_add(1, std::memory_order_relaxed);
    return true;
  }
  int recycle_blocks() {
    int freed = 0;
    for (uint32_t b = 0; b < NBLK; b++) {
      uint64_t w = r->bctl[b].load(std::memory_order_acquire);
      if (w && never_current(b, w) && recycle(b, w)) freed++;
    }
    return freed;
  }

  // FREE -> CLAIMED(word)
  int claim_block(uint64_t word) {
    uint32_t start = rr.fetch_add(1, std::memory_order_relaxed);
    for (;;) {
      for (uint32_t k = 0; k < NBLK; k++) {
        uint32_t b = (start + k) % NBLK;
        uint64_t exp = 0;
        if (r->bctl[b].load(std::memory_order_relaxed) == 0 && r->bctl[b].compare_exchange_strong(exp, word, std::memory_order_acq_rel))
          return (int)b;
      }
      if (recycle_blocks() == 0) sched_yield();  // every block is in somebody's live transaction: they finish in microseconds
    }
  }
};

namespace {

// current -> FREE once superseded, by the committer that replaced it: only while the block's word still names the
// publication `seen` made current
bool retire(Region* r, uint64_t seen) {
  uint32_t b = (uint32_t)(seen & 0xff);
  uint64_t w = r->bctl[b].load(std::memory_order_acquire);
  return w && ctl_pub(w) == ((seen >> 8) & PUB_MASK) && r->bctl[b].compare_exchange_strong(w, 0, std::memory_order_acq_rel);
}

// One transaction.  begin() hands out a private, validated copy of the current state; commit() publishes it with a
// single CAS on `cur` (false = lost the race: call begin() again).
struct Txn {
  gemhook_pool* p;
  int blk = -1;
  uint64_t claim = 0;  // CLAIMED(this handle's owner tag): our word on bctl[blk]
  uint64_t seen = 0;
  State* s = nullptr;

  explicit Txn(gemhook_pool* pool) : p(pool) {}
  ~Txn() { abort(); }
  Txn(const Txn&) = delete;
  Txn& operator=(const Txn&) = delete;

  State& begin() {
    Region* r = p->r;
    if (blk < 0) {
      claim = ctl_make(p->owner_tag(), 0);
      blk = p->claim_block(claim);
      GH_FAULT(FP_AFTER_CLAIM);
    }
    s = &r->blocks[blk];
    for (;;) {
      seen = r->h.cur.load(std::memory_order_acquire);
      gemhook_pool::copy_state(s, &r->blocks[seen & 0xff]);
      std::atomic_thread_fence(std::memory_order_acquire);
      if (r->h.cur.load(std::memory_order_relaxed) == seen) return *s;
    }
  }

  bool move(uint64_t from, uint64_t to) { return p->r->bctl[blk].compare_exchange_strong(from, to, std::memory_order_acq_rel); }
  bool publish(uint64_t seq) { return move(claim, claim | (seq & PUB_MASK)); }    // CLAIMED -> PUBLISHING(seq)
  bool unpublish(uint64_t seq) { return move(claim | (seq & PUB_MASK), claim); }  // PUBLISHING(seq) -> CLAIMED
  void abort() {                                                                   // CLAIMED -> FREE
    if (blk >= 0) move(claim, 0);
    blk = -1;
  }

  bool commit() {
    Region* r = p->r;
    uint64_t seq = next_seq(seen);
    if (!publish(seq)) {
      blk = -1;  // our block was recycled from under a stalled transaction: start over with a fresh one
      return false;
    }
    GH_FAULT(FP_BEFORE_CAS);
    uint64_t exp = seen;
    if (r->h.cur.compare_exchange_strong(exp, (seq << 8) | (uint64_t)blk, std::memory_order_acq_rel)) {
      GH_FAULT(FP_AFTER_CAS);
      retire(r, seen);
      r->h.commits.fetch_add(1, std::memory_order_relaxed);
      blk = -1;  // now the current block: not ours to touch any more
      return true;
    }
    r->h.conflicts.fetch_add(1, std::memory_order_relaxed);
    if (!unpublish(seq)) blk = -1;
    return false;
  }
};

// run `fn(Policy&)` as a transaction until it commits (or until it reports nothing to commit); returns fn's result
template <class F>
auto transact(gemhook_pool* p, F fn) -> decltype(fn(*(Policy*)nullptr)) {
  Txn t(p);
  for (;;) {
    Policy pol(t.begin(), p->r->h);
    auto rc = fn(pol);
    GH_FAULT(FP_MID_POLICY);
    if (!pol.dirty) return rc;
    if (t.commit()) return rc;
  }
}

// consistent view on a private copy: the same machinery, never committed (fn may scribble on the copy)
template <class F>
auto observe(const gemhook_pool* cp, F fn) -> decltype(fn(*(State*)nullptr)) {
  Txn t(const_cast<gemhook_pool*>(cp));
  return fn(t.begin());
}

// a few words of the current block read in place, without claiming anything: fn(block, its slot count clamped) runs
// until `cur` did not move meanwhile.  The block may be recycled and rewritten under fn, so fn is GH_NO_TSAN as well
template <class F>
GH_NO_TSAN auto read_current(const gemhook_pool* p, F fn) -> decltype(fn(*(const State*)nullptr, 0u)) {
  Region* r = p->r;
  for (;;) {
    uint64_t c = r->h.cur.load(std::memory_order_acquire);
    const State& s = r->blocks[c & 0xff];
    auto v = fn(s, s.nslots <= GEMHOOK_MAX_SLOTS ? s.nslots : (uint32_t)GEMHOOK_MAX_SLOTS);
    std::atomic_thread_fence(std::memory_order_acquire);
    if (r->h.cur.load(std::memory_order_relaxed) == c) return v;
  }
}

void wake_slot(gemhook_pool* p, int slot) {
  if (slot < 0 || slot >= GEMHOOK_MAX_SLOTS) return;
  p->r->shared[slot].wake.fetch_add(1, std::memory_order_release);
  futex(&p->r->shared[slot].wake, FUTEX_WAKE, INT_MAX, nullptr);
}

void reset_dynamic_state(gemhook_pool* p) {
  // the file outlived a reboot (hostPath): its clock origin, token holder, ledger, attachments, byte counters and
  // block claims describe processes that no longer exist.  Keep the configuration rows, drop the dynamic state.
  Region* r = p->r;
  Header& h = r->h;
  uint64_t c = h.cur.load();
  State& s = r->blocks[c & 0xff];
  for (uint32_t i = 0; i < s.nslots && i < GEMHOOK_MAX_SLOTS; i++) {
    PSlot& ps = s.slots[i];
    ps.quota = h.base_quota;
    ps.burst = 0;
    ps.last_start = ps.last_end = ps.closed_ms = 0;
    ps.grants = 0;
    ps.state = ST_IDLE;
    ps.poster = -1;
    ps.pod_quota = 0;
    ps.pod_token_us = 0;
    ps.pod_overuse = 0;
    r->shared[i].mem_used.store(0);
    r->shared[i].gpu_ns.store(0);
    r->shared[i].launches.store(0);
  }
  s.ledger_len = 0;
  s.holder = -1;
  s.deadline_ms = 0;
  memset((void*)r->attach, 0, sizeof(r->attach));
  for (uint32_t b = 0; b < NBLK; b++) r->bctl[b].store(b == (c & 0xff) ? ctl_make(NO_OWNER_TAG, c >> 8) : 0);
  h.start_ns.store(gh_now_ns());
}

// the owner's first step of closing: its entry reads FREE before the byte is unlocked (gemhook_pool_close)
void leave_attachment(gemhook_pool* p) {
  if (p->attach_idx >= 0) gemhook_pool_detach(p);
  p->r->attach[p->liveness_idx].in_use.store(FREE, std::memory_order_release);
}

}  // namespace

GH_EXPORT gemhook_pool* gemhook_pool_open(const char* path, int create, double base_quota_ms, double min_quota_ms,
                                          double window_ms, int64_t start_ns) {
  gemhook_pool* p = new gemhook_pool();
  size_t bytes = sizeof(Region);
  void* m = MAP_FAILED;
  bool fresh = false;
  if (!path || !*path) {  // private pool (tests, single-process use)
    m = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS, -1, 0);
    p->anonymous = true;
    fresh = true;
  } else {
    int fd = open(path, create ? (O_RDWR | O_CREAT) : O_RDWR, 0666);
    if (fd < 0) {
      gh_set_error("cannot open pool file %s: %s", path, strerror(errno));
      delete p;
      return nullptr;
    }
    struct stat st;
    fstat(fd, &st);
    if ((size_t)st.st_size < bytes) {
      if (!create || ftruncate(fd, (off_t)bytes) != 0) {
        gh_set_error("pool file %s is too small (%lld bytes) and may not be created", path, (long long)st.st_size);
        close(fd);
        delete p;
        return nullptr;
      }
    }
    m = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    p->fd = fd;
  }
  if (m == MAP_FAILED) {
    gh_set_error("mmap of the credit pool failed: %s", strerror(errno));
    if (p->fd >= 0) close(p->fd);
    delete p;
    return nullptr;
  }
  p->r = (Region*)m;
  Header& h = p->r->h;
  // first opener initialises: claim with CAS on magic (file content starts as zeros)
  uint64_t zero = 0;
  std::atomic<uint64_t>* magic = reinterpret_cast<std::atomic<uint64_t>*>(&h.magic);
  if (fresh || (create && magic->compare_exchange_strong(zero, POOL_MAGIC))) {
    h.magic = POOL_MAGIC;
    h.version = POOL_VERSION;
    h.nslots_max = GEMHOOK_MAX_SLOTS;
    h.base_quota = base_quota_ms;
    h.min_quota = min_quota_ms;
    h.window = window_ms;
    h.start_ns.store(start_ns ? start_ns : gh_now_ns());
    h.boot_id.store(boot_id_hash());
    State& s0 = p->r->blocks[0];
    s0.holder = -1;
    s0.nslots = 0;
    p->r->bctl[0].store(ctl_make(NO_OWNER_TAG, 1));
    h.cur.store((1ull << 8) | 0);
    h.ready.store(1, std::memory_order_release);
  } else {
    for (int i = 0; i < 20000 && !h.ready.load(std::memory_order_acquire); i++) usleep(100);
    if (h.magic != POOL_MAGIC || !h.ready.load() || h.version != POOL_VERSION) {
      gh_set_error("%s is not an initialised gemhook credit pool (layout version %u)", path, POOL_VERSION);
      gemhook_pool_close(p);
      return nullptr;
    }
    uint64_t mine = boot_id_hash();
    uint64_t seen = h.boot_id.load();
    if (seen != mine) {
      // one opener resets, the others wait for it (boot id 1 = reset in progress)
      if (seen != 1 && h.boot_id.compare_exchange_strong(seen, 1)) {
        reset_dynamic_state(p);
        h.boot_id.store(mine, std::memory_order_release);
      } else {
        for (int i = 0; i < 20000 && h.boot_id.load(std::memory_order_acquire) != mine; i++) usleep(100);
      }
    }
  }
  // a liveness byte for this handle's transactions (clients turn it into their own attachment in attach())
  if (p->fd >= 0) {
    p->liveness_idx = p->take_attachment(-1);
    if (p->liveness_idx < 0) {  // table full of entries whose owners are gone (crashed tools): clear them out, try again
      gemhook_pool_reap(p);
      p->liveness_idx = p->take_attachment(-1);
    }
  }
  return p;
}

GH_EXPORT void gemhook_pool_close(gemhook_pool* p) {
  if (!p) return;
  if (p->r) {
    if (p->liveness_idx >= 0) {
      leave_attachment(p);
      p->attach_byte(p->liveness_idx, F_OFD_SETLK, F_UNLCK);
    }
    munmap(p->r, sizeof(Region));
  }
  if (p->fd >= 0) close(p->fd);
  delete p;
}

// the part of the region the device should see: header + per-slot counters (page aligned)
void* gh_pool_region(gemhook_pool* p, size_t* bytes) {
  if (bytes) *bytes = (offsetof(Region, attach) + 4095) & ~(size_t)4095;
  return p ? (void*)p->r : nullptr;
}
// byte offset of slot 0's {mem_used, mem_limit} pair inside that part and the stride per slot (device-side mirror)
void gh_pool_shared_layout(size_t* offset, size_t* stride) {
  if (offset) *offset = offsetof(Region, shared);
  if (stride) *stride = sizeof(SlotShared);
}

// read_resource_config (scheduler.cpp:183-217): "N" then N rows "name c2 c3 mem"; a re-read replaces the
// client's ClientInfo, i.e. its adaptive quota restarts from the base quota; usage history is kept.  The reference
// never forgets a client; neither do we until the table is full -- then a slot whose pod has left the file, holds
// nothing and has nobody attached is given to the newcomer.  A row whose name does not fit is skipped (the reference
// overflows char[HOST_NAME_MAX] there), the others are still loaded.
static int load_config_stamped(gemhook_pool* p, const char* text, int swap_columns, uint64_t stamp);
GH_EXPORT int gemhook_pool_load_config(gemhook_pool* p, const char* text, int swap_columns) {
  return load_config_stamped(p, text, swap_columns, 0);
}
// stamp != 0: apply only if the pool's configuration does not carry this stamp yet -- of N clients that notice the same
// rewrite of the quota file together, exactly one reloads (a reload resets every client's adaptive quota, so a second,
// late one would be visible in the quota sequence).  Returns -2 when somebody else had already loaded this version.
static int load_config_stamped(gemhook_pool* p, const char* text, int swap_columns, uint64_t stamp) {
  if (!p || !text) return -1;
  const char* c = text;
  char* end = nullptr;
  long n = strtol(c, &end, 10);
  if (end == c || n < 0) {
    gh_set_error("quota file: bad client count");
    return -1;
  }
  c = end;
  struct Row {
    char name[64];
    double c2, c3;
    unsigned long long mem;
  };
  std::vector<Row> rows;
  long parsed = 0, skipped = 0;
  for (long i = 0; i < n; i++) {
    char name[256];
    Row rw;
    int used = 0;
    if (sscanf(c, " %255s %lf %lf %llu%n", name, &rw.c2, &rw.c3, &rw.mem, &used) != 4) break;
    c += used;
    parsed++;
    if (strlen(name) >= sizeof(rw.name)) {
      gh_set_error("quota file: pod name \"%.40s...\" is longer than %zu bytes; row skipped", name, sizeof(rw.name) - 1);
      skipped++;
      continue;
    }
    snprintf(rw.name, sizeof(rw.name), "%s", name);
    rows.push_back(rw);
  }
  bool full = false;
  uint64_t limits[GEMHOOK_MAX_SLOTS];
  uint32_t nlim = 0;
  bool reused[GEMHOOK_MAX_SLOTS];
  bool stale = false;
  int loaded = transact(p, [&](Policy& pol) {
    State& s = pol.s;
    int cnt = 0;
    full = false;
    stale = stamp != 0 && s.quota_stamp == stamp;
    if (stale) return 0;
    for (uint32_t i = 0; i < GEMHOOK_MAX_SLOTS; i++) reused[i] = false;
    for (uint32_t i = 0; i < s.nslots; i++) s.slots[i].listed = 0;
    // rows of clients we already know keep their slot; new names are placed afterwards
    std::vector<int> where(rows.size(), -1);
    for (size_t k = 0; k < rows.size(); k++)
      for (uint32_t i = 0; i < s.nslots; i++)
        if (!strncmp(s.slots[i].name, rows[k].name, sizeof(s.slots[i].name))) where[k] = (int)i;
    for (size_t k = 0; k < rows.size(); k++)
      if (where[k] >= 0) s.slots[where[k]].listed = 1;
    for (size_t k = 0; k < rows.size(); k++) {
      int idx = where[k];
      if (idx < 0) {
        for (size_t q = 0; q < k; q++)  // the same new name twice in one file: one slot
          if (where[q] >= 0 && !strcmp(rows[q].name, rows[k].name)) idx = where[q];
      }
      if (idx < 0 && s.nslots < GEMHOOK_MAX_SLOTS) {
        idx = (int)s.nslots++;
        memset((void*)&s.slots[idx], 0, sizeof(PSlot));
      } else if (idx < 0) {
        for (uint32_t i = 0; i < s.nslots && idx < 0; i++) {
          PSlot& ps = s.slots[i];
          if (ps.listed || ps.state != ST_IDLE || s.holder == (int)i) continue;
          if (p->r->shared[i].mem_used.load(std::memory_order_relaxed) != 0) continue;
          bool attached = false;
          for (uint32_t a = 0; a < MAX_ATTACH; a++)
            if (p->r->attach[a].in_use.load(std::memory_order_relaxed) && p->r->attach[a].slot.load(std::memory_order_relaxed) == (int)i)
              attached = true;
          if (attached) continue;
          idx = (int)i;  // the pod left the file and holds nothing: its slot goes to the newcomer
          uint32_t kk = 0;
          for (uint32_t e = 0; e < s.ledger_len; e++)
            if (s.ledger[e].slot != idx) s.ledger[kk++] = s.ledger[e];
          s.ledger_len = kk;
          memset((void*)&s.slots[idx], 0, sizeof(PSlot));
          reused[idx] = true;
        }
        if (idx < 0) {
          full = true;
          continue;
        }
      }
      where[k] = idx;
      PSlot& ps = s.slots[idx];
      if (!ps.name[0]) {
        snprintf(ps.name, sizeof(ps.name), "%s", rows[k].name);
        ps.poster = -1;
      }
      ps.min_frac = swap_columns ? rows[k].c3 : rows[k].c2;
      ps.max_frac = swap_columns ? rows[k].c2 : rows[k].c3;
      ps.mem_limit = rows[k].mem;
      ps.quota = pol.h.base_quota;
      ps.burst = 0.0;
      ps.configured = 1;
      ps.listed = 1;
      cnt++;
    }
    nlim = s.nslots;
    for (uint32_t i = 0; i < s.nslots; i++) limits[i] = s.slots[i].mem_limit;
    // a half-written file (fewer rows than announced) keeps the old stamp: it will be read again
    if (parsed == n && !full) s.quota_stamp = stamp;
    pol.dirty = true;
    return cnt;
  });
  if (stale) return -2;
  for (uint32_t i = 0; i < nlim; i++) {
    if (reused[i]) {
      p->r->shared[i].gpu_ns.store(0, std::memory_order_relaxed);
      p->r->shared[i].launches.store(0, std::memory_order_relaxed);
    }
    p->r->shared[i].mem_limit_mirror.store(limits[i], std::memory_order_relaxed);
  }
  if (full) gh_set_error("quota file lists more than %d clients and no departed client's slot is free", GEMHOOK_MAX_SLOTS);
  return (!full && parsed == n && loaded + skipped == n) ? (int)n : -1;
}

// Keep the pool in step with the quota file kubeshare-config rewrites (what gem-schd does with inotify,
// scheduler.cpp:219-265): cheap stat, reload only when the file's (mtime, size) stamp differs from the one recorded
// in the pool -- so of N co-resident clients only the first to notice reloads.  1 = reloaded, 0 = unchanged, -1 = error.
GH_EXPORT int gemhook_pool_sync_quota_file(gemhook_pool* p, const char* path, int swap_columns) {
  if (!p || !path || !*path) return -1;
  struct stat st;
  if (stat(path, &st) != 0) return -1;
  uint64_t stamp = ((uint64_t)st.st_mtim.tv_sec * 1000000000ULL + (uint64_t)st.st_mtim.tv_nsec) * 31ULL + (uint64_t)st.st_size + 1;
  if (p->r->h.quota_stamp.load(std::memory_order_acquire) == stamp) return 0;
  FILE* f = fopen(path, "r");
  if (!f) return -1;
  char* text = (char*)calloc(1, 1 << 16);
  size_t n = fread(text, 1, (1 << 16) - 1, f);
  fclose(f);
  text[n] = 0;
  int rc = load_config_stamped(p, text, swap_columns, stamp);
  free(text);
  if (rc == -2) {  // another client loaded this very version while we were reading the file
    p->r->h.quota_stamp.store(stamp, std::memory_order_release);
    return 0;
  }
  if (rc < 0) return -1;  // half-written file: keep the old stamp, try again at the next renewal
  p->r->h.quota_stamp.store(stamp, std::memory_order_release);
  return 1;
}

GH_EXPORT int gemhook_pool_find(const gemhook_pool* p, const char* name) {
  return observe(p, [&](const State& s) {
    for (uint32_t i = 0; i < s.nslots; i++)
      if (!strncmp(s.slots[i].name, name, sizeof(s.slots[i].name))) return (int)i;
    return -1;
  });
}
GH_EXPORT int gemhook_pool_nslots(const gemhook_pool* p) { return read_current(p, [](const State&, uint32_t n) { return (int)n; }); }

GH_EXPORT int gemhook_pool_request(gemhook_pool* p, int slot, double now_ms, double overuse_ms, double burst_ms) {
  if (!p || slot < 0 || slot >= gemhook_pool_nslots(p)) return -1;
  transact(p, [&](Policy& pol) {
    pol.request(slot, now_ms, overuse_ms, burst_ms, -1);
    return 0;
  });
  return 0;
}

GH_EXPORT int gemhook_pool_schedule(gemhook_pool* p, double now_ms, int* slot_out, double* quota_out, double* sleep_ms_out) {
  int who = -1;
  int rc = transact(p, [&](Policy& pol) {
    who = -1;
    return pol.schedule(now_ms, &who, quota_out, sleep_ms_out);
  });
  if (rc == 1) {
    if (slot_out) *slot_out = who;
    wake_slot(p, who);
  }
  return rc;
}

GH_EXPORT double gemhook_pool_usage(gemhook_pool* p, int slot, double now_ms) {
  // window_usage prunes the ledger: on the private copy, so asking for a number does not change the pool
  return observe(p, [&](State& s) {
    double usage[GEMHOOK_MAX_SLOTS] = {0}, a, b;
    Policy(s, p->r->h).window_usage(now_ms, usage, a, b);
    return (slot >= 0 && slot < GEMHOOK_MAX_SLOTS) ? usage[slot] : 0.0;
  });
}

GH_EXPORT size_t gemhook_pool_history(const gemhook_pool* cp, int* slots, double* starts, double* ends, size_t cap) {
  return observe(cp, [&](const State& s) {
    size_t n = s.ledger_len;
    for (size_t i = 0; i < n && i < cap; i++) {
      if (slots) slots[i] = s.ledger[i].slot;
      if (starts) starts[i] = s.ledger[i].start;
      if (ends) ends[i] = s.ledger[i].end;
    }
    return n;
  });
}

GH_EXPORT double gemhook_pool_now_ms(const gemhook_pool* p) { return p ? p->now_ms() : 0.0; }

GH_EXPORT double gemhook_pool_accumulated_ms(const gemhook_pool* cp, int slot) {
  if (slot < 0 || slot >= GEMHOOK_MAX_SLOTS) return 0.0;
  return observe(cp, [&](const State& s) {
    const PSlot& ps = s.slots[slot];
    return ps.grants ? ps.closed_ms + (ps.last_end - ps.last_start) : 0.0;
  });
}

GH_EXPORT int gemhook_pool_pod_launch(gemhook_pool* p, int slot, int64_t now_us, double overuse_ms, double burst_ms,
                                      double* fwd_overuse_ms, double* fwd_burst_ms, double* remain_ms) {
  return transact(p, [&](Policy& pol) {
    return pod_launch(p->r->attach, pol, slot, p->attach_idx, now_us, overuse_ms, burst_ms, fwd_overuse_ms, fwd_burst_ms, remain_ms);
  });
}
GH_EXPORT double gemhook_pool_pod_granted(gemhook_pool* p, int slot, int64_t now_us, double quota_ms) {
  return transact(p, [&](Policy& pol) { return pod_granted(pol, slot, now_us, quota_ms); });
}

// ---- live acquisition ---------------------------------------------------------------------------------------------
GH_EXPORT double gemhook_pool_acquire(gemhook_pool* p, int slot, double overuse_ms, double burst_ms) {
  return gemhook_pool_acquire_ex(p, slot, overuse_ms, burst_ms, nullptr);
}

// Post the request, then arbitrate / wait until OUR request is granted.  Processes of one pod share the slot's
// mailbox: only one request per pod is in flight (what gem-pmgr's sleeping_count hand-shake serialises,
// pod-manager.cpp:316-473); a sibling that arrives meanwhile waits for that grant and is then normally answered from
// the fresh pod token.
GH_EXPORT double gemhook_pool_acquire_ex(gemhook_pool* p, int slot, double overuse_ms, double burst_ms, int* forwarded) {
  if (forwarded) *forwarded = 1;
  // identity of a request in flight: the poster's attachment; an unattached handle (gem-arbiter serving TCP clients,
  // tests) tags its requests with -2 - slot so that a sibling thread is still told apart from "nobody"
  const int me = p->attach_idx >= 0 ? p->attach_idx : -2;
  SlotShared& sh = p->r->shared[slot];
  enum { ANSWERED, POSTED, BUSY_SIBLING };
  struct MailView { uint32_t state; int32_t poster; };
  int idle_rounds = 0;
  for (;;) {
    // ---- phase 1: pod rule, post, first decision -- one transaction
    double remain = 0.0;
    int granted_to = -1;
    int st = transact(p, [&](Policy& pol) {
      granted_to = -1;
      PSlot& ps = pol.s.slots[slot];
      if (ps.state != ST_IDLE) return (int)BUSY_SIBLING;  // a request of this pod is already in flight
      double fo = overuse_ms, fb = burst_ms;
      if (!pod_launch(p->r->attach, pol, slot, p->attach_idx, p->now_us(), overuse_ms, burst_ms, &fo, &fb, &remain)) return (int)ANSWERED;
      double now = p->now_ms();
      pol.request(slot, now, fo, fb, me);
      pol.schedule(now, &granted_to, nullptr, nullptr);
      return (int)POSTED;
    });
    if (granted_to >= 0 && granted_to != slot) wake_slot(p, granted_to);
    if (st == ANSWERED) {
      if (forwarded) *forwarded = 0;
      return remain;  // the pod's token still covers this burst (pod-manager.cpp:472)
    }
    const bool mine = st == POSTED;
    // ---- phase 2: wait for the grant of the request in flight
    for (;;) {
      uint32_t w0 = sh.wake.load(std::memory_order_acquire);
      MailView v = read_current(p, [&](const State& s, uint32_t) GH_NO_TSAN { return MailView{s.slots[slot].state, s.slots[slot].poster}; });
      if (v.state == ST_GRANTED && mine && v.poster == me) {
        bool took = false;
        double got = transact(p, [&](Policy& pol) {
          PSlot& ps = pol.s.slots[slot];
          took = false;
          if (ps.state != ST_GRANTED || ps.poster != me) return 0.0;  // reaped meanwhile
          took = true;
          double q = ps.granted_quota;
          ps.state = ST_IDLE;
          ps.poster = -1;
          return pod_granted(pol, slot, p->now_us(), q);
        });
        if (took) {
          wake_slot(p, slot);  // siblings waiting for this grant re-evaluate the pod rule
          return got;
        }
        break;  // start over
      }
      if (v.state == ST_IDLE) break;  // the request in flight is gone (consumed by its poster, or reaped): start over
      if (!mine && v.poster >= 0 && v.poster != p->attach_idx && !p->entry_alive(v.poster)) gemhook_pool_reap(p);
      // drive the policy: whoever waits runs the decisions (there is no daemon)
      int who = -1;
      double sleep_ms = 0;
      int rc = transact(p, [&](Policy& pol) {
        who = -1;
        return pol.schedule(p->now_ms(), &who, nullptr, &sleep_ms);
      });
      if (rc == 1) {
        wake_slot(p, who);
        if (who == slot) continue;
      }
      if (++idle_rounds % 8 == 0) gemhook_pool_reap(p);  // a dead holder must not stall everybody until its deadline
      // someone else holds the token, or everyone is throttled: wait on our slot's wake word until the hint expires
      // or a granter wakes us.  Short waits spin (no context switch on a quick hand-over).
      double wait_ms = (rc == 0 || rc == -2) ? sleep_ms : 0.2;
      if (wait_ms < 0.05) {
        for (int i = 0; i < 200 && sh.wake.load(std::memory_order_acquire) == w0; i++) __builtin_ia32_pause();
        continue;
      }
      if (wait_ms > 50.0) wait_ms = 50.0;  // re-evaluate periodically (config reloads, dead holders)
      struct timespec ts;
      ts.tv_sec = (time_t)(wait_ms / 1e3);
      ts.tv_nsec = (long)((wait_ms - ts.tv_sec * 1e3) * 1e6);
      futex(&sh.wake, FUTEX_WAIT, w0, &ts);
    }
  }
}

// ---- attachments ------------------------------------------------------------------------------------------
GH_EXPORT int gemhook_pool_attach(gemhook_pool* p, int slot) {
  if (!p || slot < 0) return -1;
  if (p->attach_idx >= 0) return p->attach_idx;
  int idx;
  if (p->liveness_idx >= 0) {  // the handle's observer entry becomes the client attachment: its OFD byte is already held
    idx = p->liveness_idx;
    p->r->attach[idx].bytes.store(0);
    p->r->attach[idx].burst_bits.store(0);
    p->r->attach[idx].slot.store(slot, std::memory_order_release);
  } else {
    idx = p->take_attachment(slot);
    if (idx < 0) {
      gh_set_error("credit pool: more than %u attached processes", MAX_ATTACH);
      return -1;
    }
    p->liveness_idx = idx;
  }
  p->attach_idx = idx;
  return idx;
}

GH_EXPORT void gemhook_pool_detach(gemhook_pool* p) {
  if (!p || p->attach_idx < 0) return;
  Attach& a = p->r->attach[p->attach_idx];
  uint64_t left = a.bytes.exchange(0);
  int slot = a.slot.load();
  if (left && slot >= 0) p->r->shared[slot].mem_used.fetch_sub(left, std::memory_order_acq_rel);  // exit without freeing
  a.burst_bits.store(0);
  a.slot.store(-1, std::memory_order_release);  // back to a plain observer entry: the handle may still run transactions
  p->attach_idx = -1;
}

static bool slot_has_other_live_attachment(gemhook_pool* p, int slot, int except) {
  for (uint32_t j = 0; j < MAX_ATTACH; j++) {
    if ((int)j == except) continue;
    Attach& o = p->r->attach[j];
    if (o.in_use.load(std::memory_order_acquire) == LIVE && o.slot.load(std::memory_order_relaxed) == slot && p->entry_alive((int)j)) return true;
  }
  return false;
}

// LIVE -> REAPING for an entry whose owner is dead: the reaper takes the entry's byte, which it can only once the owner
// is gone, and holds it until finish_reap.  A private pool has no file: all its entries are this process's.
static bool start_reap(gemhook_pool* p, uint32_t i) {
  Attach& a = p->r->attach[i];
  if (p->fd < 0 || (int)i == p->attach_idx || (int)i == p->liveness_idx || a.in_use.load(std::memory_order_acquire) != LIVE) return false;
  if (!p->attach_byte((int)i, F_OFD_SETLK, F_WRLCK)) return false;  // the owner lives, or a taker or reaper holds it
  if (attach_move(a, LIVE, REAPING)) return true;
  p->attach_byte((int)i, F_OFD_SETLK, F_UNLCK);
  return false;
}

// reclaim the bytes, the request and, if nobody of its pod is left, the token of the entry start_reap took, then
// REAPING -> FREE; 1 if it was a client's.  The blocks it had claimed go back in gemhook_pool_reap's recycle_blocks.
static int finish_reap(gemhook_pool* p, uint32_t i) {
  Attach& a = p->r->attach[i];
  uint64_t left = a.bytes.exchange(0);
  int slot = a.slot.load();
  if (slot >= 0 && slot < GEMHOOK_MAX_SLOTS) {
    if (left) p->r->shared[slot].mem_used.fetch_sub(left, std::memory_order_acq_rel);
    bool others = slot_has_other_live_attachment(p, slot, (int)i);
    int woken = -1;
    transact(p, [&](Policy& pol) {
      PSlot& ps = pol.s.slots[slot];
      woken = -1;
      if (ps.state != ST_IDLE && ps.poster == (int)i) {  // its request / unconsumed grant dies with it
        ps.state = ST_IDLE;
        ps.poster = -1;
        pol.dirty = true;
      }
      if (!others && pol.s.holder == slot) {
        pol.s.holder = -1;
        ps.pod_quota = 0.0;
        if (ps.state != ST_IDLE) {
          ps.state = ST_IDLE;
          ps.poster = -1;
        }
        pol.dirty = true;
        pol.schedule(p->now_ms(), &woken, nullptr, nullptr);
      }
      return 0;
    });
    wake_slot(p, slot);
    if (woken >= 0) wake_slot(p, woken);
  }
  attach_move(a, REAPING, FREE);
  p->attach_byte((int)i, F_OFD_SETLK, F_UNLCK);
  return slot >= 0 && slot < GEMHOOK_MAX_SLOTS;  // (observer entries of dead tools are recycled without being counted)
}

// reclaim what dead processes left behind: their bytes, the request they posted, the token if their pod held it and
// nobody of the pod is left, and the state blocks they had claimed
GH_EXPORT int gemhook_pool_reap(gemhook_pool* p) {
  if (!p) return 0;
  int reaped = 0;
  for (uint32_t i = 0; i < MAX_ATTACH; i++)
    if (start_reap(p, i)) reaped += finish_reap(p, i);
  p->recycle_blocks();
  return reaped;
}

// A client that is going away (process exit) hands its token back instead of letting the scheduler wait
// for the quota to time out (the reference can only time out: scheduler.cpp:507-510).  While another live process of
// the same pod is attached the pod keeps its token (they share it, pod-manager.cpp:316-473): nothing is released.
GH_EXPORT void gemhook_pool_release(gemhook_pool* p, int slot) {
  if (!p || slot < 0 || slot >= GEMHOOK_MAX_SLOTS) return;
  if (p->attach_idx >= 0 && slot_has_other_live_attachment(p, slot, p->attach_idx)) return;
  int who = -1;
  transact(p, [&](Policy& pol) {
    who = -1;
    double now = p->now_ms();
    if (pol.give_back(slot, now)) pol.schedule(now, &who, nullptr, nullptr);
    return 0;
  });
  if (who >= 0) wake_slot(p, who);
  wake_slot(p, slot);
}

// The outstanding token is declared timed out (what gem-schd concludes when its timedwait on the holder
// returns ETIMEDOUT, scheduler.cpp:507-510) without touching the ledger: trace replays use it to decouple
// decisions from wall time, a node agent can use it to revoke the token of a client it knows is dead.
GH_EXPORT void gemhook_pool_expire_token(gemhook_pool* p) {
  if (!p) return;
  transact(p, [&](Policy& pol) {
    if (pol.s.holder != -1) {
      pol.s.holder = -1;
      pol.dirty = true;
    }
    return 0;
  });
}

// 1 if some OTHER client is waiting for the token right now (a peek, used by the yield-on-idle option)
GH_EXPORT int gemhook_pool_others_waiting(const gemhook_pool* p, int slot) {
  return read_current(p, [&](const State& s, uint32_t n) GH_NO_TSAN {
    int any = 0;
    for (uint32_t i = 0; i < n; i++)
      if ((int)i != slot && s.slots[i].state == ST_WAITING) any = 1;
    return any;
  });
}

// ---- gpu_mem cap: integer exact, requested bytes (hook.cpp:590-617, pod-manager.cpp:295-313) -----------
GH_EXPORT int gemhook_pool_mem_reserve(gemhook_pool* p, int slot, uint64_t bytes) {
  SlotShared& sh = p->r->shared[slot];
  const uint64_t limit = read_current(p, [&](const State& s, uint32_t) GH_NO_TSAN { return s.slots[slot].mem_limit; });
  uint64_t used = sh.mem_used.load(std::memory_order_relaxed);
  for (;;) {
    // reference pre-hook: remain = limit - used; deny iff bytes > remain (hook.cpp:593-598).  A quota-file reload may
    // have lowered the limit below what is already in use: then nothing more fits (gem-pmgr: used + bytes > limit,
    // pod-manager.cpp:299) -- the unsigned subtraction must not wrap into "plenty of room".
    if (used > limit || bytes > limit - used) return 0;
    if (sh.mem_used.compare_exchange_weak(used, used + bytes, std::memory_order_acq_rel)) {
      if (p->attach_idx >= 0 && p->r->attach[p->attach_idx].slot.load(std::memory_order_relaxed) == slot)
        p->r->attach[p->attach_idx].bytes.fetch_add(bytes, std::memory_order_relaxed);
      return 1;
    }
  }
}
GH_EXPORT void gemhook_pool_mem_release(gemhook_pool* p, int slot, uint64_t bytes) {
  p->r->shared[slot].mem_used.fetch_sub(bytes, std::memory_order_acq_rel);
  if (p->attach_idx >= 0 && p->r->attach[p->attach_idx].slot.load(std::memory_order_relaxed) == slot)
    p->r->attach[p->attach_idx].bytes.fetch_sub(bytes, std::memory_order_relaxed);
}
GH_EXPORT void gemhook_pool_mem_info(const gemhook_pool* p, int slot, uint64_t* used, uint64_t* limit) {
  if (used) *used = p->r->shared[slot].mem_used.load(std::memory_order_acquire);
  if (limit) *limit = read_current(p, [&](const State& s, uint32_t) GH_NO_TSAN { return s.slots[slot].mem_limit; });
}
GH_EXPORT int gemhook_pool_slot_info(const gemhook_pool* cp, int slot, gemhook_slot_info* out) {
  if (!cp || !out || slot < 0 || slot >= GEMHOOK_MAX_SLOTS) return -1;
  const SlotShared& sh = cp->r->shared[slot];
  return observe(cp, [&](const State& s) {
    if (slot >= (int)s.nslots) return -1;
    const PSlot& ps = s.slots[slot];
    memset(out, 0, sizeof(*out));
    snprintf(out->name, sizeof(out->name), "%s", ps.name);
    out->min_frac = ps.min_frac;
    out->max_frac = ps.max_frac;
    out->mem_limit = ps.mem_limit;
    out->mem_used = sh.mem_used.load(std::memory_order_relaxed);
    out->gpu_ns = sh.gpu_ns.load(std::memory_order_relaxed);
    out->launches = sh.launches.load(std::memory_order_relaxed);
    out->tokens = ps.grants;
    out->quota_ms = ps.quota;
    out->accumulated_ms = ps.grants ? ps.closed_ms + (ps.last_end - ps.last_start) : 0.0;
    out->holds_token = s.holder == slot ? 1 : 0;
    out->waiting = ps.state == ST_WAITING ? 1 : 0;
    return 0;
  });
}

// transaction statistics of the pool: commits, lost publication races, recycled (leaked and recovered) state blocks
GH_EXPORT void gemhook_pool_counters(const gemhook_pool* p, uint64_t* commits, uint64_t* conflicts, uint64_t* recycled) {
  if (commits) *commits = p->r->h.commits.load(std::memory_order_relaxed);
  if (conflicts) *conflicts = p->r->h.conflicts.load(std::memory_order_relaxed);
  if (recycled) *recycled = p->r->h.recycled.load(std::memory_order_relaxed);
}

GH_EXPORT const void* gemhook_pool_shared_words(const gemhook_pool* p, int slot) {
  return (p && slot >= 0 && slot < GEMHOOK_MAX_SLOTS) ? (const void*)&p->r->shared[slot] : nullptr;
}

void gh_pool_add_usage(gemhook_pool* p, int slot, uint64_t gpu_ns, uint64_t launches) {
  p->r->shared[slot].gpu_ns.fetch_add(gpu_ns, std::memory_order_relaxed);
  p->r->shared[slot].launches.fetch_add(launches, std::memory_order_relaxed);
}

// hook.cpp:638-680: bytes charged for arrays.  CUarray_format: U8 0x01, U16 0x02, U32 0x03, S8 0x08,
// S16 0x09, S32 0x0a, HALF 0x10, FLOAT 0x20; any other format is outside the reference's switch
// (undefined there) and is charged 0 bytes here.
GH_EXPORT uint64_t gemhook_array_bytes(uint64_t w, uint64_t h, uint64_t d, uint32_t channels, uint32_t format, int is3d) {
  uint64_t fs;
  switch (format) {
    case 0x01: case 0x08: fs = 1; break;
    case 0x02: case 0x09: case 0x10: fs = 2; break;
    case 0x03: case 0x0a: case 0x20: fs = 4; break;
    default: fs = 0; break;
  }
  return (is3d ? w * h * d * channels : w * h * channels) * fs;
}

// Opt-in rule for mipmapped arrays (GEMHOOK_ACCOUNT_MANAGED=1; the reference charges nothing, hook.cpp:682-694): the
// array rule above applied to every level, extents halving (floor, at least 1) from one level to the next.
GH_EXPORT uint64_t gemhook_mipmap_bytes(uint64_t w, uint64_t h, uint64_t d, uint32_t channels, uint32_t format, uint32_t levels) {
  uint64_t total = 0;
  for (uint32_t l = 0; l < levels; l++) {
    uint64_t lw = w >> l ? w >> l : 1, lh = h ? (h >> l ? h >> l : 1) : 0, ld = d ? (d >> l ? d >> l : 1) : 0;
    total += gemhook_array_bytes(lw, lh ? lh : 1, ld ? ld : 1, channels, format, 1);
  }
  return total;
}
