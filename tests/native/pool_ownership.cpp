// tests/native/pool_ownership.cpp -- TEST: the ownership protocol of the credit pool's shared entries, one race at a time.
//
//   pool_ownership CASE DIR        CASE = a | b | c | d, DIR = a scratch directory for the pool file
//
// Each case drives the interleaving that used to go wrong step by step, through the transition functions of
// gh_pool.cpp (included here, so that the anonymous namespace is reachable), and exits 0 iff the protocol held:
//   a  a committer that was preempted between its publication CAS and freeing the block it superseded must not free
//      that block once somebody else has recycled and claimed it (one process, two handles);
//   b  the same across processes: a client stopped (SIGSTOP) at FP_AFTER_CAS, resumed after the parent recycled and
//      claimed every free block;
//   c  a recycler that judged a dead owner's control word must not free the block after the owner's attachment entry was
//      re-taken and the block claimed under the same index; a dead owner's blocks are recycled even when its entry is
//      re-taken between reaping the entry and recycling the blocks;
//   d  an entry that is no longer REAPING is not freed by the reaper's last step, and a closing owner's entry reads FREE
//      while its byte is still locked (so no reaper and no taker touches it in between).
#include "../../kubeshare_b200/csrc/gh_pool.cpp"

#include <signal.h>
#include <sys/wait.h>

#include <string>

extern "C" {
int gemhook_fault_point = 0;
long gemhook_fault_countdown = 0;
}

#define CHECK(c)                                                               \
  do {                                                                         \
    if (!(c)) {                                                                \
      fprintf(stderr, "%s:%d: check failed: %s\n", __FILE__, __LINE__, #c);    \
      exit(1);                                                                 \
    }                                                                          \
  } while (0)

static std::string g_path;

static gemhook_pool* open_pool(bool create) {
  gemhook_pool* p = create ? gemhook_pool_open(g_path.c_str(), 1, 300.0, 20.0, 10000.0, 0) : gemhook_pool_open(g_path.c_str(), 0, 0, 0, 0, 0);
  CHECK(p && p->liveness_idx >= 0);
  return p;
}

static int free_blocks(gemhook_pool* p) {
  int n = 0;
  for (uint32_t b = 0; b < NBLK; b++) n += p->r->bctl[b].load() == 0;
  return n;
}

// claim every free block with p's claim word
static std::vector<int> claim_all(gemhook_pool* p, uint64_t word) {
  std::vector<int> got;
  for (int n = free_blocks(p); n > 0; n--) got.push_back(p->claim_block(word));
  return got;
}

static bool has(const std::vector<int>& v, int x) { return std::find(v.begin(), v.end(), x) != v.end(); }

// wait (at most 10 s) until child `pid` stops (stopped = true) or exits; false on timeout
static bool wait_child(pid_t pid, bool stopped, int* status) {
  for (int i = 0; i < 10000; i++) {
    pid_t d = waitpid(pid, status, WNOHANG | (stopped ? WUNTRACED : 0));
    if (d == pid) return true;
    usleep(1000);
  }
  return false;
}

// a process that opens the pool, claims `nblocks` state blocks and dies (SIGKILL) holding them: its attachment entry
// stays LIVE with the byte unlocked.  Returns the entry's index; the blocks go to `blocks`.
static int dead_owner(int nblocks, std::vector<int>* blocks) {
  int* out = (int*)mmap(nullptr, 4096, PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS, -1, 0);
  CHECK(out != MAP_FAILED);
  out[0] = -1;
  pid_t pid = fork();
  if (pid == 0) {
    gemhook_pool* x = gemhook_pool_open(g_path.c_str(), 0, 0, 0, 0, 0);
    if (!x) _exit(3);
    for (int k = 0; k < nblocks; k++) out[2 + k] = x->claim_block(ctl_make(x->owner_tag(), 0));
    out[1] = nblocks;
    out[0] = x->liveness_idx;
    raise(SIGKILL);
  }
  int st;
  CHECK(wait_child(pid, false, &st) && WIFSIGNALED(st) && out[0] >= 0);
  int idx = out[0];
  if (blocks) blocks->assign(out + 2, out + 2 + out[1]);
  munmap(out, 4096);
  return idx;
}

// a: committer A wins the publication CAS and is preempted before freeing the superseded block; B recycles that block
// (its publication is resolved) and claims it; then A frees "the superseded block".
static void case_a() {
  gemhook_pool* a = open_pool(true);
  gemhook_pool* b = open_pool(false);
  CHECK(gemhook_pool_load_config(a, "1\nns/a 1.0 1.0 100\n", 0) == 1);
  Region* r = a->r;
  Txn t(a);
  t.begin().deadline_ms += 1.0;
  uint64_t seen = t.seen, seq = next_seq(seen);
  CHECK(t.publish(seq));
  uint64_t exp = seen;
  CHECK(r->h.cur.compare_exchange_strong(exp, (seq << 8) | (uint64_t)t.blk));
  t.blk = -1;  // the block is current now (Txn::commit does the same)
  int old = (int)(seen & 0xff);

  CHECK(b->recycle_blocks() >= 1 && r->bctl[old].load() == 0);
  uint64_t bw = ctl_make(b->owner_tag(), 0);
  std::vector<int> mine = claim_all(b, bw);
  CHECK(has(mine, old));

  retire(r, seen);  // A resumes
  for (int blk : mine) CHECK(r->bctl[blk].load() == bw);
  for (int blk : mine)
    if (blk != old) r->bctl[blk].store(0);
  std::vector<int> more = claim_all(a, ctl_make(a->owner_tag(), 0));
  CHECK(!more.empty() && !has(more, old) && r->bctl[old].load() == bw);
  for (int blk : more) r->bctl[blk].store(0);
  r->bctl[old].store(0);
  gemhook_pool_close(b);
  gemhook_pool_close(a);
}

// b: a child commits and is stopped right after its publication CAS; the parent reaps, recycles, claims every free block
// and lets the child go on.
static void case_b() {
  gemhook_pool* p = open_pool(true);
  CHECK(gemhook_pool_load_config(p, "2\nns/a 0.5 1.0 100\nns/b 0.5 1.0 100\n", 0) == 2);
  Region* r = p->r;
  pid_t pid = fork();
  if (pid == 0) {
    gemhook_pool* c = gemhook_pool_open(g_path.c_str(), 0, 0, 0, 0, 0);
    if (!c) _exit(3);
    gemhook_fault_signal = SIGSTOP;
    gemhook_fault_countdown = 1;
    gemhook_fault_point = FP_AFTER_CAS;
    gemhook_pool_request(c, 1, 1.0, 0.0, 1.0);
    gemhook_fault_point = 0;
    gemhook_pool_close(c);
    _exit(0);
  }
  int st = 0;
  if (!wait_child(pid, true, &st) || !WIFSTOPPED(st)) {
    kill(pid, SIGKILL);
    waitpid(pid, &st, 0);
    CHECK(!"the child did not stop at FP_AFTER_CAS");
  }
  gemhook_pool_reap(p);
  uint64_t pw = ctl_make(p->owner_tag(), 0);
  std::vector<int> mine = claim_all(p, pw);
  CHECK(mine.size() == NBLK - 1);
  kill(pid, SIGCONT);
  bool done = wait_child(pid, false, &st);
  if (!done) {
    kill(pid, SIGKILL);
    waitpid(pid, &st, 0);
  }
  CHECK(done && WIFEXITED(st) && WEXITSTATUS(st) == 0);
  for (int blk : mine) CHECK(r->bctl[blk].load() == pw);  // no block is claimed twice
  for (int blk : mine) r->bctl[blk].store(0);
  // `cur` names a block whose word records that very publication, and the pool still commits
  uint64_t c = r->h.cur.load();
  CHECK(ctl_pub(r->bctl[c & 0xff].load()) == ((c >> 8) & PUB_MASK));
  gemhook_slot_info info;
  CHECK(gemhook_pool_slot_info(p, 1, &info) == 0 && info.waiting == 1);
  uint64_t commits0, commits1;
  gemhook_pool_counters(p, &commits0, nullptr, nullptr);
  CHECK(gemhook_pool_request(p, 0, 2.0, 0.0, 1.0) == 0);
  gemhook_pool_counters(p, &commits1, nullptr, nullptr);
  CHECK(commits1 == commits0 + 1 && gemhook_pool_slot_info(p, 0, &info) == 0 && info.waiting == 1);
  gemhook_pool_close(p);
}

// c: the recycler's judgement and its CAS, with the owner's entry re-taken in between
static void case_c() {
  gemhook_pool* p = open_pool(true);
  gemhook_pool* rec = open_pool(false);
  Region* r = p->r;
  std::vector<int> blocks;
  int xi = dead_owner(1, &blocks);
  int b = blocks[0];
  uint64_t w = r->bctl[b].load();
  CHECK(w != 0 && rec->never_current((uint32_t)b, w));  // judged: dead owner ... and the recycler is preempted
  CHECK(gemhook_pool_reap(p) == 0 && r->bctl[b].load() == 0);
  gemhook_pool* y = open_pool(false);  // re-takes the dead owner's entry
  CHECK(y->liveness_idx == xi);
  uint64_t yw = ctl_make(y->owner_tag(), 0);
  std::vector<int> mine = claim_all(y, yw);
  CHECK(has(mine, b));
  CHECK(!rec->recycle((uint32_t)b, w) && r->bctl[b].load() == yw);  // the recycler resumes
  for (int blk : mine) r->bctl[blk].store(0);
  gemhook_pool_close(y);

  // the entry is reaped, then re-taken before the blocks are recycled
  xi = dead_owner(2, &blocks);
  CHECK(start_reap(p, (uint32_t)xi));
  finish_reap(p, (uint32_t)xi);
  y = open_pool(false);
  CHECK(y->liveness_idx == xi);
  CHECK(p->recycle_blocks() == 2 && r->bctl[blocks[0]].load() == 0 && r->bctl[blocks[1]].load() == 0);
  gemhook_pool_close(y);
  gemhook_pool_close(rec);
  gemhook_pool_close(p);
}

// d: the attachment lifecycle's two guarantees
static void case_d() {
  gemhook_pool* p = open_pool(true);
  Region* r = p->r;
  // a reaper's last step moves only an entry that is still REAPING
  int xi = dead_owner(0, nullptr);
  CHECK(start_reap(p, (uint32_t)xi) && r->attach[xi].in_use.load() == REAPING);
  r->attach[xi].in_use.store(LIVE);  // stands in for a re-take
  finish_reap(p, (uint32_t)xi);
  CHECK(r->attach[xi].in_use.load() == LIVE);
  r->attach[xi].in_use.store(FREE);

  // closing: between its two steps the entry reads FREE while its byte is still locked
  gemhook_pool* b = open_pool(false);
  gemhook_pool* c = open_pool(false);
  int bi = b->liveness_idx;
  CHECK(gemhook_pool_load_config(p, "1\nns/a 1.0 1.0 100\n", 0) == 1 && gemhook_pool_attach(b, 0) == bi);
  CHECK(gemhook_pool_mem_reserve(b, 0, 10) == 1);
  leave_attachment(b);
  CHECK(c->r->attach[bi].in_use.load() == FREE && c->attach_byte(bi, F_OFD_GETLK, F_WRLCK));
  uint64_t used, limit;
  gemhook_pool_mem_info(c, 0, &used, &limit);
  CHECK(used == 0 && gemhook_pool_reap(c) == 0 && c->r->attach[bi].in_use.load() == FREE);
  gemhook_pool* d = open_pool(false);  // a taker passes it by
  CHECK(d->liveness_idx != bi);
  gemhook_pool_close(b);
  CHECK(!c->attach_byte(bi, F_OFD_GETLK, F_WRLCK) && c->r->attach[bi].in_use.load() == FREE);
  gemhook_pool_close(d);
  gemhook_pool_close(c);
  gemhook_pool_close(p);
}

int main(int argc, char** argv) {
  if (argc < 3) {
    fprintf(stderr, "usage: pool_ownership a|b|c|d DIR\n");
    return 2;
  }
  g_path = std::string(argv[2]) + "/ownership.pool";
  unlink(g_path.c_str());
  switch (argv[1][0]) {
    case 'a': case_a(); break;
    case 'b': case_b(); break;
    case 'c': case_c(); break;
    case 'd': case_d(); break;
    default: return 2;
  }
  unlink(g_path.c_str());
  printf("ok\n");
  return 0;
}
