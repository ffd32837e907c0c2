// gh_policy.h -- the serial token policy of the credit pool, on ONE state block (a transaction's private copy), and
// the layout of that block.  Internal: included by gh_pool.cpp once the region's Header (scheduler parameters) and
// Attach (per-process bursts) are defined; how blocks are shared between processes is gh_pool.cpp's business.
//
// What stays the reference's (bit-exact, see tests/test_pool_policy.py against the oracle and the goldens):
//   * per-client adaptive quota        scheduler.cpp:160-174  (EMA 0.5, clamp [min_quota, max_frac*window])
//   * ledger of granted tokens          scheduler.cpp:144-153  Record(); :123-142 update_return_time()
//   * windowed usage with overlap split scheduler.cpp:281-367
//   * eligibility + ordering            scheduler.cpp:369-398, schd-priority.cpp:19-26
//   * ONE outstanding token per GPU     scheduler.cpp:461-529
//   * pod-level token                   pod-manager.cpp:316-473
//   * gpu_mem counter, requested bytes  pod-manager.cpp:295-313, hook.cpp:590-601
// (window_usage() and rank_before() follow scheduler.cpp:274-367 and schd-priority.cpp:19-26 step by step -- the
//  negative-timestamp trick, the overlap split, the evaluation order: bit-exact ledgers leave no freedom there.)
#pragma once
namespace {

const uint32_t LEDGER_CAP = 8192;
enum { ST_IDLE = 0, ST_WAITING = 1, ST_GRANTED = 2 };

// ---- versioned policy state -----------------------------------------------------------------------------------
struct PSlot {
  char name[64];
  double min_frac, max_frac;
  uint64_t mem_limit;
  double quota;   // quota_  (ClientInfo, scheduler.h:26-60)
  double burst;   // burst_
  uint32_t configured;
  uint32_t listed;              // present in the quota file as last loaded
  double last_start, last_end;  // latest token of this client in the FULL history (never pruned)
  // request / grant mailbox
  uint32_t state;
  int32_t poster;  // attachment that posted the request in flight (-1: none / not attached)
  double arrived_ms;
  double granted_quota;
  uint64_t req_seq;  // order of arrival (the candidates list is FIFO)
  uint64_t grants;
  double closed_ms;  // sum(end - start) over this client's finished tokens (full history)
  // pod-level token shared by the processes of one pod (gem-pmgr's role, pod-manager.cpp:97-101)
  double pod_quota;      // pod_quota
  int64_t pod_token_us;  // quota_updated_tp, microseconds since pool start
  double pod_overuse;    // pod_overuse_ms
};
static_assert(sizeof(PSlot) == 200, "policy slot layout");

struct Span {
  int32_t slot;
  int32_t _pad;
  double start, end;
};

struct State {
  int32_t holder;  // slot holding the outstanding token or -1
  uint32_t nslots;
  double deadline_ms;
  uint64_t next_req_seq;
  uint64_t total_grants;
  uint32_t ledger_len;
  uint32_t ledger_dropped;
  uint64_t quota_stamp;  // (mtime, size) stamp of the quota file this configuration was loaded from; 0 = loaded from text
  uint64_t _pad;
  PSlot slots[GEMHOOK_MAX_SLOTS];
  Span ledger[LEDGER_CAP];
};

inline double bits_to_double(uint64_t b) {
  double d;
  memcpy(&d, &b, sizeof(d));
  return d;
}
inline uint64_t double_to_bits(double d) {
  uint64_t b;
  memcpy(&b, &d, sizeof(b));
  return b;
}

struct Stamp {
  int32_t slot;
  double t;  // negative = start
};
struct Ranked {
  double missing, remaining, usage, arrived;
  int slot;
};
// schd-priority.cpp:19-26
bool rank_before(const Ranked& a, const Ranked& b) {
  if (a.missing > 0 && b.missing > 0) return a.missing / (a.missing + a.usage) > b.missing / (b.missing + b.usage);
  if (a.missing > 0 && b.missing < 0) return true;
  if (a.missing < 0 && b.missing > 0) return false;
  return a.usage < b.usage;
}

// ---- the serial policy, on ONE state block (a transaction's private copy) --------------------------------------
struct Policy {
  State& s;
  const Header& h;
  bool dirty = false;
  Policy(State& st, const Header& hd) : s(st), h(hd) {}

  // scheduler.cpp:281-367 -- prune the ledger and compute per-slot usage inside the window
  void window_usage(double now, double* usage, double& wsize, double& wstart) {
    wsize = h.window;
    wstart = now - h.window;
    if (wstart < 0) wsize = now;
    uint32_t k = 0;
    for (uint32_t i = 0; i < s.ledger_len; i++)
      if (!(s.ledger[i].end < wstart)) s.ledger[k++] = s.ledger[i];
    if (k != s.ledger_len) dirty = true;
    s.ledger_len = k;

    std::vector<Stamp> st;
    st.reserve(2 * k);
    for (uint32_t i = 0; i < k; i++) {
      st.push_back({s.ledger[i].slot, -s.ledger[i].start});
      st.push_back({s.ledger[i].slot, s.ledger[i].end});
      usage[s.ledger[i].slot] = 0;
    }
    std::sort(st.begin(), st.end(), [](Stamp a, Stamp b) { return std::abs(a.t) < std::abs(b.t); });
    std::vector<int32_t> live;
    int live_cnt = 0;
    size_t j = 0;
    for (; j < st.size(); j++) {
      if (std::abs(st[j].t) <= wstart) {
        live_cnt++;
        live.push_back(st[j].slot);
      } else {
        break;
      }
    }
    double cur = wstart;
    for (size_t i = j; i < st.size(); i++) {
      for (size_t q = 0; q < live.size(); q++) usage[live[q]] += (std::abs(st[i].t) - cur) / live_cnt;
      if (st[i].t < 0) {
        live.push_back(st[i].slot);
        live_cnt++;
      } else {
        for (size_t q = 0; q < live.size(); q++)
          if (live[q] == st[i].slot) {
            live.erase(live.begin() + q);
            break;
          }
        live_cnt--;
      }
      cur = std::abs(st[i].t);
    }
  }

  // schedule_daemon_func + select_candidate (scheduler.cpp:461-529, 274-399): one decision
  int schedule(double now, int* slot_out, double* quota_out, double* sleep_out) {
    uint32_t n = s.nslots;
    if (s.holder >= 0) {
      // scheduler.cpp:501-521: wait until the holder asks again or its quota times out
      bool back = s.slots[s.holder].state == ST_WAITING;
      if (!back && now < s.deadline_ms) {
        if (sleep_out) *sleep_out = s.deadline_ms - now;
        return -2;
      }
      s.holder = -1;
      dirty = true;
    }
    // candidates in arrival order
    int order[GEMHOOK_MAX_SLOTS];
    int nc = 0;
    for (uint32_t i = 0; i < n; i++)
      if (s.slots[i].state == ST_WAITING) order[nc++] = (int)i;
    if (nc == 0) return -1;
    std::sort(order, order + nc, [&](int a, int b) { return s.slots[a].req_seq < s.slots[b].req_seq; });

    double usage[GEMHOOK_MAX_SLOTS];
    for (uint32_t i = 0; i < n; i++) usage[i] = 0;
    double wsize, wstart;
    window_usage(now, usage, wsize, wstart);

    int pick = -1;
    bool head_seen = false;  // scheduler.cpp:312-320: head of the queue with no recent history goes first
    for (uint32_t i = 0; i < s.ledger_len; i++)
      if (s.ledger[i].slot == order[0]) {
        head_seen = true;
        break;
      }
    if (!head_seen) {
      pick = order[0];
    } else {
      std::vector<Ranked> ok;
      for (int c = 0; c < nc; c++) {
        PSlot& cs = s.slots[order[c]];
        double limit = cs.max_frac * wsize, require = cs.min_frac * wsize;
        double missing = require - usage[order[c]], remaining = limit - usage[order[c]];
        if (remaining > 0) ok.push_back({missing, remaining, usage[order[c]], cs.arrived_ms, order[c]});
      }
      if (ok.empty()) {  // scheduler.cpp:383-390
        if (sleep_out) *sleep_out = s.ledger[0].end - wstart;
        return 0;
      }
      std::sort(ok.begin(), ok.end(), rank_before);
      pick = ok[0].slot;
    }

    // get_quota (scheduler.cpp:160-174) + Record (scheduler.cpp:144-153)
    PSlot& ps = s.slots[pick];
    if (ps.burst < 1e-9) {
      ps.quota = h.base_quota;
    } else {
      ps.quota = ps.burst * 0.5 + ps.quota * (1 - 0.5);
      ps.quota = std::max(ps.quota, h.min_quota);
      ps.quota = std::min(ps.quota, ps.max_frac * h.window);
    }
    if (s.ledger_len == LEDGER_CAP) {  // cannot happen with sane quotas; keep the newest entries
      memmove(&s.ledger[0], &s.ledger[1], sizeof(Span) * (LEDGER_CAP - 1));
      s.ledger_len--;
      s.ledger_dropped++;
    }
    s.ledger[s.ledger_len++] = Span{pick, 0, now, now + ps.quota};
    if (ps.grants) ps.closed_ms += ps.last_end - ps.last_start;
    ps.last_start = now;
    ps.last_end = now + ps.quota;
    ps.grants++;
    s.total_grants++;
    s.holder = pick;
    s.deadline_ms = now + ps.quota;
    ps.granted_quota = ps.quota;
    ps.state = ST_GRANTED;
    dirty = true;
    if (slot_out) *slot_out = pick;
    if (quota_out) *quota_out = ps.quota;
    return 1;
  }

  // handle_message(REQ_QUOTA) (scheduler.cpp:417-429): update_return_time + set_burst + enqueue
  void request(int slot, double now, double overuse, double burst, int poster) {
    PSlot& ps = s.slots[slot];
    for (uint32_t i = s.ledger_len; i-- > 0;) {
      if (s.ledger[i].slot == slot) {
        s.ledger[i].end = std::min(now, s.ledger[i].end + overuse);
        break;
      }
    }
    if (ps.grants) ps.last_end = std::min(now, ps.last_end + overuse);
    ps.burst = burst;
    ps.arrived_ms = now;
    ps.req_seq = ++s.next_req_seq;
    ps.state = ST_WAITING;
    ps.poster = poster;
    dirty = true;
  }

  // A client that is going away hands its token back: the ledger entry is closed exactly as a returning client's
  // would be (update_return_time with zero overuse).  Returns true if the token was this slot's.
  bool give_back(int slot, double now) {
    bool held = s.holder == slot;
    if (held) {
      for (uint32_t i = s.ledger_len; i-- > 0;)
        if (s.ledger[i].slot == slot) {
          s.ledger[i].end = std::min(now, s.ledger[i].end);
          break;
        }
      PSlot& ps = s.slots[slot];
      if (ps.grants) ps.last_end = std::min(now, ps.last_end);
      ps.pod_quota = 0.0;  // the pod-level token is gone with it: the next request must be forwarded
      s.holder = -1;
      dirty = true;
    }
    if (s.slots[slot].state == ST_WAITING) {
      s.slots[slot].state = ST_IDLE;
      s.slots[slot].poster = -1;
      dirty = true;
    }
    return held;
  }
};

// ---- pod-level token (gem-pmgr hook_kernel_launch, pod-manager.cpp:316-473) -----------------------------------
// Processes of one pod share the pod's token: a request is answered locally with the REMAINING pod quota unless
// `elapsed + burst > pod_quota`, in which case it is forwarded to the scheduler with the pod's maximum overuse and
// the maximum burst over its processes.  Returns 1 = forward (fwd_* filled), 0 = answered (*remain_ms).
static int pod_launch(Attach* attach, Policy& pol, int slot, int attach_idx, int64_t now_us, double overuse, double burst,
                      double* fwd_overuse, double* fwd_burst, double* remain) {
  PSlot& s = pol.s.slots[slot];
  double mo = std::max(overuse, s.pod_overuse);
  if (mo != s.pod_overuse) {
    s.pod_overuse = mo;
    pol.dirty = true;
  }
  if (attach_idx >= 0) attach[attach_idx].burst_bits.store(double_to_bits(burst), std::memory_order_relaxed);
  double elapsed = (double)(now_us - s.pod_token_us) / 1e3;
  if (elapsed + burst > s.pod_quota) {
    double mx = attach_idx >= 0 ? 0.0 : burst;
    for (uint32_t i = 0; i < MAX_ATTACH; i++)
      if (attach[i].in_use.load(std::memory_order_relaxed) && attach[i].slot.load(std::memory_order_relaxed) == slot)
        mx = std::max(bits_to_double(attach[i].burst_bits.load(std::memory_order_relaxed)), mx);
    if (fwd_overuse) *fwd_overuse = s.pod_overuse;
    if (fwd_burst) *fwd_burst = mx;
    return 1;
  }
  if (remain) *remain = s.pod_quota - elapsed;
  return 0;
}
static double pod_granted(Policy& pol, int slot, int64_t now_us, double quota) {
  PSlot& s = pol.s.slots[slot];
  s.pod_quota = quota;
  s.pod_token_us = now_us;
  s.pod_overuse = 0.0;
  pol.dirty = true;
  return s.pod_quota - 0.0;
}

}  // namespace
