"""Two- and three-layer oracles: C1/C2 mixed-precision tiers and C3 approximate embeddings.

TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py.

The reference implements the multi-layer path only in C++ (mixed_precs_caching/):

  request_to_c1_c2      evlfu_32.cpp:319-461, evlfu_16.cpp:443-580, evlfu_8.cpp:669-796 (identical logic)
  request_to_c1_c2_c3   evlfu_8.cpp:492-667 (MAIN 8 / SECONDARY 4 only, cache_manager.cpp:212-220)
  phase_1 / phase_2     evlfu_8.cpp:416-457, evlfu_4.cpp:374-415, evlfu_16.cpp:400-441
  setKey / update_agg_hit   evlfu_32.cpp:206-272 (and the 16/8/4 twins)
  APRX_EV (C3)          aprx_embedding.cpp:304-329 (insert group), :360-388 (second-chance eviction),
                        :344-353 (get_altkey_str), :402-411 (set_recency_flag_c3)

Two restatements live here:

* ``SeqTiers`` -- one request at a time, statement for statement.  With ``order="stdset"`` and
  ``flush="cpp"`` it reproduces the compiled reference exactly, including its victim order (the
  buckets are libstdc++ ``unordered_set<string>``; the same container is driven through
  oracle/stdset_shim.cpp) and its flush arithmetic (``int(0.3*cap)`` keys, ``n_perfect -=``).
  tests/test_oracle_tiers.py pins it request-by-request against oracle/_ref/lib*.so.
  With ``order="fifo"`` and ``flush="py"`` every tier follows the canonical Python policy
  (cache_algo/EvLFU_C1.py: FIFO buckets, ``int(0.3*cap)+1`` flushed, ``n_perfect = len``) that the
  CUDA path implements; the routing between the tiers is the same code.
* ``BatchTiers`` -- the batch-granular generalisation the CUDA path implements (DESIGN.md): all
  keys of a batch are probed against the state at batch start, each tier applies its winners in
  position order, then flushes / evicts down to capacity, then the victims (C2's, then C1's)
  enter C3 as one group.

C3: the reference feeds it from worker threads in groups of IO_JOB_Q_SIZE=50 queued victims and
aborts on fast traces ("Too many items in the queue", aprx_embedding.cpp:146-148).  Driven with a
pause after every request it is deterministic, and ``SeqTiers(order="stdset", flush="cpp",
c3_group=50)`` reproduces it request by request (tests/test_oracle_c3_pin.py: returned rows incl.
the alternative keys' rows, perfect-hit counter).  The policy the CUDA path implements differs in
ONE documented way: the victims of a request / batch enter C3 as one group when it ends
(``c3_group=None``) instead of waiting in a 50-key job queue; lookup, routing, second-chance
eviction and the recency flag are the same code in both modes.
"""
from __future__ import annotations

import ctypes as C
import os
from collections import OrderedDict, deque

import numpy as np

from .evlfu import KEY_SHIFT, make_key, split_key

HIT_MISS, HIT_C1, HIT_C2, HIT_C3, HIT_APPROX = 0, 1, 2, 3, 4
ABSENT = 255        # no key at this position (a slice of ragged bags)
HERE = os.path.dirname(os.path.abspath(__file__))


def capacities(n_layers: int, main: int, sec: int, total: int, prop: str = "", dim: int = 36):
    """Entry capacities (c1, c2, c3) as the reference's constructors compute them, quirks included
    (cache_manager.cpp:22-52; evlfu_32.cpp:99-105; evlfu_16.cpp:93-98; evlfu_8.cpp:57-95).  The
    literal 36 of evlfu_8.cpp:79,88 is EV_DIMENSION (alt keys per fp32 row); ``dim`` here."""
    if n_layers == 1:
        return total * (32 // main), 0, 0
    if n_layers == 2:
        cs = total // 2
        if main == 32:
            return cs, {16: cs * 2, 8: cs * 4 * 4, 4: cs * 8}[sec], 0
        if main == 16:
            c1 = cs * 2
            return c1, {8: c1 * 2 * 4, 4: c1 * 4}[sec], 0
        if main == 8 and sec == 4:
            return cs * 4, cs * 8, 0
        raise ValueError("unsupported precision pair")
    if n_layers == 3:
        if (main, sec) != (8, 4):
            raise ValueError("three layers exist only for 8/4 (cache_manager.cpp:212-220)")
        if prop:
            a, b, c = (int(x) for x in prop.split("-"))
            assert a + b + c == 100
            return (a * total // 100) * 4, (b * total // 100) * 8, (c * total // 100) * dim
        return total // 3 * 4, total // 3 * 8, total // 3 * dim
    raise ValueError(n_layers)


def key_str(key: int) -> bytes:
    t, r = split_key(key)
    return f"{t + 1}-{r}".encode()          # evlfu_32.cpp:332


# ---- bucket containers ------------------------------------------------------------------------
class FifoBucket:
    """Python list semantics of EvLFU_C1.py (append / remove / pop(0))."""

    def __init__(self):
        self.d = OrderedDict()

    def __len__(self):
        return len(self.d)

    def insert(self, key):
        self.d[key] = None

    def erase(self, key):
        return self.d.pop(key, 0) is None

    def __contains__(self, key):
        return key in self.d

    def pop_begin(self):
        return self.d.popitem(last=False)[0]

    def keys(self):
        return list(self.d.keys())


_shim = None


def _load_shim():
    global _shim
    if _shim is None:
        p = os.path.join(HERE, "_ref", "libstdset_shim.so")
        if not os.path.exists(p):
            raise RuntimeError(f"{p} missing: run build() (python __graft_entry__.py), which compiles it")
        lib = C.CDLL(p)
        lib.uset_new.restype = C.c_void_p
        lib.uset_free.argtypes = [C.c_void_p]
        lib.uset_size.argtypes = [C.c_void_p]
        lib.uset_size.restype = C.c_long
        lib.uset_insert.argtypes = [C.c_void_p, C.c_char_p]
        lib.uset_erase.argtypes = [C.c_void_p, C.c_char_p]
        lib.uset_erase.restype = C.c_int
        lib.uset_contains.argtypes = [C.c_void_p, C.c_char_p]
        lib.uset_contains.restype = C.c_int
        lib.uset_pop_begin.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        lib.uset_pop_begin.restype = C.c_int
        _shim = lib
    return _shim


def shim_available() -> bool:
    return os.path.exists(os.path.join(HERE, "_ref", "libstdset_shim.so"))


class StdSetBucket:
    """libstdc++ unordered_set<string> (evlfu_32.hpp:49) through oracle/stdset_shim.cpp."""

    def __init__(self):
        self.lib = _load_shim()
        self.h = C.c_void_p(self.lib.uset_new())
        self.buf = C.create_string_buffer(64)

    def __del__(self):
        try:
            self.lib.uset_free(self.h)
        except Exception:
            pass

    def __len__(self):
        return int(self.lib.uset_size(self.h))

    def insert(self, key):
        self.lib.uset_insert(self.h, key_str(key))

    def erase(self, key):
        return bool(self.lib.uset_erase(self.h, key_str(key)))

    def __contains__(self, key):
        return bool(self.lib.uset_contains(self.h, key_str(key)))

    def pop_begin(self):
        if not self.lib.uset_pop_begin(self.h, self.buf, 64):
            raise KeyError("empty bucket")
        t, r = self.buf.value.decode().split("-")
        return make_key(int(t) - 1, int(r))


# ---- sequential restatement -------------------------------------------------------------------
class SeqTier:
    """One EVLFU_* object: vals (key -> agg_hit), lists[0..T], min pointer, n_perfect."""

    def __init__(self, cap: int, T: int = 26, order: str = "fifo", flush: str = "py",
                 flush_rate: float = 0.3, perfect_item_cap: float = 0.95):
        self.cap, self.T = int(cap), int(T)
        self.vals: dict[int, int] = {}
        mk = FifoBucket if order == "fifo" else StdSetBucket
        self.lists = [mk() for _ in range(T + 1)]
        self.min = 0
        self.n_perfect = 0
        self.max_perfect = int(self.cap * perfect_item_cap)
        self.flush_cpp = flush == "cpp"
        self.flush_n = int(flush_rate * self.cap) + (0 if self.flush_cpp else 1)
        self.evicted: list[int] = []      # normal evictions (these feed C3)
        self.flushed: list[int] = []

    def set_key(self, key: int, agg: int):
        """evlfu_32.cpp:206-251 / EvLFU_C1.py:32-63."""
        if self.n_perfect >= self.max_perfect:
            top = self.lists[self.T]
            for _ in range(min(self.flush_n, len(top))):
                k = top.pop_begin()
                del self.vals[k]
                self.flushed.append(k)
            if self.flush_cpp:
                self.n_perfect -= self.flush_n            # evlfu_32.cpp:218
            else:
                self.n_perfect = len(top)                 # EvLFU_C1.py:44
        elif len(self.vals) >= self.cap:
            while len(self.lists[self.min]) == 0:
                self.min += 1
                if self.min > self.T:
                    self.min = 1
            k = self.lists[self.min].pop_begin()
            del self.vals[k]
            self.evicted.append(k)
        self.vals[key] = agg
        self.lists[agg].insert(key)
        if agg < self.min:
            self.min = agg

    def update_agg_hit(self, key: int, agg: int) -> bool:
        """evlfu_32.cpp:254-272.  False = the entry is gone (evicted earlier in this request): the
        C++ then works on a dangling Cache_data* (undefined behaviour) and does not re-insert."""
        old = self.vals.get(key)
        if old is None:
            return False
        if old < agg:
            self.lists[old].erase(key)
            self.lists[agg].insert(key)
            self.vals[key] = agg
        return True

    def state(self):
        return [b.keys() for b in self.lists]


class C3State:
    """APRX_EV: vals_C3 key -> [alt_key, recency_flag], lists_C3 FIFO queue (may hold stale or
    duplicate keys), second-chance eviction (aprx_embedding.cpp:360-388)."""

    def __init__(self, cap: int, alt_keys, table_base: int = 0):
        self.cap = int(cap)
        self.alt = alt_keys                  # per table uint32 array: alt_row*100 + alt_table(1-based)
        self.table_base = table_base
        self.vals: dict[int, list] = {}
        self.fifo: deque[int] = deque()
        self.hits = 0
        self.evicted = 0

    def find(self, key: int):
        """get_altkey_str: the alternative key as an integer key, or None."""
        e = self.vals.get(key)
        if e is None:
            return None
        a = int(e[0])
        return make_key(a % 100 - 1, a // 100)

    def set_recency(self, key: int):
        e = self.vals.get(key)
        if e is not None:
            e[1] = True

    def _evict_one(self):
        while True:
            k = self.fifo.popleft()
            e = self.vals.get(k)
            if e is None:
                continue                      # stale / redundant queue record
            if e[1]:
                e[1] = False
                self.fifo.append(k)
            else:
                del self.vals[k]
                self.evicted += 1
                return

    def insert_group(self, keys):
        """insert_altkey_batched_obj (aprx_embedding.cpp:304-329) for a group of any size."""
        n = len(keys)
        if n == 0:
            return
        n_erase = min(max(0, len(self.vals) + n - self.cap), len(self.vals))
        for _ in range(n_erase):
            self._evict_one()
        for k in keys:
            t, r = split_key(k)
            self.fifo.append(k)
            self.vals[k] = [int(self.alt[t - self.table_base][r]), False]

    def dump(self):
        """Queue records whose key is still mapped, in FIFO order: (keys, alt, recency)."""
        ks = [k for k in self.fifo if k in self.vals]
        return ks, [self.vals[k][0] for k in ks], [int(self.vals[k][1]) for k in ks]


class SeqTiers:
    """request_to_c1_c2 / request_to_c1_c2_c3, one request of T row ids at a time."""

    def __init__(self, caps, n_layers: int = 2, T: int = 26, order: str = "fifo", flush: str = "py",
                 high_thres: int = 23, alt_keys=None, c3_group: int | None = None):
        """c3_group=None: the victims of a request enter C3 as one group when the request ends (the
        synchronous policy the CUDA path follows).  c3_group=n: the reference's own queueing -- victims
        are appended to a job queue key by key and every n-th key (IO_JOB_Q_SIZE = 50,
        aprx_embedding.hpp:29) releases the oldest n of them into C3 as one group
        (check_curr_batch_size / insert_altkey_batched_obj, aprx_embedding.cpp:125-150,304-329); this
        is what the compiled reference does when its worker threads finish before the next request."""
        self.T, self.n_layers, self.high_thres = T, n_layers, high_thres
        self.c1 = SeqTier(caps[0], T, order, flush)
        self.c2 = SeqTier(caps[1], T, order, flush)
        self.c3 = C3State(caps[2], alt_keys) if n_layers == 3 and caps[2] > 0 else None
        self.c3_group = c3_group
        self.c3_pending: list[int] = []

    def _feed_c3(self, victims):
        if self.c3_group is None:
            self.c3.insert_group(victims)
            return
        for k in victims:
            self.c3_pending.append(k)
            if len(self.c3_pending) == self.c3_group:
                self.c3.insert_group(self.c3_pending)
                self.c3_pending = []

    def request(self, row_ids):
        """Returns (code[T], val_tier[T], src_key[T], stale[T], perfect):
        code      HIT_C1 / HIT_C2 / HIT_C3 / HIT_MISS (who answered)
        val_tier  0 / 1: precision of the returned row (C1's or C2's)
        src_key   key whose row is returned (the alternative key on a C3 hit)
        stale     the C++ reads a dangling pointer here; the returned floats are undefined."""
        T, c1, c2, c3 = self.T, self.c1, self.c2, self.c3
        c1.evicted, c1.flushed, c2.evicted, c2.flushed = [], [], [], []
        keys = [make_key(i, r) for i, r in enumerate(row_ids)]
        if self.n_layers == 1:                                     # request_to_ev_lfu (evlfu_32.cpp:473-549)
            hit = [k in c1.vals for k in keys]
            agg = sum(hit)
            stale = [False] * T
            for i, k in enumerate(keys):
                if hit[i]:
                    stale[i] = not c1.update_agg_hit(k, agg)
                else:
                    c1.set_key(k, agg)
            if agg == T:
                c1.n_perfect = len(c1.lists[T])
            return [HIT_C1 if h else HIT_MISS for h in hit], [0] * T, list(keys), stale, int(agg == T)
        c2hit = [k in c2.vals for k in keys]                       # phase_1 on C2
        agg = sum(c2hit)
        c1hit = [False] * T
        c1_agg = 0
        c2_update = [True] * T
        c2_insert = [False] * T
        code = [HIT_MISS] * T
        val_tier = [0] * T
        src = list(keys)
        stale = [False] * T
        c3src = {}
        for i, k in enumerate(keys):
            if k in c1.vals:
                c1hit[i] = True
                c1_agg += 1
                c2_update[i] = False
                if not c2hit[i]:
                    agg += 1
            elif not c2hit[i]:
                akey = c3.find(k) if c3 is not None else None
                a_tier = None
                if akey is not None:                               # find_approximate_ev (evlfu_8.cpp:474-489)
                    a_tier = 0 if akey in c1.vals else (1 if akey in c2.vals else None)
                if a_tier is not None:
                    c3.set_recency(k)
                    c3.hits += 1
                    agg += 1
                    c3src[i] = (a_tier, akey)
                    c2_update[i] = False
                else:
                    c2_insert[i] = True
                    c2_update[i] = False
        jobs = set()
        should_update_c2 = True
        if len(c1.vals) >= c1.cap:
            if agg < self.high_thres:
                for i in range(T):
                    if not c2hit[i]:
                        c2_update[i] = False
                        if i % 2 == 1:
                            jobs.add(i)                            # (also for C1 hits: read, then discarded)
                            c2_insert[i] = False
        else:
            for i in range(T):
                if not c1hit[i] and i not in c3src:
                    jobs.add(i)
            should_update_c2 = False
            agg = c1_agg
        if should_update_c2:                                       # phase_2 on C2
            for i, k in enumerate(keys):
                if c2_update[i]:
                    c2.update_agg_hit(k, agg)
                    code[i], val_tier[i] = HIT_C2, 1
            for i, k in enumerate(keys):
                if c2_insert[i]:
                    c2.set_key(k, agg)
                    code[i], val_tier[i] = HIT_MISS, 1
            if agg == T:
                c2.n_perfect = len(c2.lists[T])
        for i, k in enumerate(keys):
            if c1hit[i]:
                if not c1.update_agg_hit(k, agg):
                    stale[i] = True
                code[i], val_tier[i] = HIT_C1, 0
            elif i in c3src:
                code[i] = HIT_C3
                val_tier[i], src[i] = c3src[i]
            elif i in jobs:
                c1.set_key(k, agg)
                code[i], val_tier[i] = HIT_MISS, 0
        if c3 is not None:
            self._feed_c3(c2.evicted + c1.evicted)                 # evlfu_8.cpp:617-620, 654-658
        perfect = 0
        if agg == T:
            c1.n_perfect = len(c1.lists[T])
            perfect = 1
        return code, val_tier, src, stale, perfect


# ---- batch-granular policy ----------------------------------------------------------------------
class TierState:
    """One tier under the batch-granular EvLFU policy (steps 3-6 of oracle.evlfu.BatchEvLFU)."""

    def __init__(self, cap: int, T: int = 26, flush_rate: float = 0.3, perfect_item_cap: float = 0.95):
        self.cap, self.T = int(cap), int(T)
        self.entries: dict[int, int] = {}
        self.lists = [OrderedDict() for _ in range(T + 1)]
        self.n_perfect = 0
        self.max_perfect = int(self.cap * perfect_item_cap)
        self.flush_n = int(flush_rate * self.cap) + 1
        self.inserted: list[int] = []
        self.flushed: list[int] = []
        self.evicted: list[int] = []

    def apply(self, winners: dict, any_perfect: bool, promotions_first: bool = False):
        """winners: key -> (agg, position) of the winning flagged occurrence.  They are applied in
        position order; with ``promotions_first`` (C2: phase_2 updates every hit before it inserts
        any miss, evlfu_8.cpp:416-442) all promotions come before all inserts."""
        ent, T = self.entries, self.T
        self.inserted, self.flushed, self.evicted = [], [], []
        prot, prot_rank = None, None
        order = sorted(winners.items(), key=lambda kv: kv[1][1])
        if promotions_first:
            order = [kv for kv in order if kv[0] in ent] + [kv for kv in order if kv[0] not in ent]
        for k, (a, p) in order:
            old = ent.get(k)
            if old is not None:
                del self.lists[old][k]
            else:
                self.inserted.append(k)
                if prot_rank is None or (a, p) > prot_rank:
                    prot, prot_rank = k, (a, p)
            self.lists[a][k] = None
            ent[k] = a
        if self.inserted and self.n_perfect >= self.max_perfect:
            lt = self.lists[T]
            for _ in range(min(self.flush_n, len(lt))):
                k, _v = lt.popitem(last=False)
                del ent[k]
                self.flushed.append(k)
            self.n_perfect = len(lt)
        need = len(ent) - self.cap
        b = 0
        while need > 0 and b <= T:
            lst = self.lists[b]
            victims = []
            for k in lst:
                if k == prot:
                    continue
                victims.append(k)
                if len(victims) == need:
                    break
            for k in victims:
                del lst[k]
                del ent[k]
            self.evicted.extend(victims)
            need -= len(victims)
            b += 1
        if any_perfect:
            self.n_perfect = len(self.lists[T])

    def state(self):
        return [list(l.keys()) for l in self.lists]


class BatchTiers:
    """The CUDA path's policy for 1, 2 or 3 layers.  Positions are sample-major, table-minor."""

    def __init__(self, caps, n_layers: int = 2, T: int = 26, high_thres: int = 23, alt_keys=None,
                 table_base: int = 0, n_local: int | None = None):
        self.T, self.n_layers, self.high_thres = T, n_layers, high_thres
        self.table_base = table_base
        self.c1 = TierState(caps[0], T)
        self.c2 = TierState(caps[1], T) if n_layers >= 2 else None
        self.c3 = C3State(caps[2], alt_keys, table_base) if n_layers == 3 and caps[2] > 0 else None

    def lookup_batch(self, idx, agg=None):
        """idx int [Tl, B].  Returns (code [B,Tl] uint8, val_tier [B,Tl], src_t [B,Tl], src_r [B,Tl], agg [B])."""
        idx = np.asarray(idx)
        Tl, B = idx.shape
        c1, c2, c3 = self.c1, self.c2, self.c3
        two = c2 is not None
        full = two and len(c1.entries) >= c1.cap
        code = np.zeros((B, Tl), dtype=np.uint8)
        val_tier = np.zeros((B, Tl), dtype=np.int8)
        src_t = np.tile(np.arange(Tl, dtype=np.int32) + self.table_base, (B, 1))
        src_r = np.ascontiguousarray(idx.T).astype(np.int64)
        agg_out = np.zeros(B, dtype=np.int64)
        w = [dict(), dict()]
        any_perfect = [False, False]

        def bid(tier, k, a, p):
            cur = w[tier].get(k)
            if cur is None or (a, p) > cur:
                w[tier][k] = (a, p)

        for s in range(B):
            # a negative index = no key at this position (slices of ragged bags, oracle.evlfu.expand_bags): code ABSENT
            keys = [make_key(self.table_base + t, idx[t, s]) if idx[t, s] >= 0 else None for t in range(Tl)]
            h0 = [k is not None and k in c1.entries for k in keys]
            h1 = [two and k is not None and (k in c2.entries) for k in keys]
            c3src = {}
            if c3 is not None:
                for t, k in enumerate(keys):
                    if k is not None and not h0[t] and not h1[t]:
                        akey = c3.find(k)
                        if akey is None:
                            continue
                        a_tier = 0 if akey in c1.entries else (1 if akey in c2.entries else None)
                        if a_tier is not None:
                            c3.set_recency(k)
                            c3.hits += 1
                            c3src[t] = (a_tier, akey)
            if not two:
                a = sum(h0)
            elif full:
                a = sum(1 for x, y in zip(h0, h1) if x or y) + len(c3src)
            else:
                a = sum(h0)
            if agg is not None:
                a = int(agg[s])
            agg_out[s] = a
            for t, k in enumerate(keys):
                p = s * Tl + t
                if k is None:
                    code[s, t] = ABSENT
                    src_t[s, t] = -1
                    continue
                if h0[t]:
                    code[s, t] = HIT_C1
                    if c1.entries[k] < a:
                        bid(0, k, a, p)
                elif t in c3src:
                    code[s, t] = HIT_C3
                    val_tier[s, t] = c3src[t][0]
                    at, ar = split_key(c3src[t][1])
                    src_t[s, t], src_r[s, t] = at, ar
                elif full and h1[t]:
                    code[s, t] = HIT_C2
                    val_tier[s, t] = 1
                    if c2.entries[k] < a:
                        bid(1, k, a, p)
                else:
                    tier = 0
                    if full:
                        tier = 0 if (a < self.high_thres and ((self.table_base + t) & 1)) else 1
                    val_tier[s, t] = tier
                    bid(tier, k, a, p)
            if a == self.T:
                any_perfect[0] = True
                if full:
                    any_perfect[1] = True
        if two:
            c2.apply(w[1], any_perfect[1], promotions_first=True)
        c1.apply(w[0], any_perfect[0])
        if c3 is not None:
            c3.insert_group((c2.evicted if two else []) + c1.evicted)
        return code, val_tier, src_t, src_r, agg_out


def gather_tier_rows(dec_tables, val_tier, src_t, src_r, table_base: int = 0):
    """dec_tables: [tier][table] -> decoded fp32 [rows, d].  fp32 rows for every position."""
    B, Tl = src_t.shape
    d = dec_tables[0][0].shape[1]
    out = np.zeros((B, Tl, d), dtype=np.float32)
    for tier in range(len(dec_tables)):
        for t in np.unique(src_t):
            if t < 0:
                continue
            m = (src_t == t) & (val_tier == tier)
            if m.any():
                out[m] = dec_tables[tier][int(t) - table_base][src_r[m]]
    return out
