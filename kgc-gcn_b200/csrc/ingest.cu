// N4: native text -> id ingest (host C++, no device code; SURVEY.md 8(f) row N4).
// Replaces the two per-line Python passes of DataLoader._load_data (reference data_loader.py:64-111): vocabulary in
// first-appearance order over train / valid / test, the triple arrays, and the (s, r) -> objects grouping in both
// directions - as CSR arrays the GPU batch builder (K5) and the fused scorer (K6) consume directly, instead of Python
// lists of dicts.  The reference's quirks are kept: tokens are lower-cased when the vocabulary is built
// (data_loader.py:69-71) but NOT when the triples are looked up (data_loader.py:83-85), so a mixed-case data set fails
// with the offending token (the reference raises KeyError); lines are split on ASCII whitespace and must hold three tokens.
// Tokens with non-ASCII bytes (str.lower() is Unicode-aware) and relation tokens that end in "_reverse" (they alias the
// reverse ids the reference adds) are reported as unsupported: the caller then runs the Python passes.  Query order is Python's dict insertion order: a key (s, r) or (o, r + R) is created by the first line that
// mentions it, "tail" key before "head" key within a line.
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "common.cuh"

namespace {

// open-addressing hash tables (linear probing, power-of-two capacity, load <= 0.5).  A look-up is ONE cache line: key / hash,
// id and (for tokens of <= 16 bytes, i.e. every id of WN18RR / FB15k-237 / Wikidata) the lower-cased token itself sit in the
// slot.  The tables of a real data set are far bigger than the caches, so both passes work on blocks of lines: hash the
// block, prefetch its slots, then resolve in order (std::unordered_map's node allocations dominated the first version, the
// cache misses of dependent probes the second).
struct KeyTable {                // uint64 key -> dense id in insertion order
  struct Slot { uint64_t key; int32_t id; int32_t pad; };     // id -1 = empty
  std::vector<Slot> slots;
  size_t n = 0;
  KeyTable() : slots(1 << 16, Slot{0, -1, 0}) {}
  static inline uint64_t mix(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return x;
  }
  void grow() {
    std::vector<Slot> old(slots.size() * 2, Slot{0, -1, 0});
    old.swap(slots);
    const size_t mask = slots.size() - 1;
    for (const Slot& o : old)
      if (o.id >= 0) {
        size_t p = mix(o.key) & mask;
        while (slots[p].id >= 0) p = (p + 1) & mask;
        slots[p] = o;
      }
  }
  inline void prefetch(uint64_t key) const { __builtin_prefetch(&slots[mix(key) & (slots.size() - 1)]); }
  int32_t find(uint64_t key) const {
    const size_t mask = slots.size() - 1;
    size_t p = mix(key) & mask;
    while (slots[p].id >= 0) {
      if (slots[p].key == key) return slots[p].id;
      p = (p + 1) & mask;
    }
    return -1;
  }
  int32_t find_or_insert(uint64_t key) {           // new keys get id n, n + 1, ...
    if (2 * (n + 1) > slots.size()) grow();
    const size_t mask = slots.size() - 1;
    size_t p = mix(key) & mask;
    while (slots[p].id >= 0) {
      if (slots[p].key == key) return slots[p].id;
      p = (p + 1) & mask;
    }
    slots[p].key = key; slots[p].id = (int32_t)n;
    return (int32_t)n++;
  }
};

struct Token {                   // one whitespace-separated token of a line, hashed over its lower-cased bytes
  const char* p;
  uint32_t len;
  bool upper;                    // holds an ASCII upper-case letter: the reference's case-sensitive look-up will not find it
  uint64_t hash;
  char low[16];                  // lower-cased bytes, zero padded (len <= 16)
};

struct TokenTable {              // lower-cased token bytes -> dense id in insertion order; the tokens live in `names`
  struct Slot { uint64_t hash; int32_t id; uint32_t len; char low[16]; };       // 32 bytes; id -1 = empty
  std::vector<Slot> slots;
  std::vector<std::string>* names;
  explicit TokenTable(std::vector<std::string>* nm) : slots(1 << 16, Slot{0, -1, 0, {0}}), names(nm) {}
  static inline void scan(const char* p, size_t n, Token* t) {
    uint64_t h = 1469598103934665603ull;             // FNV-1a over the lower-cased bytes
    bool up = false;
    memset(t->low, 0, sizeof(t->low));
    for (size_t i = 0; i < n; ++i) {
      unsigned char c = (unsigned char)p[i];
      if (c >= 'A' && c <= 'Z') { c = (unsigned char)(c - 'A' + 'a'); up = true; }
      if (i < sizeof(t->low)) t->low[i] = (char)c;
      h = (h ^ c) * 1099511628211ull;
    }
    t->p = p; t->len = (uint32_t)n; t->upper = up; t->hash = KeyTable::mix(h);
  }
  inline bool same(const Slot& s, const Token& t) const {
    if (s.hash != t.hash || s.len != t.len) return false;
    if (t.len <= sizeof(t.low)) return memcmp(s.low, t.low, sizeof(t.low)) == 0;
    const std::string& a = (*names)[s.id];             // long token: compare the stored lower-cased name
    for (size_t i = 0; i < t.len; ++i) {
      unsigned char c = (unsigned char)t.p[i];
      if (c >= 'A' && c <= 'Z') c = (unsigned char)(c - 'A' + 'a');
      if ((unsigned char)a[i] != c) return false;
    }
    return true;
  }
  void grow() {
    std::vector<Slot> old(slots.size() * 2, Slot{0, -1, 0, {0}});
    old.swap(slots);
    const size_t mask = slots.size() - 1;
    for (const Slot& o : old)
      if (o.id >= 0) {
        size_t q = o.hash & mask;
        while (slots[q].id >= 0) q = (q + 1) & mask;
        slots[q] = o;
      }
  }
  inline void prefetch(const Token& t) const { __builtin_prefetch(&slots[t.hash & (slots.size() - 1)]); }
  int32_t intern(const Token& t) {                   // id of the lower-cased token; new tokens get the next id
    if (2 * (names->size() + 1) > slots.size()) grow();
    const size_t mask = slots.size() - 1;
    size_t q = t.hash & mask;
    while (slots[q].id >= 0) {
      if (same(slots[q], t)) return slots[q].id;
      q = (q + 1) & mask;
    }
    Slot& s = slots[q];
    s.hash = t.hash; s.id = (int32_t)names->size(); s.len = t.len;
    memcpy(s.low, t.low, sizeof(s.low));
    names->emplace_back(t.p, t.len);
    if (t.upper)
      for (auto& c : names->back())
        if (c >= 'A' && c <= 'Z') c = (char)(c - 'A' + 'a');
    return s.id;
  }
};

struct Split {
  std::vector<int64_t> triples;  // [n][3]
};

struct Csr {
  std::vector<int64_t> triples;  // [q][3]
  // train set: ptr [q + 1] / idx = sorted, unique objects of every query.  valid / test sets: the object lists are kept ONCE
  // per (s, r) group - ptr [g + 1] / idx over the groups the set references, qg [q] = group of every query - because a hub
  // group is the filter of thousands of queries (a per-query copy was 12 GB for a 3 M-line Zipf data set)
  std::vector<int64_t> ptr;
  std::vector<int32_t> idx;
  std::vector<int32_t> qg;
};

}  // namespace

struct kgc_ingest {
  std::vector<std::string> ent_names, rel_names;     // lower-cased tokens, id order
  Split split[3];
  Csr csr[5];                                         // train, valid_tail, valid_head, test_tail, test_head
  std::string error;
};

namespace {

bool read_file(const std::string& path, std::string* out) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  fseek(f, 0, SEEK_END);
  const long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  out->resize(n > 0 ? (size_t)n : 0);
  const size_t got = n > 0 ? fread(&(*out)[0], 1, (size_t)n, f) : 0;
  fclose(f);
  return got == out->size();
}

// Python's str.split() / str.strip() with no argument split on these for ASCII text
inline bool is_space(unsigned char c) { return c == ' ' || (c >= 9 && c <= 13) || (c >= 28 && c <= 31); }

// calls fn(tok0, tok1, tok2) for every non-blank line; returns 0, or 1 (wrong token count) / 2 (non-ASCII byte)
template <typename Fn>
int for_each_line(const std::string& text, std::string* err, Fn fn) {
  size_t pos = 0, line_no = 0;
  const size_t n = text.size();
  while (pos < n) {
    size_t end = pos;
    while (end < n && text[end] != '\n' && text[end] != '\r') ++end;       // universal newlines: \n, \r, \r\n
    ++line_no;
    const char* tok[4];
    size_t len[4];
    int nt = 0;
    size_t i = pos;
    while (i < end) {
      while (i < end && is_space((unsigned char)text[i])) ++i;
      if (i >= end) break;
      const size_t b = i;
      while (i < end && !is_space((unsigned char)text[i])) {
        if ((unsigned char)text[i] >= 0x80) {
          *err = "non-ASCII token at line " + std::to_string(line_no);
          return 2;
        }
        ++i;
      }
      if (nt < 4) { tok[nt] = text.data() + b; len[nt] = i - b; }
      ++nt;
    }
    if (nt != 0) {
      if (nt != 3) {
        *err = "line " + std::to_string(line_no) + " holds " + std::to_string(nt) + " tokens, expected 3";
        return 1;
      }
      const int rc = fn(tok, len);
      if (rc) return rc;
    }
    pos = end + 1;
  }
  return 0;
}

int ingest(const std::string& dir, kgc_ingest* h) {
  static const char* kNames[3] = {"train.txt", "valid.txt", "test.txt"};
  std::string text[3];
  for (int s = 0; s < 3; ++s)
    if (!read_file(dir + "/" + kNames[s], &text[s])) {
      h->error = "cannot read " + dir + "/" + kNames[s];
      return 3;
    }
  // ---- pass 1: ids in first-appearance order over the lower-cased tokens, and with them the triples.  The reference looks
  // the tokens up a second time AS WRITTEN (data_loader.py:83-85) in the lower-cased vocabulary: a token without an ASCII
  // upper-case letter is its own lower-cased form (found, same id), any other token cannot be in the vocabulary (KeyError) -
  // so the second text pass reduces to remembering the first such token in reading order.
  TokenTable ent(&h->ent_names), rel(&h->rel_names);
  constexpr size_t kWindow = 16;                       // lines between a slot prefetch and its use
  std::vector<Token> win(3 * kWindow);
  std::string first_upper;
  bool any_upper = false;
  for (int s = 0; s < 3; ++s) {
    std::vector<int64_t>& tri = h->split[s].triples;
    tri.reserve(3 * (text[s].size() / 12 + 1));        // a line of three tokens holds >= 6 bytes; typical lines 15-40
    size_t seen = 0, done = 0;
    auto resolve = [&](const Token* t) {
      const int64_t a = ent.intern(t[0]), r = rel.intern(t[1]), o = ent.intern(t[2]);
      tri.insert(tri.end(), {a, r, o});
      if (!any_upper && (t[0].upper || t[1].upper || t[2].upper)) {
        const Token& u = t[0].upper ? t[0] : (t[1].upper ? t[1] : t[2]);
        first_upper.assign(u.p, u.len);
        any_upper = true;
      }
    };
    const int rc = for_each_line(text[s], &h->error, [&](const char** tok, const size_t* len) {
      if (seen - done == kWindow) resolve(&win[3 * (done++ % kWindow)]);
      Token* t = &win[3 * (seen++ % kWindow)];
      for (int k = 0; k < 3; ++k) TokenTable::scan(tok[k], len[k], &t[k]);
      ent.prefetch(t[0]);
      ent.prefetch(t[2]);
      return 0;
    });
    if (rc) {
      h->error = std::string(kNames[s]) + ": " + h->error;
      return rc;
    }
    while (done < seen) resolve(&win[3 * (done++ % kWindow)]);
    tri.shrink_to_fit();
  }
  const int64_t R = (int64_t)h->rel_names.size();
  for (const auto& name : h->rel_names)
    if (name.size() >= 8 && name.compare(name.size() - 8, 8, "_reverse") == 0) {
      // relation2id[name + '_reverse'] = id + R (data_loader.py:75-76) would alias it: leave such data to the Python passes
      h->error = "relation token ends with _reverse";
      return 2;
    }
  if (h->ent_names.size() >= (1ull << 31) || (uint64_t)(2 * R) >= (1ull << 31)) {
    h->error = "more than 2^31 entities or relations";
    return 3;
  }
  if (any_upper) {
    h->error = first_upper;                              // the reference raises KeyError(token) here
    return 4;
  }
  // ---- pass 2 (over the id triples): every line adds o to group (s, r) and s to group (o, r + R).  Groups get dense ids in
  // creation order (= Python's dict insertion order); memberships are kept as flat (group, value) pairs
  KeyTable gid;
  std::vector<int32_t> pair_g, pair_v;
  size_t n_train_groups = 0, n_train_pairs = 0;
  {
    size_t total = 0;
    for (int s = 0; s < 3; ++s) total += h->split[s].triples.size() / 3;
    pair_g.reserve(2 * total);
    pair_v.reserve(2 * total);
  }
  for (int s = 0; s < 3; ++s) {
    const std::vector<int64_t>& tri = h->split[s].triples;
    const size_t n_line = tri.size() / 3;
    auto key_tail = [&](size_t i) { return ((uint64_t)tri[3 * i] << 32) | (uint64_t)tri[3 * i + 1]; };
    auto key_head = [&](size_t i) { return ((uint64_t)tri[3 * i + 2] << 32) | (uint64_t)(tri[3 * i + 1] + R); };
    for (size_t i = 0; i < n_line && i < kWindow; ++i) { gid.prefetch(key_tail(i)); gid.prefetch(key_head(i)); }
    for (size_t i = 0; i < n_line; ++i) {
      if (i + kWindow < n_line) { gid.prefetch(key_tail(i + kWindow)); gid.prefetch(key_head(i + kWindow)); }
      pair_g.push_back(gid.find_or_insert(key_tail(i)));
      pair_v.push_back((int32_t)tri[3 * i + 2]);
      pair_g.push_back(gid.find_or_insert(key_head(i)));
      pair_v.push_back((int32_t)tri[3 * i]);
    }
    if (s == 0) {
      n_train_groups = gid.n;
      n_train_pairs = pair_g.size();
    }
  }
  const size_t n_groups = gid.n;
  std::vector<uint64_t> group_key(n_groups);
  for (const KeyTable::Slot& sl : gid.slots)
    if (sl.id >= 0) group_key[sl.id] = sl.key;
  // counting sort of the pairs by group: segment [ptr[g], ptr[g + 1]) holds group g's values in arrival order
  auto bucket = [&](size_t n_pairs, size_t n_g, std::vector<int64_t>* ptr, std::vector<int32_t>* val) {
    ptr->assign(n_g + 1, 0);
    for (size_t i = 0; i < n_pairs; ++i) ++(*ptr)[pair_g[i] + 1];
    for (size_t g = 0; g < n_g; ++g) (*ptr)[g + 1] += (*ptr)[g];
    val->resize(n_pairs);
    std::vector<int64_t> fill(ptr->begin(), ptr->end() - 1);
    for (size_t i = 0; i < n_pairs; ++i) (*val)[fill[pair_g[i]]++] = pair_v[i];
  };
  // ---- train queries: one per group created during the train split, train-only objects, sorted and unique
  {
    std::vector<int64_t> ptr;
    std::vector<int32_t> val;
    bucket(n_train_pairs, n_train_groups, &ptr, &val);
    Csr& c = h->csr[0];
    c.ptr.assign(n_train_groups + 1, 0);
    c.triples.resize(3 * n_train_groups);
    c.idx.reserve(val.size());
    for (size_t g = 0; g < n_train_groups; ++g) {
      int32_t* b = val.data() + ptr[g];
      int32_t* e = val.data() + ptr[g + 1];
      std::sort(b, e);
      e = std::unique(b, e);
      c.idx.insert(c.idx.end(), b, e);
      c.ptr[g + 1] = (int64_t)c.idx.size();
      c.triples[3 * g] = (int64_t)(group_key[g] >> 32);
      c.triples[3 * g + 1] = (int64_t)(group_key[g] & 0xffffffffu);
      c.triples[3 * g + 2] = -1;
    }
  }
  // ---- valid / test queries: the objects of ALL splits; a group is sorted the first time a query needs it and shared
  // by every later query (a hub group is referenced by thousands of queries)
  std::vector<int64_t> all_ptr, all_len;
  std::vector<int32_t> all_val;
  bucket(pair_g.size(), n_groups, &all_ptr, &all_val);
  all_len.assign(n_groups, -1);
  auto all_objs = [&](int64_t a, int64_t r, const int32_t** b) -> int64_t {
    const int32_t g = gid.find(((uint64_t)a << 32) | (uint64_t)r);
    int32_t* lo = all_val.data() + all_ptr[g];
    if (all_len[g] < 0) {
      int32_t* hi = all_val.data() + all_ptr[g + 1];
      std::sort(lo, hi);
      all_len[g] = std::unique(lo, hi) - lo;
    }
    *b = lo;
    return all_len[g];
  };
  for (int s = 1; s < 3; ++s) {
    const auto& tr = h->split[s].triples;
    for (int head = 0; head < 2; ++head) {
      Csr& c = h->csr[2 * s - 1 + head];
      std::vector<int32_t> local(n_groups, -1);             // group id -> its index among this set's groups
      c.ptr.assign(1, 0);
      for (size_t i = 0; i + 2 < tr.size(); i += 3) {
        const int64_t a = head ? tr[i + 2] : tr[i], r = head ? tr[i + 1] + R : tr[i + 1], o = head ? tr[i] : tr[i + 2];
        const int32_t g = gid.find(((uint64_t)a << 32) | (uint64_t)r);
        if (local[g] < 0) {
          const int32_t* b;
          const int64_t n = all_objs(a, r, &b);
          local[g] = (int32_t)c.ptr.size() - 1;
          c.idx.insert(c.idx.end(), b, b + n);
          c.ptr.push_back((int64_t)c.idx.size());
        }
        c.qg.push_back(local[g]);
        c.triples.insert(c.triples.end(), {a, r, o});
      }
    }
  }
  return 0;
}

}  // namespace

extern "C" int kgc_ingest_open(const char* data_dir, kgc_ingest_t** out) {
  if (!data_dir || !out) return kgc::fail(__func__, "null argument");
  kgc_ingest* h = new kgc_ingest();
  int rc;
  try {
    rc = ingest(data_dir, h);
  } catch (const std::exception& e) {
    h->error = e.what();
    rc = 3;
  }
  if (rc) {
    kgc::set_error(h->error);
    delete h;
    *out = nullptr;
    return rc;                     // 1 malformed line, 2 non-ASCII token (use the Python passes), 3 I/O, 4 unknown token
  }
  *out = h;
  return 0;
}

extern "C" void kgc_ingest_close(kgc_ingest_t* h) { delete h; }

// what: 0 entities, 1 relations (R, un-doubled), 2/3/4 triples of train / valid / test, 5/6 bytes of the token blobs,
//       10 + 2q / 11 + 2q = queries / stored label entries of query set q (0 train, 1 valid_tail, 2 valid_head, 3 test_tail,
//       4 test_head), 20 + q = rows of its ptr array (queries for train, referenced groups for valid / test)
extern "C" int64_t kgc_ingest_count(const kgc_ingest_t* h, int32_t what) {
  if (!h) return -1;
  if (what == 0) return (int64_t)h->ent_names.size();
  if (what == 1) return (int64_t)h->rel_names.size();
  if (what >= 2 && what <= 4) return (int64_t)h->split[what - 2].triples.size() / 3;
  if (what == 5 || what == 6) {                    // bytes of all entity / relation tokens, each followed by '\n'
    int64_t n = 0;
    for (const auto& t : (what == 5 ? h->ent_names : h->rel_names)) n += (int64_t)t.size() + 1;
    return n;
  }
  if (what >= 10 && what < 20) {                   // queries / stored label entries of a set
    const Csr& c = h->csr[(what - 10) / 2];
    return (what - 10) % 2 == 0 ? (int64_t)c.triples.size() / 3 : (int64_t)c.idx.size();
  }
  if (what >= 20 && what < 25) return (int64_t)h->csr[what - 20].ptr.size() - 1;     // rows of ptr: queries (train) / groups
  return -1;
}

// array: 5/6 entity / relation tokens in id order, each followed by '\n'; 2/3/4 triples of a split (int64 [n,3]); 10 + 3q triples (int64 [Q,3]), 11 + 3q ptr (int64 [rows+1]), 12 + 3q idx (int32), 30 + q query -> group (int32 [Q], valid / test)
extern "C" int kgc_ingest_copy(const kgc_ingest_t* h, int32_t array, void* dst, int64_t capacity_bytes) {
  if (!h || !dst) return kgc::fail(__func__, "null argument");
  const void* src = nullptr;
  size_t bytes = 0;
  if (array == 5 || array == 6) {                  // all tokens in id order, '\n'-separated
    char* out = static_cast<char*>(dst);
    int64_t used = 0;
    for (const auto& t : (array == 5 ? h->ent_names : h->rel_names)) {
      if (used + (int64_t)t.size() + 1 > capacity_bytes) return kgc::fail(__func__, "destination too small");
      memcpy(out + used, t.data(), t.size());
      used += (int64_t)t.size();
      out[used++] = '\n';
    }
    return 0;
  }
  if (array >= 2 && array <= 4) {
    src = h->split[array - 2].triples.data(); bytes = h->split[array - 2].triples.size() * 8;
  } else if (array >= 30 && array < 35) {          // query -> group of a valid / test set (empty for train)
    const Csr& c = h->csr[array - 30];
    src = c.qg.data(); bytes = c.qg.size() * 4;
  } else if (array >= 10 && array < 25) {
    const Csr& c = h->csr[(array - 10) / 3];
    switch ((array - 10) % 3) {
      case 0: src = c.triples.data(); bytes = c.triples.size() * 8; break;
      case 1: src = c.ptr.data(); bytes = c.ptr.size() * 8; break;
      default: src = c.idx.data(); bytes = c.idx.size() * 4; break;
    }
  } else {
    return kgc::fail(__func__, "unknown array id");
  }
  if ((int64_t)bytes > capacity_bytes) return kgc::fail(__func__, "destination too small");
  if (bytes) memcpy(dst, src, bytes);
  return 0;
}

// kind 0: entity token of id, kind 1: relation token of id (< R); NULL when out of range
extern "C" const char* kgc_ingest_name(const kgc_ingest_t* h, int32_t kind, int64_t id) {
  if (!h || id < 0) return nullptr;
  const auto& names = kind == 0 ? h->ent_names : h->rel_names;
  return (size_t)id < names.size() ? names[(size_t)id].c_str() : nullptr;
}
