// CTC prefix beam search for sm_100a, one warp per line (SURVEY.md 8(f) row 4: the search that replaces the toy
// per-frame beam of model_window/test_with_kenlm.py:25-59 in the LM-rescoring evaluation).
//
// The reference's `simple_ctc_beam_search_with_lm` ranks ALIGNMENT PATHS (ctc_kbest_kernel, beam.cu, restates it bit
// for bit); this kernel ranks LABELLINGS: every beam entry is a collapsed prefix l with the log-probability mass of
// all alignments of the frames seen so far that collapse to l, split into "ends in blank" (pb) and "ends in its last
// label" (pnb).  Per frame, with lp = the frame's log-probs and tot = lae(pb, pnb)  (lae = log-add-exp):
//   stay   l      : pb' = tot + lp[0];  pnb' = pnb + lp[last(l)]
//   extend l + c  : pnb' = (c == last(l) ? pb : tot) + lp[c];  pb' = -inf          for every label c >= 1
//   if l + c is itself an entry of the beam, its mass is ADDED to that entry's pnb' (one prefix, one entry)
//   the K entries with the largest lae(pb', pnb') survive; ties: stay entries (by rank) before extensions (by
//   parent rank, then label).
// With a beam wide enough to hold every prefix this is the exact labelling posterior (tests pin it to a brute-force
// enumeration of all alignments); all classes are extended, nothing is pruned by a per-frame class cut-off.
//
// Layout: the frame's log-probs live in registers (8 classes per lane) and in a per-warp smem row (for the stay
// terms); the two beam generations, the stay candidates and the winners of the selection rounds in per-warp smem;
// prefixes are identified by a 64-bit hash chain (the merge test is hash(parent) == hash of an entry one label
// shorter) and spelled out at the end from a per-line node array (parent node << 16 | label) in smem.  Scores are
// float64 in log space.  Selection = K rounds of a warp arg-max over the nb * (C - 1) + nb candidates in the strict
// total order (score desc, candidate number asc); a round looks for the best candidate that comes AFTER the previous
// winner in that order, so nothing has to be marked as taken.
//
// The LM-fused instantiation (LM = true, htrvt_ctc_prefix_beam_lm) ranks by lae(pb', pnb') + lm' instead, where lm is
// an entry's float64 sum of alpha * ln10 * log10 p(label | context) + beta over its labels (character n-gram, ARPA
// backoff).  The LM term of an extension depends only on (entry, label), so it is computed once, when the entry is
// created: the 32 lanes fill the entry's row of lm + term(c) for every class (and its </s> term) in a per-warp row pool
// of 2K rows; an entry that stays keeps its row.  The CTC masses (pb, pnb) are exactly those of the plain search.
//
// The lexicon-constrained instantiation (LEX = true, htrvt_ctc_prefix_beam_lex; with or without the LM) only accepts
// labellings whose every maximal run of word characters is a lexicon word (Scheidl et al. 2018, "Words" mode).  Each
// entry carries a trie node (0: between words) that its prefix alone determines, so the merge test stays valid.  Its
// pool row (the LM's bookkeeping, kept when LEX is on without the LM) holds two class bitmasks filled by the warp when
// the entry is created: `allow` (the classes the state machine permits from that node) and `allow_last` (those whose
// target state is between words or a word end).  The disallowed (entry, class) pairs are ORed into the fold mask
// `excl`, so the selection rounds skip them; in the line's last frame `allow_last` is used and an entry left inside an
// unfinished word cannot stay.  Ranking and scores are otherwise those of the plain / LM search: the lexicon only
// removes candidates.
//
// The word-LM instantiation (LM = LEX = true with PbWlmArgs, htrvt_ctc_prefix_beam_lex_wlm) scores the WORDS of the
// lexicon-constrained search with a word n-gram LM (Scheidl et al. 2018, "NGrams" mode).  Each pool row holds `done`
// (the float64 sum of alpha * ln10 * log10 p(word | <s> previous words) + beta over the entry's finished words) and the
// word context; its ranking value lm is done, plus alpha * ln10 * smear(node) inside a word (the best unigram
// log10 prob of the lexicon words below the node).  A created row costs at most two n-gram queries: the completion of
// the word ending at its node and the </s> term after it.
#include "common.cuh"
#include <climits>

namespace htrvt {

constexpr int kPbMaxK = 16;         // beam entries
constexpr int kPbCpl = 8;           // classes per lane held in registers: C <= 256
constexpr int kLmMaxOrder = 8;      // n-gram order: contexts of up to 7 tokens, keys of up to 8 16-bit fields
constexpr int kWlmMaxOrder = 6;     // word n-gram order: keys of up to 6 21-bit fields
constexpr int kWlmBits = 21;        // key-field width of the word LM's table (token ids < 2^21 - 1)
constexpr double kLn10 = 2.302585092994046;
constexpr int kLmUnk = 0, kLmBos = 1, kLmEos = 2;   // token ids of <unk>, <s>, </s>

// One slot of the LM's open-addressing table (32 bytes, one sector).  Key = the n-gram's tokens, LAST token first, as
// FB-bit fields (token + 1; 0 = no token), 64 / FB of them per word: lo holds the first, hi the next (character LM:
// FB = 16, fields 0-3 and 4-7; word LM: FB = 21, fields 0-2 and 3-5); lo == 0 marks an empty slot.  Keys are compared
// in full, so a hash collision never matches.  Linear probing from lm_hash(lo, hi) & (slots - 1).
struct PbLmSlot {
  unsigned long long lo, hi;
  float p, b;                        // log10 probability, log10 backoff
  unsigned long long pad;
};
struct PbLmArgs {
  const PbLmSlot* table;
  unsigned long long mask;           // slots - 1
  int order;
  const int* tok_map;                // class id -> token id (ids >= n_map: <unk>)
  int n_map;
  double alpha, beta;
  double* ctc_scores;
};
struct PbLmWarp {                   // LM state of one line; per pool row (2K rows), except row[] / skey[]
  double lm[2 * kPbMaxK];                                   // the row's entry: sum of its labels' LM terms
  double eos[2 * kPbMaxK];                                  // alpha ln10 log10 p(</s> | context)
  double skey[kPbMaxK];                                     // ranking key of every entry's stay candidate
  unsigned long long clo[2 * kPbMaxK], chi[2 * kPbMaxK];    // context, most recent token first, key-field layout
  int clen[2 * kPbMaxK];
  int row[2][kPbMaxK];                                      // pool row of entry j of generation g
  int nrow[kPbMaxK];                                        // rows created this frame
  float bow[kPbMaxK][kLmMaxOrder];                          // log10 bow of their contexts' suffixes (0: unlisted)
};

// Word lexicon as a trie in CSR form (htr-vt_b200/lexicon.py packs it): node 0 = root; the edges of node n are
// first[n] .. first[n + 1] - 1, sorted by label; is_word: class id -> word character (ids >= n_map: free).
struct PbLexArgs {
  const int* first;
  const int* label;
  const int* child;
  const unsigned char* word_end;
  const unsigned char* is_word;
  int n_map;
};
struct PbLexWarp {                  // lexicon state of one line; per pool row (2K rows), except freem[]
  int node[2 * kPbMaxK];                                    // trie node of the row's entry (0: between words)
  int fin[2 * kPbMaxK];                                     // node is 0 or ends a word
  unsigned allow[2 * kPbMaxK][kPbCpl];                      // bit (c & 31) of word c >> 5: c may extend the entry
  unsigned allow_last[2 * kPbMaxK][kPbCpl];                 // ... and leaves it between words or at a word end
  unsigned freem[kPbCpl];                                   // the free classes 1 .. C - 1
};

// Word n-gram LM over the lexicon's trie (htr-vt_b200/wordlm.py packs it); the table, order and weights come in
// PbLmArgs (tok_map unused), the trie in PbLexArgs.  node_tok: trie node -> token id of the word ending there; smear:
// trie node -> the largest unigram log10 prob of the lexicon words that start with the node's prefix.
struct PbWlmArgs {
  const int* node_tok;
  const float* smear;
};
struct PbWlmWarp {                  // word-LM state of one line
  double done[2 * kPbMaxK];                                 // per pool row: the finished words' LM terms
  double comp[kPbMaxK], eosq[kPbMaxK];                      // per row created this frame: completion, </s> term
};

struct PbGen {                      // one beam generation of one line
  double pb[kPbMaxK], pnb[kPbMaxK], tot[kPbMaxK];
  unsigned long long hash[kPbMaxK], phash[kPbMaxK];
  int last[kPbMaxK], len[kPbMaxK], node[kPbMaxK];
};
struct PbWarp {
  PbGen gen[2];
  double spb[kPbMaxK], spnb[kPbMaxK], stot[kPbMaxK];        // the stay candidate of every entry
  double win_s[kPbMaxK];
  int win_n[kPbMaxK];
  int mrg_i[kPbMaxK], mrg_c[kPbMaxK];                       // entry j absorbed the extension (mrg_i, mrg_c), or -1
  float lp[32 * kPbCpl];
};

__device__ __forceinline__ double lae(double a, double b) {
  if (a == -INFINITY) return b;
  if (b == -INFINITY) return a;
  return fmax(a, b) + log1p(exp(-fabs(a - b)));
}
__device__ __forceinline__ unsigned long long pb_hash(unsigned long long h, int c) {
  h = (h ^ (static_cast<unsigned long long>(c) + 0x9e3779b97f4a7c15ull)) * 0xff51afd7ed558ccdull;
  return h ^ (h >> 32);
}
// order-preserving integer image of a double (-0.0 folded onto +0.0), its inverse, and the candidate order
// (score descending, candidate number ascending)
__device__ __forceinline__ long long pb_key(double s) {
  long long b = __double_as_longlong(s);
  if ((b << 1) == 0) b = 0;
  return b ^ ((b >> 63) & 0x7fffffffffffffffLL);
}
__device__ __forceinline__ double pb_unkey(long long k) {
  return __longlong_as_double(k ^ ((k >> 63) & 0x7fffffffffffffffLL));
}
__device__ __forceinline__ bool pb_before(long long k, int n, long long bk, int bn) {  // (k, n) ranks before (bk, bn)
  return k > bk || (k == bk && n < bn);
}

// ---- character n-gram LM ------------------------------------------------------------------------------------------
// (mirrored bit for bit by htr-vt_b200/lm.py::lm_hash, which packs the table)
__device__ __forceinline__ unsigned long long lm_hash(unsigned long long lo, unsigned long long hi) {
  unsigned long long h = lo * 0x9e3779b97f4a7c15ull + hi * 0xc2b2ae3d27d4eb4full;
  h ^= h >> 31;
  h *= 0xbf58476d1ce4e5b9ull;
  return h ^ (h >> 29);
}
__device__ __forceinline__ ulonglong2 lm_key_at(const PbLmSlot* t, unsigned long long i) {
  return __ldg(reinterpret_cast<const ulonglong2*>(t + i));
}
__device__ __forceinline__ float2 lm_val_at(const PbLmSlot* t, unsigned long long i) {
  return __ldg(reinterpret_cast<const float2*>(t + i) + 2);
}
// the rest of a probe whose first slot (i, s) is already loaded: the slot holding (lo, hi), or -1
__device__ __forceinline__ long long lm_walk(const PbLmSlot* t, unsigned long long mask, unsigned long long lo,
                                             unsigned long long hi, unsigned long long i, ulonglong2 s) {
  for (unsigned long long n = 0; n <= mask; ++n) {
    if (s.x == lo && s.y == hi) return static_cast<long long>(i);
    if (s.x == 0ull) return -1;
    i = (i + 1) & mask;
    s = lm_key_at(t, i);
  }
  return -1;
}
// the first m fields of a context (key-field layout, FB-bit fields)
template <int FB>
__device__ __forceinline__ void lm_ctx_prefix(unsigned long long clo, unsigned long long chi, int m,
                                              unsigned long long& lo, unsigned long long& hi) {
  constexpr int P = 64 / FB;                               // fields per word
  if (m >= P) {
    lo = clo;
    hi = chi & ((1ull << (FB * (m - P))) - 1ull);
  } else {
    lo = clo & ((1ull << (FB * m)) - 1ull);
    hi = 0ull;
  }
}
// (lo, hi) shifted by one field with token tok in field 0: a key (w first) or a context (most recent token first)
template <int FB>
__device__ __forceinline__ void lm_push(unsigned long long lo, unsigned long long hi, int tok, unsigned long long& klo,
                                        unsigned long long& khi) {
  constexpr int P = 64 / FB;
  constexpr unsigned long long used = FB * P == 64 ? ~0ull : (1ull << (FB * P)) - 1ull;
  klo = ((lo << FB) | static_cast<unsigned long long>(tok + 1)) & used;
  khi = ((hi << FB) | (lo >> (FB * (P - 1)))) & used;
}
__device__ __forceinline__ int lm_tok(const PbLmArgs& a, int c) { return c < a.n_map ? __ldg(a.tok_map + c) : kLmUnk; }

// log10 p(w | context) by ARPA backoff over the levels m = M .. 0 of one query, whose first slots are already loaded
// (level m: key (klo[m], khi[m]) = (last m context tokens, w), first slot ix[m] with key s[m] and prob p[m]): the listed
// prob of the longest level in the table, plus the bow of every longer level's context, summed in float64
// longest-context bow first and the found prob last; unk when no level is listed.  add_bow(m, S) adds level m's
// context bow (0 when that context is unlisted) to S.
template <int N, typename AddBow>
__device__ __forceinline__ double lm_backoff(const PbLmArgs& a, const unsigned long long* klo,
                                             const unsigned long long* khi, const unsigned long long* ix,
                                             const ulonglong2* s, const float* p, int M, float unk, AddBow add_bow) {
  double S = 0.0;
  bool found = false;
#pragma unroll
  for (int m = N - 1; m >= 0; --m) {
    if (m <= M && !found) {
      if (s[m].x == klo[m] && s[m].y == khi[m]) {
        S += static_cast<double>(p[m]);
        found = true;
      } else {
        const long long f = s[m].x == 0ull ? -1 : lm_walk(a.table, a.mask, klo[m], khi[m], ix[m], s[m]);
        if (f >= 0) {
          S += static_cast<double>(lm_val_at(a.table, static_cast<unsigned long long>(f)).x);
          found = true;
        } else if (m > 0) {
          add_bow(m, S);
        }
      }
    }
  }
  if (!found) S += static_cast<double>(unk);
  return S;
}

// Fill the rows L->nrow[0 .. nE) (their lm / context already set): row[c] = lm + alpha ln10 S(c) + beta for every label
// c, eos = alpha ln10 S(</s>), with S(w) = log10 p(w | context) (lm_backoff; the context bows are looked up first, once
// per row).  All 32 lanes, (row, class) pairs spread over lanes; a lane issues the first-slot loads of every level of
// its query before it looks at any of them.
__device__ __forceinline__ void lm_fill_rows(const PbLmArgs& a, PbLmWarp* L, double* rows, int nE, int C, float unk,
                                          int lane) {
  const int M1 = a.order - 1;
  for (int idx = lane; idx < nE * M1; idx += 32) {            // context bows: (row, suffix length k = 1 .. clen)
    const int e = idx / M1, k = idx - e * M1 + 1;
    const int r = L->nrow[e];
    float bw = 0.f;
    if (k <= L->clen[r]) {
      unsigned long long lo, hi;
      lm_ctx_prefix<16>(L->clo[r], L->chi[r], k, lo, hi);
      const unsigned long long i = lm_hash(lo, hi) & a.mask;
      const long long f = lm_walk(a.table, a.mask, lo, hi, i, lm_key_at(a.table, i));
      if (f >= 0) bw = lm_val_at(a.table, static_cast<unsigned long long>(f)).y;
    }
    L->bow[e][k - 1] = bw;
  }
  __syncwarp();
  const int Cm = C - 1;
  for (int idx = lane; idx < nE * C; idx += 32) {             // nE * (C - 1) labels, then nE </s> queries
    int e, c, tok;
    if (idx < nE * Cm) {
      e = idx / Cm;
      c = idx - e * Cm + 1;
      tok = lm_tok(a, c);
    } else {
      e = idx - nE * Cm;
      c = -1;
      tok = kLmEos;
    }
    const int r = L->nrow[e];
    const int M = L->clen[r];
    const unsigned long long clo = L->clo[r], chi = L->chi[r];
    unsigned long long klo[kLmMaxOrder], khi[kLmMaxOrder], ix[kLmMaxOrder];
    ulonglong2 s[kLmMaxOrder];
    float p[kLmMaxOrder];
#pragma unroll
    for (int m = 0; m < kLmMaxOrder; ++m) {                   // key of (last m context tokens, w): w first
      if (m <= M) {
        unsigned long long lo, hi;
        lm_ctx_prefix<16>(clo, chi, m, lo, hi);
        lm_push<16>(lo, hi, tok, klo[m], khi[m]);
        ix[m] = lm_hash(klo[m], khi[m]) & a.mask;
        s[m] = lm_key_at(a.table, ix[m]);
        p[m] = lm_val_at(a.table, ix[m]).x;
      }
    }
    const double S = lm_backoff<kLmMaxOrder>(a, klo, khi, ix, s, p, M, unk, [&](int m, double& sum) {
      sum += static_cast<double>(L->bow[e][m - 1]);
    });
    const double t = __dmul_rn(a.alpha, __dmul_rn(kLn10, S));   // no contraction: the oracle's arithmetic
    if (c < 0) L->eos[r] = t;
    else rows[r * C + c] = __dadd_rn(L->lm[r], __dadd_rn(t, a.beta));
  }
  __syncwarp();
}

// ---- word lexicon ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool lex_free(const PbLexArgs& a, int c) { return c >= a.n_map || !__ldg(a.is_word + c); }

// Fill the masks of rows L->nrow[0 .. nE) (their node / fin already set).  From a finished node (0 or a word end) every
// free class leads back to state 0, which both masks accept; a child edge c leads to the child, which allow_last
// accepts only when the child ends a word.  All 32 lanes: first the free-class part word by word, then the child edges.
// WLM: the child edges' LM row entries too, done + alpha ln10 smear(child) (the other classes are already filled).
template <int CPL, bool WLM>
__device__ __forceinline__ void lex_fill_rows(const PbLexArgs& a, const PbLmWarp* L, PbLexWarp* X, int nE, int C,
                                              int lane, double* rows, const double* done, const float* smear,
                                              double alpha) {
  for (int idx = lane; idx < nE * CPL; idx += 32) {
    const int e = idx / CPL, w = idx - e * CPL;
    const int r = L->nrow[e];
    const unsigned m = X->fin[r] ? X->freem[w] : 0u;
    X->allow[r][w] = m;
    X->allow_last[r][w] = m;
  }
  __syncwarp();
  for (int e = 0; e < nE; ++e) {
    const int r = L->nrow[e];
    const int n = X->node[r];
    const int j1 = __ldg(a.first + n + 1);
    for (int j = __ldg(a.first + n) + lane; j < j1; j += 32) {
      const int c = __ldg(a.label + j);
      if (c < C) {
        const unsigned bit = 1u << (c & 31);
        atomicOr(&X->allow[r][c >> 5], bit);
        if (__ldg(a.word_end + __ldg(a.child + j))) atomicOr(&X->allow_last[r][c >> 5], bit);
        if constexpr (WLM) {
          const double sm = static_cast<double>(__ldg(smear + __ldg(a.child + j)));
          rows[r * C + c] = __dadd_rn(done[r], __dmul_rn(alpha, __dmul_rn(kLn10, sm)));
        }
      }
    }
  }
  __syncwarp();
}
// the trie node an entry at node n moves to by the allowed class c: 0 for a free class, else child(n, c)
__device__ __forceinline__ int lex_step(const PbLexArgs& a, int n, int c) {
  if (lex_free(a, c)) return 0;
  int lo = __ldg(a.first + n), hi = __ldg(a.first + n + 1) - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(a.label + mid) < c) lo = mid + 1;
    else hi = mid;
  }
  return __ldg(a.child + lo);
}

// ---- word n-gram LM -------------------------------------------------------------------------------------------------
// log10 p(tok | context) (lm_backoff) for one query in one lane: context (clo, chi) of M <= kWlmMaxOrder - 1 tokens;
// the first slots of every level's n-gram key and context key are loaded before any of them is looked at.
__device__ __forceinline__ double wlm_logprob(const PbLmArgs& a, unsigned long long clo, unsigned long long chi, int M,
                                              int tok, float unk) {
  unsigned long long klo[kWlmMaxOrder], khi[kWlmMaxOrder], ix[kWlmMaxOrder];
  unsigned long long blo[kWlmMaxOrder], bhi[kWlmMaxOrder], bix[kWlmMaxOrder];
  ulonglong2 s[kWlmMaxOrder], bs[kWlmMaxOrder];
  float p[kWlmMaxOrder], bw[kWlmMaxOrder];
#pragma unroll
  for (int m = 0; m < kWlmMaxOrder; ++m) {                   // level m: (last m context tokens, tok) and its context
    if (m <= M) {
      lm_ctx_prefix<kWlmBits>(clo, chi, m, blo[m], bhi[m]);
      lm_push<kWlmBits>(blo[m], bhi[m], tok, klo[m], khi[m]);
      ix[m] = lm_hash(klo[m], khi[m]) & a.mask;
      s[m] = lm_key_at(a.table, ix[m]);
      p[m] = lm_val_at(a.table, ix[m]).x;
      if (m > 0) {
        bix[m] = lm_hash(blo[m], bhi[m]) & a.mask;
        bs[m] = lm_key_at(a.table, bix[m]);
        bw[m] = lm_val_at(a.table, bix[m]).y;
      }
    }
  }
  return lm_backoff<kWlmMaxOrder>(a, klo, khi, ix, s, p, M, unk, [&](int m, double& sum) {
    if (bs[m].x == blo[m] && bs[m].y == bhi[m]) {
      sum += static_cast<double>(bw[m]);
    } else {
      const long long g = bs[m].x == 0ull ? -1 : lm_walk(a.table, a.mask, blo[m], bhi[m], bix[m], bs[m]);
      if (g >= 0) sum += static_cast<double>(lm_val_at(a.table, static_cast<unsigned long long>(g)).y);
    }
  });
}

// Fill the word-LM rows L->nrow[0 .. nE) (node / fin, done and context already set), before lex_fill_rows<CPL, true>
// writes their child edges.  An entry at a finished node n (0 or a word end) with context h: comp = alpha ln10
// log10 p(node_tok[n] | h) + beta when n != 0, eos = [comp +] alpha ln10 log10 p(</s> | h') with h' = node_tok[n] h
// truncated (h when n == 0); row[c] = done (+ comp when n != 0) for the free classes c.  Inside a word nothing is
// queried (no free class is allowed there and the entry cannot end the line).  Query lane 2 e: comp, 2 e + 1: </s>.
__device__ __forceinline__ void wlm_fill_rows(const PbLmArgs& a, const PbWlmArgs& w, PbLmWarp* L, const PbLexWarp* X,
                                              PbWlmWarp* Y, double* rows, int nE, int C, float unk, int lane) {
  const int M1 = a.order - 1;
  for (int idx = lane; idx < 2 * nE; idx += 32) {
    const int e = idx >> 1, r = L->nrow[e], n = X->node[r];
    if (!X->fin[r]) continue;
    unsigned long long lo = L->clo[r], hi = L->chi[r];
    int M = L->clen[r], tok = kLmEos;
    if ((idx & 1) == 0) {
      if (n == 0) {
        Y->comp[e] = 0.0;
        continue;
      }
      tok = __ldg(w.node_tok + n);
    } else if (n != 0) {
      lm_push<kWlmBits>(lo, hi, __ldg(w.node_tok + n), lo, hi);
      lm_ctx_prefix<kWlmBits>(lo, hi, M1, lo, hi);
      M = min(M + 1, M1);
    }
    const double t = __dmul_rn(a.alpha, __dmul_rn(kLn10, wlm_logprob(a, lo, hi, M, tok, unk)));
    if ((idx & 1) == 0) Y->comp[e] = __dadd_rn(t, a.beta);
    else Y->eosq[e] = t;
  }
  __syncwarp();
  const int Cm = C - 1;
  for (int idx = lane; idx < nE * C; idx += 32) {             // nE * (C - 1) labels, then nE eos terms
    const int e = idx < nE * Cm ? idx / Cm : idx - nE * Cm;
    const int r = L->nrow[e];
    const bool wend = X->fin[r] && X->node[r] != 0;
    if (idx < nE * Cm) {
      const int c = idx - e * Cm + 1;
      const bool fr = (X->freem[c >> 5] >> (c & 31)) & 1u;
      rows[r * C + c] = (fr && wend) ? __dadd_rn(Y->done[r], Y->comp[e]) : Y->done[r];
    } else {
      L->eos[r] = !X->fin[r] ? 0.0 : wend ? __dadd_rn(Y->comp[e], Y->eosq[e]) : Y->eosq[e];
    }
  }
  __syncwarp();
}

// Shared memory of a CTA of `warps` lines: the byte offset of each region and the total.  Region-major over the warps,
// in this order: PbWarp; PbLmWarp (LM or LEX: the pool rows' bookkeeping); the LM row pool, 2K rows of C doubles (LM);
// PbLexWarp (LEX); PbWlmWarp (WLM); the node array, T K + 1 entries.  A region starts at warps times the per-warp bytes
// of the regions before it.  The launcher sizes the launch with it and the kernel finds its warp's state with it.
struct PbSmem {
  size_t lm, rows, lex, wlm, nodes, bytes;
};
__host__ __device__ __forceinline__ PbSmem pb_smem_layout(bool LM, bool LEX, bool WLM, int K, int C, int T, int warps) {
  // (the pool rows' bytes summed first: ptxas schedules the LM kernels' prologue by the grouping of these sums)
  const size_t pool = (LM || LEX) ? sizeof(PbLmWarp) + (LM ? sizeof(double) * 2 * K * C : 0) : 0;
  const size_t lm = sizeof(PbWarp);
  const size_t rows = lm + ((LM || LEX) ? sizeof(PbLmWarp) : 0);
  const size_t lex = lm + pool;
  const size_t wlm = lex + (LEX ? sizeof(PbLexWarp) : 0);
  const size_t nodes = wlm + (WLM ? sizeof(PbWlmWarp) : 0);
  const size_t bytes = nodes + (static_cast<size_t>(T) * K + 1) * 4;
  return {lm * warps, rows * warps, lex * warps, wlm * warps, nodes * warps, bytes * warps};
}

// class slots per lane: C <= 32 * CPL; LM: fused n-gram LM; LEX: word lexicon constraint; WLM (with LM and LEX): the
// LM is the word LM, every character-LM step inside `if constexpr (!WLM)`.  Every instantiation takes the three
// argument structs; a variant leaves those it does not use zero-filled, and every state it does not use is touched
// only inside `if constexpr` on its flag.
// (Min. blocks 1 for LEX: without it ptxas caps some lexicon instantiations at 56-128 registers and spills.)
template <int CPL, bool LM, bool LEX, bool WLM>
__global__ void __launch_bounds__(128, LEX ? 1 : 0) ctc_prefix_beam_kernel(const float* __restrict__ x, long long sb, long long st,
                                                              const int* __restrict__ lengths, int B, int T, int C,
                                                              int K, int* __restrict__ ids, int* __restrict__ lens,
                                                              double* __restrict__ scores, PbLmArgs la, PbLexArgs xa,
                                                              PbWlmArgs wa) {
  static_assert(!WLM || (LM && LEX), "the word LM runs inside the lexicon-constrained LM search");
  extern __shared__ __align__(16) uint8_t pb_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  const int b = blockIdx.x * warps + warp;
  if (b >= B) return;
  PbWarp* W = reinterpret_cast<PbWarp*>(pb_smem) + warp;
  const PbSmem sm = pb_smem_layout(LM, LEX, WLM, K, C, T, warps);
  PbLmWarp* L = reinterpret_cast<PbLmWarp*>(pb_smem + sm.lm) + warp;
  double* rows = reinterpret_cast<double*>(pb_smem + sm.rows) + static_cast<size_t>(warp) * 2 * K * C;
  PbLexWarp* X = reinterpret_cast<PbLexWarp*>(pb_smem + sm.lex) + warp;
  PbWlmWarp* Y = reinterpret_cast<PbWlmWarp*>(pb_smem + sm.wlm) + warp;
  uint32_t* nodes = reinterpret_cast<uint32_t*>(pb_smem + sm.nodes) +
                    static_cast<size_t>(warp) * (static_cast<size_t>(T) * K + 1);
  int Tb = lengths ? lengths[b] : T;
  Tb = min(max(Tb, 0), T);
  const float* xb = x + static_cast<long long>(b) * sb;

  int cur = 0, nb = 1, nnodes = 1;
  if (lane == 0) {
    PbGen& g = W->gen[0];
    g.pb[0] = 0.0; g.pnb[0] = -INFINITY; g.tot[0] = 0.0;
    g.hash[0] = 0x243f6a8885a308d3ull; g.phash[0] = 0ull;
    g.last[0] = -1; g.len[0] = 0; g.node[0] = 0;
    nodes[0] = 0u;
  }
  unsigned used = 1u;                 // LM / LEX: pool rows held by the current generation
  float unk = -100.f;                 // LM: log10 p(<unk>) (-100 when the LM does not list it)
  if constexpr (LM) {
    const ulonglong2 s = lm_key_at(la.table, lm_hash(kLmUnk + 1, 0ull) & la.mask);
    const long long f = lm_walk(la.table, la.mask, kLmUnk + 1, 0ull, lm_hash(kLmUnk + 1, 0ull) & la.mask, s);
    if (f >= 0) unk = lm_val_at(la.table, static_cast<unsigned long long>(f)).x;
    if (lane == 0) {                                     // the empty prefix: context <s>, row 0
      L->row[0][0] = 0; L->nrow[0] = 0; L->lm[0] = 0.0;
      L->clen[0] = min(1, la.order - 1);
      L->clo[0] = la.order > 1 ? static_cast<unsigned long long>(kLmBos + 1) : 0ull;
      L->chi[0] = 0ull;
      if constexpr (WLM) Y->done[0] = 0.0;
    }
    __syncwarp();
    if constexpr (!WLM) lm_fill_rows(la, L, rows, 1, C, unk, lane);
  }
  if constexpr (LEX) {
#pragma unroll
    for (int u = 0; u < CPL; ++u) {
      const int c = lane + 32 * u;
      const unsigned fw = __ballot_sync(0xffffffffu, c >= 1 && c < C && lex_free(xa, c));
      if (lane == 0) X->freem[u] = fw;
    }
    if (lane == 0) {                                     // the empty prefix: between words, row 0
      L->row[0][0] = 0; L->nrow[0] = 0;
      X->node[0] = 0; X->fin[0] = 1;
    }
    __syncwarp();
    if constexpr (WLM) wlm_fill_rows(la, wa, L, X, Y, rows, 1, C, unk, lane);
    lex_fill_rows<CPL, WLM>(xa, L, X, 1, C, lane, rows, Y->done, wa.smear, la.alpha);
  }
  float v[CPL], vn[CPL];
#pragma unroll
  for (int u = 0; u < CPL; ++u) {
    const int c = lane + 32 * u;
    v[u] = (c < C && Tb > 0) ? __ldg(xb + c) : -INFINITY;
    vn[u] = -INFINITY;
  }
  __syncwarp();

  for (int t = 0; t < Tb; ++t) {
    if (t + 1 < Tb) {
      const float* xr = xb + static_cast<long long>(t + 1) * st;
#pragma unroll
      for (int u = 0; u < CPL; ++u) {
        const int c = lane + 32 * u;
        if (c < C) vn[u] = __ldg(xr + c);
      }
    }
#pragma unroll
    for (int u = 0; u < CPL; ++u) W->lp[lane + 32 * u] = v[u];
    __syncwarp();
    const PbGen& g = W->gen[cur];
    PbGen& gn = W->gen[cur ^ 1];

    // ---- stay candidates; an extension that spells an existing entry is folded into that entry ----------
    if (lane < nb) {
      const int j = lane;
      const double totj = g.tot[j];
      const double npb = totj + static_cast<double>(W->lp[0]);
      double npnb = g.len[j] > 0 ? g.pnb[j] + static_cast<double>(W->lp[g.last[j]]) : -INFINITY;
      int mi = -1;
      if (g.len[j] > 0) {
        const unsigned long long ph = g.phash[j];
        for (int i = 0; i < nb; ++i)
          if (g.hash[i] == ph && g.len[i] == g.len[j] - 1) mi = i;
      }
      if (mi >= 0) {
        const int c = g.last[j];
        const double base = (g.len[mi] > 0 && g.last[mi] == c) ? g.pb[mi] : g.tot[mi];
        npnb = lae(npnb, base + static_cast<double>(W->lp[c]));
      }
      W->mrg_i[j] = mi;
      W->mrg_c[j] = g.last[j];
      W->spb[j] = npb;
      W->spnb[j] = npnb;
      W->stot[j] = lae(npb, npnb);
      if constexpr (LM) L->skey[j] = W->stot[j] + L->lm[L->row[cur][j]];
    }
    __syncwarp();
    unsigned excl[CPL];                                   // bit i of excl[u]: extension (i, lane + 32 u) was folded
#pragma unroll
    for (int u = 0; u < CPL; ++u) {                       // the blank and classes beyond C are never extensions
      const int c = lane + 32 * u;
      excl[u] = (c >= 1 && c < C) ? 0u : 0xffffffffu;
    }
    for (int j = 0; j < nb; ++j) {
      const int mi = W->mrg_i[j], mc = W->mrg_c[j];
      if (mi >= 0 && (mc & 31) == lane) {
#pragma unroll
        for (int u = 0; u < CPL; ++u)
          if (u == (mc >> 5)) excl[u] |= 1u << mi;
      }
    }
    if constexpr (LEX) {                                  // the extensions the lexicon forbids join the folded ones
      const bool last = t + 1 == Tb;
      for (int i = 0; i < nb; ++i) {
        const int r = L->row[cur][i];
        const unsigned* m = last ? X->allow_last[r] : X->allow[r];
#pragma unroll
        for (int u = 0; u < CPL; ++u)
          if (!((m[u] >> lane) & 1u)) excl[u] |= 1u << i;
      }
    }

    // ---- K selection rounds ---------------------------------------------------------------------------------
    // Scores are compared as order-preserving 64-bit integer images of the doubles; the sentinel (LLONG_MIN, INT_MAX)
    // loses against every real candidate.  Every lane scans ITS candidates (its class slots x all entries, + its
    // stay candidate) ONCE per frame for its local best; a round is then a warp arg-max over the 32 local bests, and
    // only the winner's lane needs a new local best (the best of its candidates that comes after the winner in the
    // strict order) - found by all 32 lanes together, <= ceil((nb * CPL + 1) / 32) candidates each, from the smem
    // copy of the frame's log-probs.  K scans of nb * CPL candidates per lane become one.
    long long lk = LLONG_MIN;                                // this lane's best remaining candidate
    int ln = 0x7fffffff;
    {
      long long bku[CPL];
      int bnu[CPL];
#pragma unroll
      for (int u = 0; u < CPL; ++u) { bku[u] = LLONG_MIN; bnu[u] = 0x7fffffff; }
      bool stay = lane < nb;
      if constexpr (LEX)                                  // last frame: no stay inside an unfinished word
        stay = stay && (t + 1 < Tb || X->fin[L->row[cur][lane]]);
      if (stay) { bku[0] = pb_key(LM ? L->skey[lane] : W->stot[lane]); bnu[0] = lane; }
#pragma unroll 4
      for (int i = 0; i < nb; ++i) {
        const double ti = g.tot[i], pbi = g.pb[i];
        const int li = g.len[i] > 0 ? g.last[i] : -1;
        const int n0 = K + i * C;
        const double* rw = LM ? rows + L->row[cur][i] * C : nullptr;
#pragma unroll
        for (int u = 0; u < CPL; ++u) {
          const int c = lane + 32 * u;
          if (!((excl[u] >> i) & 1u)) {
            double s = (c == li ? pbi : ti) + static_cast<double>(v[u]);
            if constexpr (LM) s = s + rw[c];
            const long long k = pb_key(s);
            if (pb_before(k, n0 + c, bku[u], bnu[u])) { bku[u] = k; bnu[u] = n0 + c; }
          }
        }
      }
      lk = bku[0]; ln = bnu[0];
#pragma unroll
      for (int u = 1; u < CPL; ++u)
        if (pb_before(bku[u], bnu[u], lk, ln)) { lk = bku[u]; ln = bnu[u]; }
    }
    int nnew = 0;
    for (int r = 0; r < K; ++r) {
      long long bk = lk;
      int bn = ln;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const long long ok = __shfl_xor_sync(0xffffffffu, bk, o);
        const int on = __shfl_xor_sync(0xffffffffu, bn, o);
        if (pb_before(ok, on, bk, bn)) { bk = ok; bn = on; }
      }
      if (bn == 0x7fffffff) break;                            // fewer than K candidates exist
      if (lane == 0) { W->win_s[r] = pb_unkey(bk); W->win_n[r] = bn; }
      nnew = r + 1;
      if (r + 1 == K) break;
      // the owner lane of the winner and its class slots' fold masks
      const int own = bn < K ? bn : (((bn - K) % C) & 31);
      unsigned oex[CPL];
#pragma unroll
      for (int u = 0; u < CPL; ++u) oex[u] = __shfl_sync(0xffffffffu, excl[u], own);
      long long ck = LLONG_MIN;
      int cn = 0x7fffffff;
      const int M = nb * CPL;
      for (int idx = lane; idx <= M; idx += 32) {
        long long k;
        int n;
        bool ok;
        if (idx == M) {                                       // the owner's stay candidate
          ok = own < nb;
          if constexpr (LEX)                              // left out: a LLONG_MIN key would still beat the sentinel
            ok = ok && (t + 1 < Tb || X->fin[L->row[cur][own]]);
          k = ok ? pb_key(LM ? L->skey[own] : W->stot[own]) : LLONG_MIN;
          n = own;
        } else {
          const int i = idx / CPL, u = idx - i * CPL;
          const int c = own + 32 * u;
          unsigned ex = 0u;
#pragma unroll
          for (int q = 0; q < CPL; ++q)
            if (q == u) ex = oex[q];
          ok = !((ex >> i) & 1u);                             // (invalid classes carry an all-ones mask)
          const int li = g.len[i] > 0 ? g.last[i] : -1;
          if (ok) {
            double s = (c == li ? g.pb[i] : g.tot[i]) + static_cast<double>(W->lp[c]);
            if constexpr (LM) s = s + rows[L->row[cur][i] * C + c];
            k = pb_key(s);
          } else {
            k = LLONG_MIN;
          }
          n = K + i * C + c;
        }
        if (ok && pb_before(bk, bn, k, n) && pb_before(k, n, ck, cn)) { ck = k; cn = n; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const long long ok2 = __shfl_xor_sync(0xffffffffu, ck, o);
        const int on = __shfl_xor_sync(0xffffffffu, cn, o);
        if (pb_before(ok2, on, ck, cn)) { ck = ok2; cn = on; }
      }
      if (lane == own) { lk = ck; ln = cn; }
    }
    __syncwarp();

    // ---- the next generation: lane r builds entry r -------------------------------------------------------
    int n = 0, pi = 0, c = 0;
    bool ext = false;
    if (lane < nnew) {
      n = W->win_n[lane];
      ext = n >= K;
      if (ext) { pi = (n - K) / C; c = (n - K) - pi * C; }
    }
    const unsigned em = __ballot_sync(0xffffffffu, ext);
    int nr = 0;                                               // LM / LEX: the entry's pool row
    if (lane < nnew) {
      // (win_s is the ranking key; with the LM it is not the CTC mass, which is then recomputed: + 0.0 folds -0.0
      // onto +0.0 as the integer image of win_s does, so that alpha = beta = 0 reproduces the plain search bit for bit)
      if (!ext) {
        gn.pb[lane] = W->spb[n]; gn.pnb[lane] = W->spnb[n]; gn.tot[lane] = LM ? W->stot[n] + 0.0 : W->win_s[lane];
        gn.hash[lane] = g.hash[n]; gn.phash[lane] = g.phash[n];
        gn.last[lane] = g.last[n]; gn.len[lane] = g.len[n]; gn.node[lane] = g.node[n];
        if constexpr (LM || LEX) { nr = L->row[cur][n]; L->row[cur ^ 1][lane] = nr; }
      } else {
        const int q = __popc(em & ((1u << lane) - 1u));
        const int nd = nnodes + q;
        nodes[nd] = (static_cast<uint32_t>(g.node[pi]) << 16) | static_cast<uint32_t>(c);
        double s = W->win_s[lane];
        if constexpr (LM) {
          const int li = g.len[pi] > 0 ? g.last[pi] : -1;
          s = ((c == li ? g.pb[pi] : g.tot[pi]) + static_cast<double>(W->lp[c])) + 0.0;
        }
        gn.pb[lane] = -INFINITY; gn.pnb[lane] = s; gn.tot[lane] = s;
        gn.hash[lane] = pb_hash(g.hash[pi], c); gn.phash[lane] = g.hash[pi];
        gn.last[lane] = c; gn.len[lane] = g.len[pi] + 1; gn.node[lane] = nd;
        if constexpr (LM || LEX) {                            // a free row (not held by generation cur), q-th of them
          unsigned fr = ~used & (K == 16 ? 0xffffffffu : (1u << (2 * K)) - 1u);
          for (int z = 0; z < q; ++z) fr &= fr - 1u;
          nr = __ffs(fr) - 1;
        }
        if constexpr (LM) {
          const int pr = L->row[cur][pi];
          L->lm[nr] = rows[pr * C + c];
          const int M = L->clen[pr];
          const int M1 = la.order - 1;
          if constexpr (WLM) {                                // a free class after a word end finishes that word
            const int pn = X->node[pr];
            unsigned long long lo = L->clo[pr], hi = L->chi[pr];
            int m = M;
            if (lex_free(xa, c)) {
              Y->done[nr] = L->lm[nr];
              if (pn != 0) {
                lm_push<kWlmBits>(lo, hi, __ldg(wa.node_tok + pn), lo, hi);
                lm_ctx_prefix<kWlmBits>(lo, hi, M1, lo, hi);
                m = min(M + 1, M1);
              }
            } else {
              Y->done[nr] = Y->done[pr];
            }
            L->clo[nr] = lo; L->chi[nr] = hi; L->clen[nr] = m;
          } else {
            unsigned long long lo = (L->clo[pr] << 16) | static_cast<unsigned long long>(lm_tok(la, c) + 1);
            unsigned long long hi = (L->chi[pr] << 16) | (L->clo[pr] >> 48);
            lm_ctx_prefix<16>(lo, hi, M1, lo, hi);
            L->clo[nr] = lo; L->chi[nr] = hi; L->clen[nr] = min(M + 1, M1);
          }
        }
        if constexpr (LM || LEX) {                            // after the LM's row state (keeps the LM kernels' code)
          L->nrow[q] = nr;
          L->row[cur ^ 1][lane] = nr;
        }
        if constexpr (LEX) {
          const int nn = lex_step(xa, X->node[L->row[cur][pi]], c);
          X->node[nr] = nn;
          X->fin[nr] = nn == 0 || __ldg(xa.word_end + nn);
        }
      }
    }
    nnodes += __popc(em);
    nb = nnew;
    cur ^= 1;
    if constexpr (LM || LEX) used = __reduce_or_sync(0xffffffffu, lane < nnew ? 1u << nr : 0u);
    if constexpr (LM && !WLM) {
      if (em) {
        __syncwarp();
        lm_fill_rows(la, L, rows, __popc(em), C, unk, lane);
      }
    }
    if constexpr (LEX) {
      if (em) {
        __syncwarp();
        if constexpr (WLM) wlm_fill_rows(la, wa, L, X, Y, rows, __popc(em), C, unk, lane);
        lex_fill_rows<CPL, WLM>(xa, L, X, __popc(em), C, lane, rows, Y->done, wa.smear, la.alpha);
      }
    }
#pragma unroll
    for (int u = 0; u < CPL; ++u) v[u] = vn[u];
    __syncwarp();
  }

  // ---- spell the surviving prefixes --------------------------------------------------------------------------
  // LM: the key gains the </s> term and the survivors are re-ranked by it, stably (ties keep beam rank)
  int slot = lane;
  double fused = 0.0;
  if constexpr (LM) {
    const PbGen& g = W->gen[cur];
    long long mk = LLONG_MIN;
    if (lane < nb) {
      const int r = L->row[cur][lane];
      if constexpr (WLM)                                  // (every survivor is between words or at a word end)
        fused = (g.tot[lane] + Y->done[r]) + L->eos[r];
      else
        fused = (g.tot[lane] + L->lm[r]) + L->eos[r];
      mk = pb_key(fused);
    }
    int rank = 0;
    for (int j = 0; j < nb; ++j) {
      const long long kj = __shfl_sync(0xffffffffu, mk, j);
      if (kj > mk || (kj == mk && j < lane)) ++rank;
    }
    if (lane < nb) slot = rank;
  }
  if (lane < K) {
    const PbGen& g = W->gen[cur];
    int* out = ids + (static_cast<long long>(b) * K + slot) * T;
    const bool live = lane < nb;
    int n = 0;
    if (live) {
      n = g.len[lane];
      int nd = g.node[lane];
      for (int p = n - 1; p >= 0; --p) {
        const uint32_t e = nodes[nd];
        out[p] = static_cast<int>(e & 0xFFFFu);
        nd = static_cast<int>(e >> 16);
      }
    }
    for (int p = n; p < T; ++p) out[p] = 0;
    lens[b * K + slot] = live ? n : -1;
    scores[b * K + slot] = live ? (LM ? fused : g.tot[lane]) : -INFINITY;
    if constexpr (LM || LEX) la.ctc_scores[b * K + slot] = live ? g.tot[lane] : -INFINITY;
  }
}

// Shared launcher: shared memory as pb_smem_layout; fewer warps per CTA above 200 KB.
template <bool LM, bool LEX, bool WLM>
static int pb_launch(const float* log_probs, long long stride_b, long long stride_t, const int* lengths, int B, int T,
                     int C, int K, int* ids, int* lens, double* scores, const PbLmArgs& la, const PbLexArgs& xa,
                     const PbWlmArgs& wa, cudaStream_t stream) {
  if (B <= 0 || T <= 0 || C <= 0 || !log_probs || !ids || !lens || !scores) return HTRVT_ERR_SHAPE;
  if (K < 1 || K > kPbMaxK || C > 32 * kPbCpl || static_cast<long long>(T) * K >= 65535) return HTRVT_ERR_SHAPE;
  int warps = 4;
  while (warps > 1 && pb_smem_layout(LM, LEX, WLM, K, C, T, warps).bytes > 200 * 1024) warps >>= 1;
  const size_t smem = pb_smem_layout(LM, LEX, WLM, K, C, T, warps).bytes;
  if (smem > 227 * 1024) return HTRVT_ERR_SHAPE;
  const dim3 grid((B + warps - 1) / warps), block(warps * 32);
#define PB_LAUNCH(CPL)                                                                                         \
  do {                                                                                                         \
    if (smem > 48 * 1024 && !HTRVT_ENSURE_SMEM((ctc_prefix_beam_kernel<CPL, LM, LEX, WLM>), 227 * 1024))      \
      return HTRVT_ERR_LAUNCH;                                                                                 \
    ctc_prefix_beam_kernel<CPL, LM, LEX, WLM><<<grid, block, smem, stream>>>(                                  \
        log_probs, stride_b, stride_t, lengths, B, T, C, K, ids, lens, scores, la, xa, wa);                   \
  } while (0)
  if (C <= 32) PB_LAUNCH(1);
  else if (C <= 64) PB_LAUNCH(2);
  else if (C <= 96) PB_LAUNCH(3);
  else if (C <= 128) PB_LAUNCH(4);
  else PB_LAUNCH(8);
#undef PB_LAUNCH
  HTRVT_LAUNCH_CHECK();
  return HTRVT_OK;
}

// The LM arguments of htrvt_ctc_prefix_beam_lm / _lex, checked
static int pb_lm_args(const void* lm_table, long long lm_slots, int lm_order, const int* tok_map, int n_tok_map,
                      double alpha, double beta, double* ctc_scores, PbLmArgs& la) {
  if (!lm_table || !ctc_scores || lm_slots < 2 || (lm_slots & (lm_slots - 1)) != 0) return HTRVT_ERR_SHAPE;
  if (lm_order < 1 || lm_order > kLmMaxOrder || n_tok_map < 0 || (n_tok_map > 0 && !tok_map)) return HTRVT_ERR_SHAPE;
  if (!isfinite(alpha) || !isfinite(beta)) return HTRVT_ERR_SHAPE;
  if ((reinterpret_cast<uintptr_t>(lm_table) & 31) != 0) return HTRVT_ERR_ALIGN;
  la.table = static_cast<const PbLmSlot*>(lm_table);
  la.mask = static_cast<unsigned long long>(lm_slots - 1);
  la.order = lm_order;
  la.tok_map = tok_map;
  la.n_map = n_tok_map;
  la.alpha = alpha;
  la.beta = beta;
  la.ctc_scores = ctc_scores;
  return HTRVT_OK;
}

// The trie arguments of htrvt_ctc_prefix_beam_lex / _lex_wlm, checked for presence
static int pb_trie_args(const int* first, const int* label, const int* child, const unsigned char* word_end,
                        int n_nodes, const unsigned char* is_word, int n_class_map, PbLexArgs& xa) {
  if (!first || !label || !child || !word_end || n_nodes < 1) return HTRVT_ERR_SHAPE;
  if (n_class_map < 0 || (n_class_map > 0 && !is_word)) return HTRVT_ERR_SHAPE;
  xa.first = first;
  xa.label = label;
  xa.child = child;
  xa.word_end = word_end;
  xa.is_word = is_word;
  xa.n_map = n_class_map;
  return HTRVT_OK;
}

}  // namespace htrvt

using namespace htrvt;

// ids int32 [B, K, T] (labels of the K most probable prefixes, zero padded), lens int32 [B, K] (-1: fewer than K
// prefixes exist), scores float64 [B, K] = log P(labelling's alignments over the line's frames), best first.
// log_probs fp32 through element strides (class axis contiguous).  K <= 16, C <= 256, T * K < 65535.
extern "C" int htrvt_ctc_prefix_beam(const float* log_probs, long long stride_b, long long stride_t,
                                     const int* lengths, int B, int T, int C, int K, int* ids, int* lens,
                                     double* scores, cudaStream_t stream) {
  return pb_launch<false, false, false>(log_probs, stride_b, stride_t, lengths, B, T, C, K, ids, lens, scores,
                                        PbLmArgs{}, PbLexArgs{}, PbWlmArgs{}, stream);
}

// The same search with a character n-gram LM fused into the ranking (header: include/htrvt.h).  lm_table: lm_slots
// (a power of two) PbLmSlot records with at least one empty slot; token ids <unk> = 0, <s> = 1, </s> = 2; tok_map:
// class id -> token id for ids < n_tok_map, <unk> beyond.  scores = fused score with the </s> term, ctc_scores =
// log P(labelling's alignments), both float64 [B, K], entries in fused order.
extern "C" int htrvt_ctc_prefix_beam_lm(const float* log_probs, long long stride_b, long long stride_t,
                                        const int* lengths, int B, int T, int C, int K, const void* lm_table,
                                        long long lm_slots, int lm_order, const int* tok_map, int n_tok_map,
                                        double alpha, double beta, int* ids, int* lens, double* scores,
                                        double* ctc_scores, cudaStream_t stream) {
  PbLmArgs la;
  const int st = pb_lm_args(lm_table, lm_slots, lm_order, tok_map, n_tok_map, alpha, beta, ctc_scores, la);
  if (st != HTRVT_OK) return st;
  return pb_launch<true, false, false>(log_probs, stride_b, stride_t, lengths, B, T, C, K, ids, lens, scores, la,
                                       PbLexArgs{}, PbWlmArgs{}, stream);
}

// The same search constrained to a word lexicon, with or without the LM (header: include/htrvt.h).  The trie (CSR,
// node 0 = root, edges sorted by label within a node, child ids < n_nodes) is the documented contract that
// htr-vt_b200/lexicon.py packs and checks; it is not re-validated here.  lm_table == nullptr: no LM, alpha = beta = 0.
extern "C" int htrvt_ctc_prefix_beam_lex(const float* log_probs, long long stride_b, long long stride_t,
                                         const int* lengths, int B, int T, int C, int K, const int* first,
                                         const int* label, const int* child, const unsigned char* word_end,
                                         int n_nodes, const unsigned char* is_word, int n_class_map,
                                         const void* lm_table, long long lm_slots, int lm_order, const int* tok_map,
                                         int n_tok_map, double alpha, double beta, int* ids, int* lens,
                                         double* scores, double* ctc_scores, cudaStream_t stream) {
  PbLexArgs xa;
  const int sx = pb_trie_args(first, label, child, word_end, n_nodes, is_word, n_class_map, xa);
  if (sx != HTRVT_OK || !ctc_scores) return HTRVT_ERR_SHAPE;
  if (!lm_table) {
    if (alpha != 0.0 || beta != 0.0) return HTRVT_ERR_SHAPE;
    PbLmArgs la{};
    la.ctc_scores = ctc_scores;
    return pb_launch<false, true, false>(log_probs, stride_b, stride_t, lengths, B, T, C, K, ids, lens, scores, la,
                                         xa, PbWlmArgs{}, stream);
  }
  PbLmArgs la;
  const int st = pb_lm_args(lm_table, lm_slots, lm_order, tok_map, n_tok_map, alpha, beta, ctc_scores, la);
  if (st != HTRVT_OK) return st;
  return pb_launch<true, true, false>(log_probs, stride_b, stride_t, lengths, B, T, C, K, ids, lens, scores, la, xa,
                                      PbWlmArgs{}, stream);
}

// The lexicon-constrained search with a word n-gram LM (header: include/htrvt.h).  Trie as htrvt_ctc_prefix_beam_lex;
// lm_table as htrvt_ctc_prefix_beam_lm with 21-bit key fields (htr-vt_b200/wordlm.py packs it), lm_order 1..6;
// node_tok int32 / smear float32 [n_nodes], not re-validated here.
extern "C" int htrvt_ctc_prefix_beam_lex_wlm(const float* log_probs, long long stride_b, long long stride_t,
                                             const int* lengths, int B, int T, int C, int K, const int* first,
                                             const int* label, const int* child, const unsigned char* word_end,
                                             int n_nodes, const unsigned char* is_word, int n_class_map,
                                             const void* lm_table, long long lm_slots, int lm_order,
                                             const int* node_tok, const float* smear, double alpha, double beta,
                                             int* ids, int* lens, double* scores, double* ctc_scores,
                                             cudaStream_t stream) {
  PbLexArgs xa;
  if (pb_trie_args(first, label, child, word_end, n_nodes, is_word, n_class_map, xa) != HTRVT_OK)
    return HTRVT_ERR_SHAPE;
  if (!node_tok || !smear || lm_order > kWlmMaxOrder) return HTRVT_ERR_SHAPE;
  PbWlmArgs wa;
  wa.node_tok = node_tok;
  wa.smear = smear;
  PbLmArgs la;
  const int st = pb_lm_args(lm_table, lm_slots, lm_order, nullptr, 0, alpha, beta, ctc_scores, la);
  if (st != HTRVT_OK) return st;
  return pb_launch<true, true, true>(log_probs, stride_b, stride_t, lengths, B, T, C, K, ids, lens, scores, la, xa, wa,
                                     stream);
}
