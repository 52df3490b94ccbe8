// TEST-ONLY backend: executes the constraint netlist (gatekeeper_b200/csrc/program.h GkOp) on the CPU with the
// whole batch as one tile, using the same per-row core (csrc/vm_core.h: gk_atom, gk_match) as the CUDA tile
// executor, so the lowering + flattening logic can be unit-tested in the authoring container (no GPU).
// It is linked ONLY into tests/_hostemu/libgk_hostemu.so.  The product library
// (gatekeeper_b200/libgk_engine.so) links kernels.cu instead and has no CPU path at all.
#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <memory>
#include <mutex>

#include "../../gatekeeper_b200/csrc/backend.hpp"
#include "../../gatekeeper_b200/csrc/vm_core.h"
#include "../../gatekeeper_b200/csrc/ingest_core.h"
#include "../../gatekeeper_b200/csrc/spec_codegen.hpp"

#include <dlfcn.h>
#include <unistd.h>

#include <fstream>
#include <functional>
#include <map>

namespace gk {

struct EmuBatch {
  PackedBatch pb;
  GkBatch hdr{};
  uint32_t n = 0, words = 1;
  bool gvk_uniform = false;
  std::vector<uint32_t> scope_rows;
  std::vector<std::vector<uint32_t>> scope_off;   // host copies for range lookups
};

class HostEmuBackend : public Backend {
 public:
  const char* name() const override { return "hostemu-TEST-ONLY"; }
  void set_program(const Compiled& c) override {
    std::lock_guard<std::mutex> l(mu_);
    prog_ = &c;
  }
  // the dictionary is replaced, never edited in place: an evaluation keeps the copy it started with
  void sync_strings(const StringTable& st) override {
    auto d = std::make_shared<Dict>();
    st.snapshot(d->off, d->bytes);
    std::lock_guard<std::mutex> l(mu_);
    dict_ = std::move(d);
  }
  void* upload(const HostBatch& hb, const Compiled& c, double* ms, uint64_t* bytes) override {
    auto* b = new EmuBatch();
    pack_batch(hb, c, b->pb);
    b->hdr = rebase_batch(b->pb, b->pb.arena.data(), b->pb.arena.data());
    b->n = hb.n;
    b->words = std::max<uint32_t>(1, (uint32_t)((c.cons_match.size() + 31) / 32));
    b->scope_rows = hb.scope_rows;
    b->scope_off = hb.scope_off;
    b->gvk_uniform = hb.gvk_hi == 0 || hb.gvk_lo == hb.gvk_hi;
    if (ms) *ms = 0;
    if (bytes) *bytes = b->pb.arena.size();
    return b;
  }
  void release(void* b) override { delete static_cast<EmuBatch*>(b); }
  void* fork_batch(void* bb, const Compiled& other) override {
    auto* b = static_cast<EmuBatch*>(bb);
    auto* f = new EmuBatch();
    f->hdr = b->hdr;   // (points into the parent's arena: the fork is released first)
    f->n = b->n;
    f->words = std::max<uint32_t>(1, (uint32_t)((other.cons_match.size() + 31) / 32));
    f->gvk_uniform = b->gvk_uniform;
    f->scope_rows = b->scope_rows;
    f->scope_off = b->scope_off;
    return f;
  }
  void identity(void* bb, BatchIdentity& out) override {
    auto* b = static_cast<EmuBatch*>(bb);
    const uint32_t n = b->n;
    out.uniform_gvk = b->gvk_uniform;
    out.flags.assign(b->hdr.flags, b->hdr.flags + n);
    out.ns_off.assign(b->hdr.nsn_off, b->hdr.nsn_off + n + 1);
    out.name_off.assign(b->hdr.name_off, b->hdr.name_off + n + 1);
    out.ns_bytes.assign(b->hdr.nsn_bytes, b->hdr.nsn_bytes + out.ns_off[n]);
    out.name_bytes.assign(b->hdr.name_bytes, b->hdr.name_bytes + out.name_off[n]);
  }

  // The device ingest path, run by CPU loops over the SAME per-object code the CUDA kernels run (ingest_core.h): tokenise,
  // count, scan, write (+ host-filled lookups), then the arrays are handed to upload() like a host-flattened batch.
  void* ingest(const IngestReq& rq, IngestStats* st, std::vector<uint32_t>* status) override {
    std::lock_guard<std::mutex> l(ingest_mu_);
    const XProgHost& xh = *rq.xprog;
    const uint32_t n = (uint32_t)rq.n, NS = (uint32_t)xh.scopes.size(), NK = xh.ncounters(), NC = (uint32_t)xh.cols.size();
    if (sid_.nstrings != rq.strings->size()) build_sid_table(*rq.strings, sid_);
    if (lut_.mask == 0) lut_.init(1u << 12);
    // excluder patterns ride in xkeys / xbytes copies
    std::vector<uint32_t> xkeys = xh.xkeys;
    std::vector<uint8_t> xbytes = xh.xbytes;
    GkXProg xp{};
    xp.excl_off = (uint32_t)xkeys.size();
    for (auto& pat : rq.excluded) {
      bool pre = !pat.empty() && pat.front() == '*', suf = pat.size() > (pre ? 1u : 0u) && pat.back() == '*';
      std::string core = pat.substr(pre ? 1 : 0, pat.size() - (pre ? 1 : 0) - (suf ? 1 : 0));
      xkeys.push_back(pre && suf ? GK_W_CONTAINS : pre ? GK_W_SUFFIX : suf ? GK_W_PREFIX : GK_W_EXACT);
      xkeys.push_back((uint32_t)xbytes.size());
      xkeys.push_back((uint32_t)core.size());
      xbytes.insert(xbytes.end(), core.begin(), core.end());
      ++xp.excl_n;
    }
    xbytes.push_back(0);
    NsTableHost ns = *rq.ns;
    xp.cl = xh.cl.data();
    xp.cols = xh.cols.data();
    xp.scopes = xh.scopes.data();
    xp.col_order = xh.col_order.data();
    xp.xkeys = xkeys.data();
    xp.xargs = xh.xargs.data();
    xp.xbytes = xbytes.data();
    xp.ncl = (uint32_t)xh.cl.size();
    xp.ncols = NC;
    xp.nscopes = NS;
    xp.nbytecols = xh.nbytecols;
    xp.sid_tab = sid_.tab.view();
    xp.sid_true = sid_.sid_true;
    xp.sid_false = sid_.sid_false;
    xp.sid_null = sid_.sid_null;
    xp.ns_tab = ns.tab.view();
    ns.nsn_bytes.push_back(0);
    xp.nsn_off = ns.nsn_off.data();
    xp.nsn_bytes = ns.nsn_bytes.data();
    // ---- tokenise
    std::vector<unsigned long long> tape((size_t)(rq.ooff[n] / 2 + 4ull * n + 16));
    std::vector<uint32_t> ntape(std::max(n, 1u)), stat(std::max(n, 1u)), counts((size_t)NK * std::max(n, 1u)), nmiss(1, 0);
    std::vector<GkMiss> misses(1u << 16);
    GkIngestIn in{};
    in.blob = rq.blob;
    in.ooff = rq.ooff;
    in.tape = tape.data();
    in.ntape = ntape.data();
    in.status = stat.data();
    in.n = n;
    in.source = rq.source;
    in.counts = counts.data();
    in.misses = misses.data();
    in.nmiss = nmiss.data();
    in.miss_cap = (uint32_t)misses.size();
    for (uint32_t i = 0; i < n; ++i) gk_tape_obj(in, i);
    if (status) status->assign(stat.begin(), stat.begin() + n);
    // ---- header counts + scan, then the scopes level by level (the same per-row steps the CUDA kernels run, in plain loops)
    std::vector<uint32_t> cur(GK_CNT_EXTRA);
    counts.assign((size_t)GK_CNT_EXTRA * std::max(n, 1u), 0);
    in.counts = counts.data();
    std::vector<uint32_t> flags_tmp(std::max(n, 1u), 0);
    GkIngestOut outc{};
    outc.flags = flags_tmp.data();
    xp.lut_tab = lut_.view();
    xp.lut_vals = lut_vals_.data();
    for (uint32_t i = 0; i < n; ++i) gk_ingest_obj<GK_PASS_COUNT>(xp, in, outc, i, GkCur{cur.data(), 1}, 0, 1);
    auto scan = [](uint32_t* a2, size_t len) {   // exclusive, in place; returns the total
      uint32_t acc = 0;
      for (size_t i = 0; i < len; ++i) {
        const uint32_t v = a2[i];
        a2[i] = acc;
        acc += v;
      }
      return acc;
    };
    std::vector<uint32_t> htot(GK_CNT_EXTRA, 0);
    for (uint32_t k = 0; k < GK_CNT_EXTRA; ++k) htot[k] = scan(counts.data() + (size_t)k * n, n);
    std::vector<uint32_t> total(NS, 0);
    total[0] = n;
    std::vector<std::vector<uint32_t>> cnt(NS), coll(NS);
    std::vector<std::vector<GkRowRec>> rh(NS);
    std::vector<GkRowRec*> p_rh(NS, nullptr);
    outc.row_rec = p_rh.data();
    for (uint32_t t = 1; t < NS; ++t) {   // (scopes are numbered parents first)
      const uint32_t prows = total[xh.scopes[t].parent];
      cnt[t].assign((size_t)prows + 1, 0);
      coll[t].assign((size_t)prows + 1, GK_NONE);
      for (uint32_t r = 0; r < prows; ++r) cnt[t][r] = gk_scope_count(xp, in, outc, t, r, &coll[t][r]);
      total[t] = scan(cnt[t].data(), prows);
      cnt[t][prows] = total[t];
      rh[t].assign((size_t)total[t] + 1, GkRowRec{0, 0, 0, 0});
      p_rh[t] = rh[t].data();
      for (uint32_t r = 0; r < prows; ++r) gk_scope_fill(xp, in, outc, t, r, coll[t][r], cnt[t][r]);
    }
    std::vector<std::vector<uint32_t>> blen(xh.nbytecols);
    std::vector<uint32_t> btot(xh.nbytecols, 0);
    for (uint32_t ci = 0; ci < NC; ++ci) {
      const GkXCol& xc = xh.cols[ci];
      if (!(xc.enc & GK_ENC_BYTES)) continue;
      const uint32_t rows = total[xc.scope];
      auto& bl = blen[xc.bytes_slot];
      bl.assign((size_t)rows + 1, 0);
      for (uint32_t r = 0; r < rows; ++r) bl[r] = gk_bcol_len(xp, in, outc, ci, r);
      btot[xc.bytes_slot] = scan(bl.data(), rows);
      bl[rows] = btot[xc.bytes_slot];
    }
    // ---- destination arrays (a HostBatch) and the write pass
    HostBatch hb;
    hb.n = n;
    hb.schema_version = rq.c->version;
    hb.flags.assign(n, 0), hb.kind_sid.assign(n, 0), hb.group_sid.assign(n, 0), hb.nsrow.assign(n, GK_NONE);
    hb.name_off.assign(n + 1, 0), hb.gen_off.assign(n + 1, 0), hb.lbl_off.assign(n + 1, 0), hb.nsn_off.assign(n + 1, 0);
    hb.name_bytes.assign(htot[0], 0), hb.gen_bytes.assign(htot[1], 0), hb.lbl_kv.assign(2 * (size_t)htot[2], 0);
    hb.nsn_bytes.assign(htot[3], 0);
    hb.nsl_off = rq.ns->nsl_off;
    hb.nsl_kv = rq.ns->nsl_kv;
    hb.scope_off.resize(NS);
    hb.scope_rows.assign(NS, 0);
    std::vector<uint32_t*> p_scope(NS, nullptr);
    for (uint32_t s2 = 1; s2 < NS; ++s2) {
      hb.scope_rows[s2] = total[s2];
      hb.scope_off[s2] = cnt[s2];   // the CSR offsets are the scanned member counts
      p_scope[s2] = hb.scope_off[s2].data();
    }
    hb.cols.resize(NC);
    std::vector<uint8_t*> p_vt(NC, nullptr), p_bytes(NC, nullptr);
    std::vector<uint32_t*> p_sid(NC, nullptr), p_boff(NC, nullptr), p_head(NC, nullptr);
    std::vector<long long*> p_num(NC, nullptr);
    for (uint32_t ci = 0; ci < NC; ++ci) {
      const GkXCol& xc = xh.cols[ci];
      const size_t rows = total[xc.scope];
      HostColumn& hc = hb.cols[ci];
      if (xc.enc & GK_ENC_VT) hc.vt.assign(rows, 0), p_vt[ci] = hc.vt.data();
      if (xc.enc & GK_ENC_SID) hc.sid.assign(rows, 0), p_sid[ci] = hc.sid.data();
      if (xc.enc & GK_ENC_NUM) hc.num.assign(rows, 0), p_num[ci] = reinterpret_cast<long long*>(hc.num.data());
      if (xc.enc & GK_ENC_HEAD) hc.head.assign(rows * GK_HEAD_WORDS, 0), p_head[ci] = hc.head.data();
      if (xc.enc & GK_ENC_BYTES) {
        hc.boff = blen[xc.bytes_slot], p_boff[ci] = hc.boff.data();
        hc.bytes.assign((size_t)btot[xc.bytes_slot] + 1, 0), p_bytes[ci] = hc.bytes.data();
      }
    }
    hb.name_bytes.push_back(0), hb.gen_bytes.push_back(0), hb.nsn_bytes.push_back(0), hb.lbl_kv.push_back(0);
    GkIngestOut out{};
    out.flags = hb.flags.data();
    out.kind_sid = hb.kind_sid.data();
    out.group_sid = hb.group_sid.data();
    out.name_off = hb.name_off.data();
    out.name_bytes = hb.name_bytes.data();
    out.gen_off = hb.gen_off.data();
    out.gen_bytes = hb.gen_bytes.data();
    out.lbl_off = hb.lbl_off.data();
    out.lbl_kv = hb.lbl_kv.data();
    out.nsrow = hb.nsrow.data();
    out.nsn_off = hb.nsn_off.data();
    out.nsn_bytes = hb.nsn_bytes.data();
    out.scope_off = p_scope.data();
    out.vt = p_vt.data();
    out.sid = p_sid.data();
    out.num = p_num.data();
    out.boff = p_boff.data();
    out.bytes = p_bytes.data();
    out.head = p_head.data();
    out.row_rec = p_rh.data();
    std::vector<unsigned long long> gvk(std::max(n, 1u), 0);
    out.gvk = gvk.data();
    uint64_t total_miss = 0;
    for (int round = 0; round < 64; ++round) {
      nmiss[0] = 0;
      xp.lut_tab = lut_.view();
      xp.lut_vals = lut_vals_.data();
      for (uint32_t i = 0; i < n; ++i) gk_ingest_obj<GK_PASS_HEADER>(xp, in, out, i, GkCur{cur.data(), 1}, 0, 1);
      for (uint32_t ci = 0; ci < NC; ++ci)
        if (xh.cols[ci].enc & GK_ENC_BYTES)
          for (uint32_t r = 0, R = total[xh.cols[ci].scope]; r < R; ++r) gk_bcol_write(xp, in, out, ci, r);
      for (uint32_t s2 = 0; s2 < NS; ++s2)
        for (uint32_t r = 0, R = total[s2]; r < R; ++r) gk_ingest_row(xp, in, out, s2, r, 0, 1);
      const uint32_t m = std::min<uint32_t>(nmiss[0], in.miss_cap);
      if (nmiss[0] == 0) break;
      total_miss += m;
      std::vector<GkLutVal> vals;
      rq.lut_fill(misses.data(), m, vals);
      for (uint32_t j = 0; j < m; ++j) {
        lut_.vals[misses[j].slot] = (uint32_t)lut_vals_.size();
        lut_vals_.push_back(vals[j]);
      }
      lut_.used += m;
      if (lut_.used * 2 > lut_.mask) {   // grow: re-insert the filled entries, drop the pending ones
        HashTabHost big;
        big.init((lut_.mask + 1) * 4);
        for (uint32_t i2 = 0; i2 <= lut_.mask; ++i2)
          if (lut_.keys[i2] && lut_.vals[i2] < GK_HT_LOST) big.put(lut_.keys[i2], lut_.vals[i2]);
        lut_ = std::move(big);
      }
      if (round == 63) throw BackendError{"device ingest: lookups did not converge"};
    }
    hb.name_bytes.pop_back(), hb.gen_bytes.pop_back(), hb.nsn_bytes.pop_back(), hb.lbl_kv.pop_back();
    for (uint32_t ci = 0; ci < NC; ++ci)
      if (xh.cols[ci].enc & GK_ENC_BYTES) hb.cols[ci].bytes.pop_back();
    hb.obj_errors.assign(n, std::string());
    uint64_t b = 0;
    auto sz = [&](auto& v) { b += (uint64_t)v.size() * sizeof(v[0]); };
    sz(hb.flags), sz(hb.kind_sid), sz(hb.group_sid), sz(hb.nsn_off), sz(hb.nsn_bytes), sz(hb.name_off), sz(hb.gen_off), sz(hb.lbl_off), sz(hb.lbl_kv);
    sz(hb.name_bytes), sz(hb.gen_bytes), sz(hb.nsrow), sz(hb.nsl_off), sz(hb.nsl_kv);
    for (uint32_t s2 = 1; s2 < NS; ++s2) sz(hb.scope_off[s2]);
    for (auto& col : hb.cols) sz(col.vt), sz(col.sid), sz(col.num), sz(col.boff), sz(col.bytes), sz(col.head);
    hb.alg_bytes = b;
    if (st) {
      st->lut_misses = total_miss;
      st->alg_bytes = b;
    }
    if (getenv("GK_TRACE_INGEST")) fprintf(stderr, "[ingest hostemu] n=%u lookups missed (host-evaluated) %llu, table entries %u\n", n, (unsigned long long)total_miss, lut_.used);
    for (uint32_t i = 0; i < n; ++i)
      if (gvk[i]) hb.gvk_lo = std::min<uint64_t>(hb.gvk_lo, gvk[i]), hb.gvk_hi = std::max<uint64_t>(hb.gvk_hi, gvk[i]);
    last_ingest_ = hb;   // (tests compare these arrays with the host flattener's)
    return upload(hb, *rq.c, nullptr, nullptr);
  }
  const HostBatch& last_ingest() const { return last_ingest_; }

  void eval(void* bb, const std::vector<uint32_t>& active, EvalOut& out, bool) override {
    auto* b = static_cast<EmuBatch*>(bb);
    std::shared_ptr<const Dict> dict;
    const Compiled* progp;
    {
      std::lock_guard<std::mutex> l(mu_);
      dict = dict_;
      progp = prog_;
    }
    const Compiled& c = *progp;
    const uint32_t C = (uint32_t)c.cons_match.size(), W = b->words, n = b->n;
    GkBatch h = b->hdr;
    if (dict) {
      h.dict_off = dict->off.data();
      h.dict_bytes = dict->bytes.data();
      h.dict_n = (uint32_t)dict->off.size() - 1;
    }
    out.n = n;
    out.nconstraints = C;
    out.words = W;
    out.viol.assign((size_t)n * W, 0);
    out.err.assign((size_t)n * W, 0);
    out.totals.assign(C, 0);
    out.err_totals.assign(C, 0);
    out.errlist.clear();
    auto t0 = std::chrono::steady_clock::now();
    auto rows_of = [&](uint32_t level) -> uint32_t { return level == 0 ? n : b->scope_rows[level]; };
    std::vector<std::vector<uint8_t>> slot(c.slot_level.size());
    for (size_t s = 0; s < slot.size(); ++s) slot[s].assign(rows_of(c.slot_level[s]), 0);
    for (const GkOp& op : c.ops) {
      const uint32_t kind = op.w0 & 0xffu, level = (op.w0 >> 8) & 0xffu, o = op.w0 >> 16;
      if (kind == GK_N_END) break;
      if (kind == GK_N_PHASE) continue;
      switch (kind) {
        case GK_N_CONST:
          std::fill(slot[o].begin(), slot[o].end(), (uint8_t)(op.w1 & 1));
          break;
        case GK_N_ATOM: {
          const GkColumn& col = h.cols[op.w1 >> 8];
          const uint32_t aop = op.w1 & 0xffu, R = rows_of(level);
          for (uint32_t r = 0; r < R; ++r) slot[o][r] = gk_atom(col, r, aop, op.w2, op.w3, c.pool.data(), c.cbytes.data());
          break;
        }
        case GK_N_ATOMS: {
          const GkColumn& col = h.cols[op.w1 >> 8];
          const uint32_t R = rows_of(level);
          for (uint32_t j = 0; j < op.w3; ++j) {
            const uint32_t* e = &c.pool[op.w2 + j * GK_ATOMS_ENT];
            auto& dst = slot[e[0] >> 16];
            for (uint32_t r = 0; r < R; ++r) dst[r] = gk_atom(col, r, e[0] & 0xffu, e[1], e[2], c.pool.data(), c.cbytes.data());
          }
          break;
        }
        case GK_N_GATE: {
          const uint32_t f = op.w2, R = rows_of(level);
          for (uint32_t r = 0; r < R; ++r) {
            bool v = !(f & GK_G_OR);
            for (uint32_t j = 0; j < op.w3; ++j) {
              const uint32_t e = c.pool[op.w1 + j];
              bool x = slot[e & 0xffffu][r] ^ ((e >> 31) != 0);
              v = (f & GK_G_OR) ? (v || x) : (v && x);
            }
            slot[o][r] = v ^ ((f & GK_G_NEG_OUT) != 0);
          }
          break;
        }
        case GK_N_BCAST: {
          const auto& off = b->scope_off[level];
          for (uint32_t j = 0; j < op.w3; ++j) {
            const uint32_t e = c.pool[op.w1 + j];
            const auto& in = slot[e & 0xffffu];
            auto& dst = slot[e >> 16];
            for (size_t p = 0; p + 1 < off.size(); ++p)
              for (uint32_t r = off[p]; r < off[p + 1]; ++r) dst[r] = in[p];
          }
          break;
        }
        case GK_N_ACC2:
        case GK_N_ACC: {
          const auto& off = b->scope_off[level];
          const uint32_t need = kind == GK_N_ACC2 ? 2u : 1u;
          for (uint32_t j = 0; j < op.w3; ++j) {
            const uint32_t e = c.pool[op.w1 + j];
            const auto& in = slot[e & 0xffffu];
            auto& dst = slot[e >> 16];
            for (size_t p = 0; p + 1 < off.size(); ++p) {
              uint32_t cnt = 0;
              for (uint32_t r = off[p]; r < off[p + 1]; ++r) cnt += in[r] ? 1u : 0u;
              dst[p] = cnt >= need;
            }
          }
          break;
        }
        case GK_N_MATCH: {
          auto& err = slot[op.w1 & 0xffffu];
          for (uint32_t obj = 0; obj < n; ++obj) {
            int m = (h.flags[obj] & GK_F_SKIP) ? 0 : gk_match(h, c.pool.data(), c.cbytes.data(), c.match[op.w2], obj);
            slot[o][obj] = m > 0;
            err[obj] = m < 0;
            if (m < 0) {
              out.errlist.push_back(obj);
              out.errlist.push_back(op.w2);
              out.errlist.push_back((uint32_t)-m);
            }
          }
          break;
        }
        default: throw BackendError{"hostemu: unknown netlist op"};
      }
    }
    for (uint32_t cix = 0; cix < C; ++cix) {
      if (!active[cix]) continue;
      const GkOutEnt& oe = c.outs[cix];
      const auto &prog = slot[oe.prog_slot], &mt = slot[oe.match_slot], &er = slot[oe.err_slot];
      for (uint32_t obj = 0; obj < n; ++obj) {
        bool pv = (oe.flags & 1) ? true : (oe.flags & 2) ? false : prog[obj] != 0;
        if (pv && mt[obj]) {
          out.viol[(size_t)obj * W + cix / 32] |= 1u << (cix & 31);
          out.totals[cix]++;
        }
        if (er[obj]) {
          out.err[(size_t)obj * W + cix / 32] |= 1u << (cix & 31);
          out.err_totals[cix]++;
        }
      }
    }
    out.kernel_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    out.launches = 0;
    if (getenv("GK_SPEC_CHECK") || getenv("GK_SPEC_DUMP")) spec_check(c, h, active, out);
  }

  // GK_SPEC_CHECK=1: the text spec_codegen.cpp writes for this constraint set (what NVRTC compiles into gk_spec_kernel on the GPU)
  // is compiled for the host with g++ and must give, object by object, the words the interpreted netlist gave above.
  // GK_SPEC_DUMP=<path> writes the text out.
  typedef int (*SpecHostFn)(const GkKParams*, uint32_t, uint32_t*, uint32_t*);
  static SpecHostFn spec_host_fn(const std::string& src) {
    static std::mutex mu;
    static std::map<size_t, SpecHostFn> cache;
    std::lock_guard<std::mutex> l(mu);
    const size_t hv = std::hash<std::string>{}(src);
    auto it = cache.find(hv);
    if (it != cache.end()) return it->second;
    // compiled in a directory of its own (mkdtemp: a new name, mode 0700), so that only a library this process built is loaded; the
    // files are removed once loaded (the mapping outlives them), and kept only when the compile fails, for its log
    const char* td = getenv("TMPDIR");
    std::string dir = std::string(td && *td ? td : "/tmp") + "/gk_spec_host_XXXXXX";
    if (!mkdtemp(&dir[0])) throw BackendError{"GK_SPEC_CHECK: cannot create a directory under " + dir.substr(0, dir.rfind('/'))};
    const std::string cpp = dir + "/spec.cpp", so = dir + "/spec.so", log = dir + "/spec.log";
    {
      std::ofstream f(cpp);
      f << src;
    }
    const std::string cmd = "g++ -std=c++17 -O1 -w -shared -fPIC -DGK_SPEC_HOST -x c++ '" + cpp + "' -o '" + so + "' 2> '" + log + "'";
    if (system(cmd.c_str()) != 0) throw BackendError{"GK_SPEC_CHECK: the generated source does not compile for the host: see " + log};
    void* hnd = dlopen(so.c_str(), RTLD_NOW | RTLD_LOCAL);
    const std::string dl_err = hnd ? "" : dlerror();
    for (const std::string& f : {so, cpp, log}) unlink(f.c_str());
    rmdir(dir.c_str());
    if (!hnd) throw BackendError{"GK_SPEC_CHECK: dlopen: " + dl_err};
    auto fn = reinterpret_cast<SpecHostFn>(dlsym(hnd, "gk_spec_host"));
    if (!fn) throw BackendError{"GK_SPEC_CHECK: gk_spec_host missing"};
    cache[hv] = fn;
    return fn;
  }
  static void spec_check(const Compiled& c, const GkBatch& h, const std::vector<uint32_t>& active, const EvalOut& out) {
    const SpecSource ss = spec_codegen(c);
    if (const char* d = getenv("GK_SPEC_DUMP")) {
      std::ofstream f(d);
      f << ss.src;
    }
    if (!getenv("GK_SPEC_CHECK")) return;
    SpecHostFn fn = spec_host_fn(ss.src);
    const uint32_t W = out.words, n = out.n;
    if (ss.words != W) throw BackendError{"GK_SPEC_CHECK: word count differs"};
    GkKParams p{};
    p.batch = h;
    p.prog.pool = c.pool.data();
    p.prog.cbytes = c.cbytes.data();
    p.active = active.data();
    std::vector<uint32_t> errlist((size_t)3 * (64 + (size_t)n * std::max<size_t>(1, c.match.size())));
    uint32_t errcount = 0;
    p.out.errlist = errlist.data();
    p.out.errcount = &errcount;
    p.out.errcap = (uint32_t)(errlist.size() / 3);
    std::vector<uint32_t> vw(W), ew(W);
    std::vector<uint8_t> big(std::max(n, 1u), 0);
    size_t nbig = 0;
    for (uint32_t obj = 0; obj < n; ++obj) {
      if (fn(&p, obj, vw.data(), ew.data())) {
        big[obj] = 1;
        ++nbig;
        continue;
      }
      for (uint32_t w = 0; w < W; ++w)
        if (vw[w] != out.viol[(size_t)obj * W + w] || ew[w] != out.err[(size_t)obj * W + w])
          throw BackendError{"GK_SPEC_CHECK: object " + std::to_string(obj) + " word " + std::to_string(w) + ": generated code " + std::to_string(vw[w]) + "/" +
                             std::to_string(ew[w]) + ", interpreter " + std::to_string(out.viol[(size_t)obj * W + w]) + "/" + std::to_string(out.err[(size_t)obj * W + w])};
    }
    // the matcher-error list, as a set
    std::vector<std::array<uint32_t, 3>> a, b;
    for (uint32_t i = 0; i < errcount; ++i)
      if (!big[errlist[3 * i]]) a.push_back({errlist[3 * i], errlist[3 * i + 1], errlist[3 * i + 2]});   // (a too-big object's are listed again by the interpreter)
    for (size_t i = 0; i + 2 < out.errlist.size(); i += 3)
      if (!big[out.errlist[i]]) b.push_back({out.errlist[i], out.errlist[i + 1], out.errlist[i + 2]});
    std::sort(a.begin(), a.end());
    std::sort(b.begin(), b.end());
    if (a != b) throw BackendError{"GK_SPEC_CHECK: matcher error lists differ (" + std::to_string(a.size()) + " vs " + std::to_string(b.size()) + ")"};
    if (getenv("GK_SPEC_TRACE"))
      fprintf(stderr, "[spec check] %u objects identical (%zu too big for the mask registers), %zu atoms as immediates, %zu generic\n", n, nbig, ss.n_fast, ss.n_generic);
  }
  // "device" buffers are host memory here: the same address arithmetic as the CUDA backend (bitmap shard and totals of this
  // rank stored into every peer's receive buffer), so the C ABI's peer addressing can be tested without GPUs
  void eval_into(void* b, const std::vector<uint32_t>& active, const DevOutPtrs& dst) override {
    EvalOut out;
    eval(b, active, out, true);
    const size_t nw = out.viol.size();
    if (dst.err && nw) memcpy(dst.err, out.err.data(), nw * 4);
    if (dst.totals) memcpy(dst.totals, out.totals.data(), out.totals.size() * 8);
    if (dst.err_totals) memcpy(dst.err_totals, out.err_totals.data(), out.err_totals.size() * 8);
    if (dst.npeers == 0) {
      if (dst.viol && nw) memcpy(dst.viol, out.viol.data(), nw * 4);
      return;
    }
    for (uint32_t q = 0; q < dst.npeers; ++q) {
      if (nw) memcpy(reinterpret_cast<void*>(dst.peer_viol[q]), out.viol.data(), nw * 4);
      auto* t = reinterpret_cast<unsigned long long*>(dst.peer_tot[q]);
      for (size_t c = 0; c < out.totals.size(); ++c) {
        t[c] = out.totals[c];
        t[dst.tot_stride + c] = out.err_totals[c];
      }
    }
  }

 private:
  struct Dict {
    std::vector<uint32_t> off;
    std::vector<uint8_t> bytes;
  };
  std::mutex mu_, ingest_mu_;
  SidTable sid_;
  HashTabHost lut_;
  std::vector<GkLutVal> lut_vals_;
  HostBatch last_ingest_;
  const Compiled* prog_ = nullptr;
  std::shared_ptr<const Dict> dict_;
};

Backend* make_backend(int) { return new HostEmuBackend(); }

}  // namespace gk
