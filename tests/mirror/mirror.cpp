// mirror.cpp -- TEST INFRASTRUCTURE.  Strings the __host__ __device__ format logic of
// phyngsc_b200/csrc/phy_core.cuh together serially on the CPU so that tokeniser, classification, Huffman,
// header layout, walkers and bit sinks can be checked against the oracle without a GPU.  It is not a
// fallback: nothing in the product links or loads it.
#include <stddef.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../phyngsc_b200/csrc/phy_core.cuh"
#include "../../phyngsc_b200/csrc/phy_fast.cuh"

using namespace phy;

static void amax(u32 &a, u32 v) { if (v > a) a = v; }


// ---- single-walk encoder, emulated serially (one "warp" = 32 lanes run one after the other) ------------------------
struct HostStream {
  StreamState st; std::vector<u32> cc; u32 *slot; u32 slot_words; bool over;
  void init(u32 *slot_, u32 words) { st.init(); cc.assign(4096, 0); slot = slot_; slot_words = words; over = false; }
  void flush(u32 bits) {
    u32 nf = st.full_words(bits);
    if (st.tpos + nf + 1 > slot_words) over = true; else for (u32 j = 0; j < nf; ++j) slot[st.tpos + j] = cc[j];
    u32 rem = cc[nf];
    for (u32 j = 0; j <= nf; ++j) cc[j] = 0;
    cc[0] = rem;
    st.advance(bits);
  }
  // pieces of the 32 lanes: lp[lane * lpw ...], nbits[lane]
  void append(const u32 *lp, u32 lpw, const u32 *nbits) {
    u32 excl = 0;
    for (u32 l = 0; l < 32; ++l) { if (nbits[l]) lane_concat(cc.data(), st.carry + excl, lp + l * lpw, 1u, nbits[l]); excl += nbits[l]; }
    flush(excl);
  }
  void pad_to_byte() { u32 p = st.pad_to_byte(); if (p) flush(p); }
  u32 finish() { if (st.carry && st.tpos < slot_words) slot[st.tpos] = cc[0]; return st.total; }
};

static int fast_encode(const u8 *b, const u8 *lut, const std::vector<u32> &te, const std::vector<u32> &se, const std::vector<u32> &rstart,
                       const std::vector<u16> &kx, const std::vector<u32> &vals, u32 nf, u32 *arena, u32 AW, SbClass *C, u32 G, u8 *out, u32 out_cap) {
  (void)AW;
  const u32 R = C->R;
  TableDesc *td = (TableDesc *)(arena + C->tabdesc_off);
  // k_slots
  u32 qsum = 0, qmax = 0;
  for (u32 p = 1; p <= C->max_qlen; ++p) { qsum += td[C->tq0 + p].maxlen; if (td[C->tq0 + p].maxlen > qmax) qmax = td[C->tq0 + p].maxlen; }
  const u32 tb = title_bound_part(*C, arena, td, 0u, 1u);
  const u32 seg_max = seg_len(C->max_qlen, G), dper = C->plain ? 2u : td[C->tdna].maxlen;
  const u32 lpw_q = (seg_max * (qmax > dper ? qmax : dper) + 31) / 32 + 2;
  if (C->nnc + tb > 32u * (LPW_T - 1)) return 1000; // the GPU would take the two-walk kernels
  C->strd_q = (u32)((u64)TASK_RECORDS * qsum / 32) + 3; C->strd_d = (u32)((u64)TASK_RECORDS * C->max_qlen * dper / 32) + 3;
  C->strd_t = (u32)((u64)TASK_BLOCKS * ((C->nnc + 32ull * tb + 7) / 8 * 8) / 32) + 3;
  C->info_words = (u32)(((u64)R * C->nb_len + 31) / 32) + 1;
  const u32 strd = C->strd_q + C->strd_d + C->strd_t;
  std::vector<u32> tmp((size_t)C->info_words + (size_t)C->ntask * strd, 0xDEADBEEFu); // stale contents must not matter
  u32 *len3 = arena + C->task_off, *base3 = len3 + 3 * C->ntask;
  auto prev_of = [&](u32 r) { return [&, r](u32 f, i32) { return r ? (i32)vals[(size_t)(r - 1) * nf + f] : 0; }; };
  bool over = false;
  std::vector<u32> lp(32 * (lpw_q > LPW_T ? lpw_q : LPW_T));
  for (u32 task = 0; task < C->ntask; ++task) {
    u32 *slot = tmp.data() + C->info_words + (size_t)task * strd;
    // k_enc_title
    HostStream T; T.init(slot + C->strd_q + C->strd_d, C->strd_t);
    for (u32 g = task * TASK_BLOCKS; g < (task + 1) * TASK_BLOCKS && g < C->nblk; ++g) {
      u32 lo = g * 32, nrec = R - lo < 32 ? R - lo : 32, flags = arena[C->flagbits_off + g];
      u32 ci[32] = {0};
      for (u32 l = 0; l < nrec && C->nb_len; ++l) {
        u32 L = se[lo + l] - te[lo + l] - 1, pos = l * C->nb_len, sh = pos & 31, v = L << (32 - C->nb_len);
        cc_or(ci, pos >> 5, v >> sh);
        if (sh + C->nb_len > 32) cc_or(ci, (pos >> 5) + 1, v << (32 - sh));
      }
      for (u32 l = 0; l < (nrec * C->nb_len + 31) / 32; ++l) tmp[g * C->nb_len + l] = ci[l];
      if (!C->nnc) continue;
      u32 nb[32];
      for (u32 l = 0; l < 32; ++l) {
        nb[l] = 0;
        if (l >= nrec) continue;
        LaneSinkT<PtrStore> sk; sk.init(PtrStore{lp.data() + l * LPW_T, 1u}, LPW_T);
        if (l == 0) { u32 v = 0; for (u32 k = 0; k < C->nnc; ++k) v = (v << 1) | ((flags >> C->ncf[k]) & 1u); sk.put(v, C->nnc); }
        title_record(b, lut, rstart[lo + l], te[lo + l], *C, C->f, C->ncf, C->ncskip, arena, flags, l == 0, prev_of(lo + l), sk);
        nb[l] = sk.finish(); over = over || sk.over;
      }
      T.append(lp.data(), LPW_T, nb);
      T.pad_to_byte();
    }
    len3[2 * C->ntask + task] = T.finish() >> 3; over = over || T.over;
    // k_enc_qd<G>
    HostStream Q, D; Q.init(slot, C->strd_q); D.init(slot + C->strd_q, C->strd_d);
    const u32 RW = 32 / G, rec0 = task * TASK_RECORDS, rec1 = rec0 + TASK_RECORDS < R ? rec0 + TASK_RECORDS : R;
    const u64 *qcl = (const u64 *)(arena + td[C->tq0].cl_off);
    const u64 *dcl = C->plain ? (const u64 *)0 : (const u64 *)(arena + td[C->tdna].cl_off);
    for (u32 i0 = rec0; i0 < rec1; i0 += RW) {
      u32 qn[32], dn[32];
      std::vector<u32> lpd(32 * lpw_q);
      for (u32 l = 0; l < 32; ++l) {
        qn[l] = dn[l] = 0;
        u32 i = i0 + l / G, part = l % G;
        if (i >= rec1) continue;
        u32 L = se[i] - te[i] - 1, seg = seg_len(L, G), a = part * seg < L ? part * seg : L, e = a + seg < L ? a + seg : L;
        bool xf = kx[i] >> 15;
        const u8 *sp = b + te[i] + 1, *qp = b + se[i] + 3;
        LaneSinkT<PtrStore> sq; sq.init(PtrStore{lp.data() + l * lpw_q, 1u}, lpw_q);
        for (u32 j = a; j < e; ++j) {
          u8 q = qp[j];
          if (xf) { u32 am = amb_code(sp[j]); if (am > 1) q = xfer_qual(am, q); }
          u64 en = qcl[(size_t)(j + 1) * C->nq + C->qua_code[q]];
          sq.put((u32)en, (u32)(en >> 32));
        }
        qn[l] = sq.finish(); over = over || sq.over;
        LaneSinkT<PtrStore> sd; sd.init(PtrStore{lpd.data() + l * lpw_q, 1u}, lpw_q);
        for (u32 j = a; j < e; ++j) {
          u8 c = sp[j];
          if (xf && !is_acgt(c)) continue;
          if (C->plain) sd.put(C->sym_code[c], 2); else { u64 en = dcl[C->sym_code[c]]; sd.put((u32)en, (u32)(en >> 32)); }
        }
        dn[l] = sd.finish(); over = over || sd.over;
      }
      Q.append(lp.data(), lpw_q, qn);
      D.append(lpd.data(), lpw_q, dn);
    }
    len3[task] = Q.finish(); len3[C->ntask + task] = D.finish(); over = over || Q.over || D.over;
  }
  if (over) return E_CAPACITY;
  // k_layout
  std::vector<u32> tlen(C->ntab), tdst(C->ntab);
  for (u32 i = 0; i < C->ntab; ++i) tlen[i] = td[i].tree_len;
  if (!layout_headers(b, *C, arena, tlen.data(), tdst.data())) return E_UNSUPPORTED;
  u8 *stage = (u8 *)(arena + C->stage_off);
  for (u32 i = 0; i < C->ntab; ++i) memcpy(stage + tdst[i], (u8 *)(arena + td[i].tree_off), td[i].tree_len);
  u64 tot[3] = {0, 0, 0};
  for (u32 k = 0; k < 3; ++k) for (u32 t = 0; t < C->ntask; ++t) { base3[k * C->ntask + t] = (u32)tot[k]; tot[k] += len3[k * C->ntask + t]; }
  finish_layout(*C, (u32)tot[2], tot[0], tot[1]);
  if (C->payload_len > out_cap) return E_CAPACITY;
  // k_place
  memset(out, 0, (C->payload_len + 7) & ~3u);
  u32 *outw = (u32 *)out;
  ByteWriter w; w.p = out; w.n = 0;
  w.word(C->R); w.word(C->max_qlen); w.word(C->max_slen); w.byte((u8)C->nsym); w.byte(0); w.byte((u8)C->nq); w.word(C->flags);
  const u32 o_title = C->info_len, o_qual = o_title + C->title_len, o_dna = o_qual + C->qual_len;
  memcpy(out + o_title, stage, C->thdr_len);
  memcpy(out + o_qual, stage + C->thdr_cap, C->qhdr_len);
  memcpy(out + o_dna, stage + C->thdr_cap + C->qhdr_cap, C->dhdr_len);
  auto place = [&](u64 dbit, const u32 *src, u32 nbits) {
    if (!nbits) return;
    u32 sh = (u32)(dbit & 31), nsrc = (nbits + 31) / 32, nd = (sh + nbits + 31) / 32;
    for (u32 j = 0; j < nd; ++j) outw[(dbit >> 5) + j] |= bswap32(shifted_word(src, nsrc, sh, j));
  };
  const u64 info_bits = (u64)R * C->nb_len;
  for (u64 b0 = 0; b0 < info_bits; b0 += 32ull * PIECE_WORDS)
    place((u64)INFO_FIXED * 8 + b0, tmp.data() + b0 / 32, (u32)(info_bits - b0 < 32ull * PIECE_WORDS ? info_bits - b0 : 32ull * PIECE_WORDS));
  const u64 bit0[3] = {(u64)(o_qual + C->qhdr_len) * 8, (u64)(o_dna + C->dhdr_len) * 8, (u64)(o_title + C->thdr_len) * 8};
  for (u32 task = 0; task < C->ntask; ++task)
    for (u32 k = 0; k < 3; ++k) {
      u32 bits = len3[k * C->ntask + task] * (k == 2 ? 8u : 1u);
      const u32 *src = tmp.data() + C->info_words + (size_t)task * strd + (k == 0 ? 0u : k == 1 ? C->strd_q : C->strd_q + C->strd_d);
      u64 tbase = (u64)base3[k * C->ntask + task] * (k == 2 ? 8u : 1u);
      for (u32 b0 = 0; b0 < bits; b0 += 32 * PIECE_WORDS)
        place(bit0[k] + tbase + b0, src + b0 / 32, bits - b0 < 32 * PIECE_WORDS ? bits - b0 : 32 * PIECE_WORDS);
    }
  return 0;
}

// fastG = 0: the two-walk encoder (count, scan, write).  fastG = 1, 2, 4, 8: the single-walk encoder of phy_fast.cuh /
// phy_encode.cuh emulated lane by lane -- lane-private sinks, warp concatenation with carry, task slots in a temporary
// buffer, scans of the task totals, placement with shifted_word -- with fastG lanes per record for quality and DNA.
static int mirror_window(const u8 *b, u64 readable, i64 rsize, u32 rec_start, i32 overlap, u32 cap,
                         u8 *out, u32 out_cap, u32 *sec_len, u32 *n_records, u64 *bytes_consumed, u32 fastG) {
  // record split, serial (same rule as the plan kernel: phyNGSC.cpp:254-331)
  std::vector<u32> te, se, rstart;
  {
    u64 pos = rec_start;
    rstart.push_back((u32)pos);
    i64 lim = rsize < (i64)readable ? rsize : (i64)readable;
    for (;;) {
      const u8 *q = (const u8 *)memchr(b + pos, '\n', readable - pos);
      if (!q) break;
      u64 t = q - b;
      if (!te.empty() && (i64)t >= lim) break;
      q = (const u8 *)memchr(b + t + 1, '\n', readable - t - 1);
      if (!q) return E_MALFORMED;
      u64 s = q - b;
      u64 nx = 2 * s - t + 3;
      if (nx > readable + 1) return E_MALFORMED;
      te.push_back((u32)t); se.push_back((u32)s); rstart.push_back((u32)nx);
      pos = nx;
      if (te.size() > 1) {
        if ((i64)nx >= rsize - overlap) break;
        if (te.size() > cap) break;
      }
      if (pos >= readable) break;
    }
  }
  u32 R = (u32)te.size();
  if (!R) return E_MALFORMED;
  u8 lut[256];
  fill_char_lut(lut);
  std::vector<u16> kx(R);
  SbAcc *A = (SbAcc *)calloc(1, sizeof(SbAcc));
  // stat1
  TitleCursor c0; c0.init(b, rstart[0], te[0], lut);
  Tok t; u32 nf = 0; u32 off0[MAXF], len0[MAXF];
  while (c0.next(t)) { if (nf < (u32)MAXF) { off0[nf] = t.start - rstart[0]; len0[nf] = t.end - t.start; } ++nf; }
  if (nf == 0 || nf > (u32)MAXF) return E_UNSUPPORTED;
  std::vector<u32> vals((size_t)R * nf);
  for (u32 r = 0; r < R; ++r) {
    u32 L = se[r] - te[r] - 1, qs = se[r] + 3;
    if (L == 0 || b[se[r] + 1] != '+' || b[se[r] + 2] != '\n') return E_MALFORMED;
    SeqStat st;
    seqqual_stat(b, te[r] + 1, L, qs, st, [&](u8 c) { A->dna_occ[c]++; }, [&](u8 q) { A->qpresent[q >> 5] |= 1u << (q & 31); });
    if (st.err) return E_UNSUPPORTED;
    A->dna_occ['A'] += st.acgt[0]; A->dna_occ['C'] += st.acgt[1]; A->dna_occ['G'] += st.acgt[2]; A->dna_occ['T'] += st.acgt[3];
    kx[r] = (u16)(st.kept | (st.xfer << 15));
    amax(A->max_qlen, L); amax(A->max_slen, st.kept); amax(A->inv_min_qlen, ~L);
    if (count_seps(b, rstart[r], te[r]) != nf) return E_FIELDS;
    TitleCursor cur; cur.init(b, rstart[r], te[r], lut);
    for (u32 f = 0; f < nf; ++f) {
      cur.next(t);
      u32 len = t.end - t.start;
      FieldAcc &a = A->f[f];
      amax(a.inv_min_len, ~len); amax(a.max_len, len);
      if (!t.num) a.not_num = 1;
      amax(a.kmax_v, key_of((i32)t.v)); amax(a.kinvmin_v, ~key_of((i32)t.v));
      if (r >= 1) { u32 kd = key_of((i32)(t.v - vals[(size_t)(r - 1) * nf + f])); amax(a.kmax_d, kd); amax(a.kinvmin_d, ~kd); }
      vals[(size_t)r * nf + f] = t.v;
      u32 m = len < len0[f] ? len : len0[f];
      for (u32 p = 0; p < m && p < (u32)MAXLEN0; ++p) if (b[t.start + p] != b[rstart[0] + off0[f] + p]) a.mism[p >> 5] |= 1u << (p & 31);
    }
  }
  const u32 AW = (8u << 20) / 4;
  u32 *arena = (u32 *)calloc(AW, 4);
  SbClass *C = (SbClass *)calloc(1, sizeof(SbClass));
  classify_subblock(b, lut, *A, R, rstart[0], te[0], arena, AW, *C);
  int rc = C->status;
  std::vector<u32> qoff(R + 1), doff(R + 1), blkoff((R + 31) / 32 + 1);
  if (!rc) {
    TableDesc *td = (TableDesc *)(arena + C->tabdesc_off);
    for (u32 i = C->zero_begin; i < C->zero_end; ++i) arena[i] = 0;
    if (!C->plain) for (u32 i = 0; i < C->nsym; ++i) arena[C->dnastat_off + i] = A->dna_occ[C->symbols[i]];
    // qhist
    u32 *gq = arena + C->qstat_off;
    for (u32 r = 0; r < R; ++r) {
      u32 L = se[r] - te[r] - 1, qs = se[r] + 3;
      for (u32 p = 0; p < L; ++p) {
        u8 q = b[qs + p];
        if (kx[r] >> 15) { u32 a = amb_code(b[te[r] + 1 + p]); if (a > 1) q = xfer_qual(a, q); }
        gq[(p + 1) * C->nq + C->qua_code[q]]++; gq[C->qua_code[q]]++;
      }
    }
    // stat2: histograms + block flags
    for (u32 lo = 0; lo < R; lo += 32) {
      u32 hi = lo + 32 < R ? lo + 32 : R, flags = 0;
      for (u32 f = 0; f < nf; ++f) {
        const FieldClass &F = C->f[f];
        if (F.kind == K_CONST) continue;
        bool bit = true;
        i32 bd = 0;
        u32 st_lo = 0, len_lo = 0;
        for (u32 r = lo; r < hi; ++r) {
          TitleCursor cur; cur.init(b, rstart[r], te[r], lut);
          for (u32 k = 0; k <= f; ++k) cur.next(t);
          u32 len = t.end - t.start;
          i32 v = (i32)t.v, pv = r ? (i32)vals[(size_t)(r - 1) * nf + f] : 0;
          if (F.kind == K_STR) {
            if (r == lo) { st_lo = t.start; len_lo = len; }
            else if (len != len_lo || memcmp(b + t.start, b + st_lo, len)) bit = false;
            const u16 *sm = (const u16 *)(arena + F.slotmap_off);
            for (u32 j = 0; j < len; ++j)
              if (j >= F.len0 || ((F.mism[j >> 5] >> (j & 31)) & 1u)) arena[td[sm[j < 128 ? j : 128]].freq_off + b[t.start + j]]++;
          } else if (F.is_delta) {
            i32 dl = wsub(v, pv);
            if (r == lo + 1) bd = dl; else if (r > lo + 1 && dl != bd) bit = false;
            if (F.has_table && r >= 1) arena[td[F.tab].freq_off + (u32)wsub(dl, F.base)]++;
          } else {
            if (v != (i32)vals[(size_t)lo * nf + f]) bit = false;
            if (F.has_table) arena[td[F.tab].freq_off + (u32)wsub(v, F.base)] += r == 0 ? 2 : 1;
          }
        }
        if (F.kind == K_NUM && F.is_delta && bd != F.min_d) bit = false;
        if (bit) flags |= 1u << f;
      }
      arena[C->flagbits_off + lo / 32] = flags;
    }
    // huffman
    HuffScratch *HS = new HuffScratch;
    for (u32 i = 0; i < C->ntab; ++i)
      td[i].tree_len = huff_table(arena + td[i].freq_off, td[i].n, (u64 *)(arena + td[i].cl_off), (u8 *)(arena + td[i].tree_off), *HS, 0u, 1u, NoSync());
    delete HS;
    for (u32 i = 0; i < C->ntab; ++i) {
      u32 ml = 0;
      for (u32 k = 0; k < td[i].n && td[i].tree_len; ++k) { u32 l = (u32)(((const u64 *)(arena + td[i].cl_off))[k] >> 32); if (l > ml) ml = l; }
      td[i].maxlen = ml;
    }
    if (fastG) {
      rc = fast_encode(b, lut, te, se, rstart, kx, vals, nf, arena, AW, C, fastG, out, out_cap);
      if (!rc) {
        sec_len[0] = C->info_len; sec_len[1] = C->title_len; sec_len[2] = C->qual_len; sec_len[3] = C->dna_len;
        *n_records = R; *bytes_consumed = rstart[R];
      }
      free(A); free(arena); free(C);
      return rc;
    }
    // lengths
    auto prev_of = [&](u32 r) { return [&, r](u32 f, i32) { return r ? (i32)vals[(size_t)(r - 1) * nf + f] : 0; }; };
    for (u32 r = 0; r < R; ++r) {
      u32 L = se[r] - te[r] - 1; bool xf = kx[r] >> 15;
      CountSink q; q.init();
      QFull qt; qt.cl = (const u64 *)(arena + td[C->tq0].cl_off); qt.nq = C->nq;
      quality_record(b, te[r] + 1, L, se[r] + 3, xf, C->qua_code, qt, q);
      qoff[r] = (u32)q.bits;
      CountSink dn; dn.init();
      dna_record(b, te[r] + 1, L, xf, C->plain != 0, C->sym_code, C->plain ? (const u64 *)0 : (const u64 *)(arena + td[C->tdna].cl_off), dn);
      doff[r] = (u32)dn.bits;
    }
    for (u32 lo = 0; lo < R && C->nnc; lo += 32) {
      u32 hi = lo + 32 < R ? lo + 32 : R; u64 bits = C->nnc;
      for (u32 r = lo; r < hi; ++r) {
        CountSink ts; ts.init();
        title_record(b, lut, rstart[r], te[r], *C, C->f, C->ncf, C->ncskip, arena, arena[C->flagbits_off + lo / 32], r == lo, prev_of(r), ts);
        bits += ts.bits;
      }
      blkoff[lo / 32] = (u32)((bits + 7) / 8);
    }
    // layout
    std::vector<u32> tlen(C->ntab), tdst(C->ntab);
    for (u32 i = 0; i < C->ntab; ++i) tlen[i] = td[i].tree_len;
    if (!layout_headers(b, *C, arena, tlen.data(), tdst.data())) rc = E_UNSUPPORTED;
    for (u32 i = 0; i < C->ntab; ++i) td[i].dst = tdst[i];
    if (!rc) {
      u8 *stage = (u8 *)(arena + C->stage_off);
      for (u32 i = 0; i < C->ntab; ++i) memcpy(stage + td[i].dst, (u8 *)(arena + td[i].tree_off), td[i].tree_len);
      u64 qb = 0, db = 0, tb = 0;
      for (u32 r = 0; r < R; ++r) { u32 v = qoff[r]; qoff[r] = (u32)qb; qb += v; v = doff[r]; doff[r] = (u32)db; db += v; }
      for (u32 k = 0; k < C->nblk && C->nnc; ++k) { u32 v = blkoff[k]; blkoff[k] = (u32)tb; tb += v; }
      finish_layout(*C, (u32)tb, qb, db);
      if (C->payload_len > out_cap) rc = E_CAPACITY;
    }
    // the 16-bit packed copy of the quality tables the GPU keeps in shared memory
    std::vector<u16> pk((size_t)(C->max_qlen + 1) * C->nq);
    bool use_packed = true;
    for (size_t i = 0; i < pk.size(); ++i) use_packed = qpack_entry(((const u64 *)(arena + td[C->tq0].cl_off))[i], pk[i]) && use_packed;
    if (!rc) {
      memset(out, 0, (C->payload_len + 7) & ~3u);
      u32 *outw = (u32 *)out;
      ByteWriter w; w.p = out; w.n = 0;
      w.word(C->R); w.word(C->max_qlen); w.word(C->max_slen); w.byte((u8)C->nsym); w.byte(0); w.byte((u8)C->nq); w.word(C->flags);
      const u32 o_title = C->info_len, o_qual = o_title + C->title_len, o_dna = o_qual + C->qual_len;
      const u8 *stage = (const u8 *)(arena + C->stage_off);
      memcpy(out + o_title, stage, C->thdr_len);
      memcpy(out + o_qual, stage + C->thdr_cap, C->qhdr_len);
      memcpy(out + o_dna, stage + C->thdr_cap + C->qhdr_cap, C->dhdr_len);
      for (u32 r = 0; r < R; ++r) {
        u32 L = se[r] - te[r] - 1; bool xf = kx[r] >> 15;
        OrSink k; k.init(outw, (u64)INFO_FIXED * 8 + (u64)r * C->nb_len); k.put(L, C->nb_len); k.finish();
        OrSink q; q.init(outw, (u64)(o_qual + C->qhdr_len) * 8 + qoff[r]);
        if (use_packed) { QPacked qp; qp.pk = pk.data(); qp.nq = C->nq; quality_record(b, te[r] + 1, L, se[r] + 3, xf, C->qua_code, qp, q); }
        else { QFull qt; qt.cl = (const u64 *)(arena + td[C->tq0].cl_off); qt.nq = C->nq; quality_record(b, te[r] + 1, L, se[r] + 3, xf, C->qua_code, qt, q); }
        q.finish();
        OrSink dn; dn.init(outw, (u64)(o_dna + C->dhdr_len) * 8 + doff[r]);
        dna_record(b, te[r] + 1, L, xf, C->plain != 0, C->sym_code, C->plain ? (const u64 *)0 : (const u64 *)(arena + td[C->tdna].cl_off), dn); dn.finish();
      }
      for (u32 lo = 0; lo < R && C->nnc; lo += 32) {
        u32 hi = lo + 32 < R ? lo + 32 : R, flags = arena[C->flagbits_off + lo / 32];
        OrSink ts; ts.init(outw, (u64)(o_title + C->thdr_len + blkoff[lo / 32]) * 8);
        u32 v = 0;
        for (u32 f = 0; f < nf; ++f) if (C->f[f].kind != K_CONST) v = (v << 1) | ((flags >> f) & 1u);
        ts.put(v, C->nnc);
        for (u32 r = lo; r < hi; ++r) title_record(b, lut, rstart[r], te[r], *C, C->f, C->ncf, C->ncskip, arena, flags, r == lo, prev_of(r), ts);
        ts.finish();
      }
      sec_len[0] = C->info_len; sec_len[1] = C->title_len; sec_len[2] = C->qual_len; sec_len[3] = C->dna_len;
      *n_records = R; *bytes_consumed = rstart[R];
    }
  }
  free(A); free(arena); free(C);
  return rc;
}

extern "C" int mirror_compress_window(const u8 *b, u64 readable, i64 rsize, u32 rec_start, i32 overlap, u32 cap,
                                      u8 *out, u32 out_cap, u32 *sec_len, u32 *n_records, u64 *bytes_consumed) {
  return mirror_window(b, readable, rsize, rec_start, overlap, cap, out, out_cap, sec_len, n_records, bytes_consumed, 0);
}
extern "C" int mirror_compress_window_fast(const u8 *b, u64 readable, i64 rsize, u32 rec_start, i32 overlap, u32 cap,
                                           u8 *out, u32 out_cap, u32 *sec_len, u32 *n_records, u64 *bytes_consumed, u32 lanes_per_record) {
  return mirror_window(b, readable, rsize, rec_start, overlap, cap, out, out_cap, sec_len, n_records, bytes_consumed, lanes_per_record);
}

/* where the encoder-path fields sit in SbClass, for tests that decode the GPU's per-subblock records
 * (phy_debug_read(ctx, "cls", ...)): sizeof, then the byte offsets of status, fast, qpk_esc, max_qlen, nq */
extern "C" u32 mirror_sbclass_layout(u32 *v, u32 n) {
  const u32 w[6] = {(u32)sizeof(SbClass), (u32)offsetof(SbClass, status), (u32)offsetof(SbClass, fast), (u32)offsetof(SbClass, qpk_esc),
                    (u32)offsetof(SbClass, max_qlen), (u32)offsetof(SbClass, nq)};
  for (u32 i = 0; i < n && i < 6; ++i) v[i] = w[i];
  return 6;
}

extern "C" u32 mirror_huffman(const u32 *freq, u32 n, u64 *cl, u8 *tree) {
  /* tables of up to 64 symbols take the small scratch on the GPU (k_huff's first launch): same function, other capacity */
  if (n <= HuffScratchSmall::CAP) {
    HuffScratchSmall *HS = new HuffScratchSmall;
    u32 k = huff_table(freq, n, cl, tree, *HS, 0u, 1u, NoSync());
    delete HS;
    return k;
  }
  HuffScratch *HS = new HuffScratch;
  u32 k = huff_table(freq, n, cl, tree, *HS, 0u, 1u, NoSync());
  delete HS;
  return k;
}
