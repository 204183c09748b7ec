// draco_sharp_b200/csrc/dcb_mesh_host.cu -- HOST code: Edgebreaker connectivity + attribute traversal helper
// (SURVEY.md 8f-1).  north_star keeps connectivity decoding on the host because it is inherently sequential; in
// the drop-in the C# reference does it (MeshEdgeBreakerDecoder) and hands the tables over through
// dcb_set_mesh_maps.  This helper is the same step for callers without the C# host (Python, C++, the tests):
// dcb_host_connectivity(batch, buf) decodes the connectivity of one mesh buffer on the CPU and installs the
// attribute-section offset and the per-decoder maps.  Nothing here runs on the GPU and nothing here decodes
// attribute values.
//
// Reference code restated ("D/" = src/Draco/):
//   D/IO/Mesh/MeshEdgeBreakerDecoder.cs:25-134 (header), :136-230 (topology splits), :232-442 (symbol loop),
//   :450-470 (IsTopologySplit), :502-535 (attribute seams), :537-638 (points / faces), :640-760 (decoder wiring)
//   D/IO/Mesh/MeshEdgeBreakerTraversalDecoder.cs:27-108, MeshEdgeBreakerTraversalValenceDecoder.cs:22-150
//   D/IO/BitCoders/RAnsBitDecoder.cs:12-35, D/IO/Entropy/AnsDecoder.cs:12-56 (B-17: 1-byte init reads offset-1)
//   D/IO/Mesh/CornerTable.cs:59-260, MeshAttributeCornerTable.cs:78-190
//   D/IO/Mesh/Traverser/DepthFirstTraverser.cs:9-99, MeshTraversalSequencer.cs:13-31,
//   MeshAttributeIndicesEncodingObserver.cs:14-21
// Not restated: predictive traversal (type 1), MaxPredictionDegree traversal -> DCB_ERR_UNSUPPORTED.
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "dcb_internal.h"
#include "dcb_mesh_host.h"

namespace {

constexpr uint32_t INV = 0xFFFFFFFFu;

struct Reader {
  const uint8_t *p;
  uint64_t len, pos;
  int err = 0;
  uint32_t u8() {
    if (err || pos >= len) { err = DCB_ERR_EOF; return 0; }
    return p[pos++];
  }
  uint64_t varint() {
    uint64_t v = 0;
    unsigned sh = 0;
    if (err) return 0;
    for (int i = 0; i < 10; ++i) {
      if (pos >= len) { err = DCB_ERR_EOF; return 0; }
      const uint32_t b = p[pos++];
      v |= (uint64_t)(b & 0x7F) << sh;
      if (!(b & 0x80)) return v;
      sh += 7;
    }
    err = DCB_ERR_EOF;
    return 0;
  }
};

// rABS binary decoder (AnsDecoder.cs:12-56; L = 4096, 8-bit probabilities)
struct RabsBits {
  const uint8_t *buf = nullptr;
  int64_t off = 0;
  uint32_t state = 0;
  uint32_t prob_zero = 0;
  int start(Reader &r) {
    prob_zero = r.u8();
    const uint64_t n = r.varint();
    if (r.err) return r.err;
    if (r.len - r.pos < n) return DCB_ERR_EOF;
    const uint8_t *b = r.p + r.pos;
    r.pos += n;
    if (n < 1) return DCB_ERR_CONNECTIVITY;
    const uint32_t x = (uint32_t)b[n - 1] >> 6;
    buf = b;
    if (x == 0) { off = (int64_t)n - 1; state = b[n - 1] & 0x3Fu; }
    else if (x == 1) { if (n < 2) return DCB_ERR_CONNECTIVITY; off = (int64_t)n - 2; state = ((uint32_t)b[n - 2] | ((uint32_t)b[n - 1] << 8)) & 0x3FFFu; }
    else if (x == 2) { if (n < 3) return DCB_ERR_CONNECTIVITY; off = (int64_t)n - 3; state = ((uint32_t)b[n - 3] | ((uint32_t)b[n - 2] << 8) | ((uint32_t)b[n - 1] << 16)) & 0x3FFFFFu; }
    else return DCB_ERR_CONNECTIVITY;
    state += 4096u;
    return state >= 4096u * 256u ? DCB_ERR_CONNECTIVITY : DCB_OK;
  }
  uint32_t bit() {
    const uint32_t p = (256u - prob_zero) & 0xFFu;
    if (state < 4096u && off > 0) state = state * 256u + buf[--off];
    const uint32_t x = state, quot = x >> 8, rem = x & 255u, xn = quot * p;
    const bool val = rem < p;
    state = val ? xn + rem : x - xn - p;
    return val ? 1u : 0u;
  }
};

// Raw / Tagged symbols of the valence contexts and of sequential-mesh indices (SymbolDecoding.cs:7-67), host side.
// raw_loc != NULL: a Raw stream is only checked and located (RANS_TABLE at raw_loc->off, payload behind it), not decoded;
// raw_loc->located stays false for a Tagged one, which is decoded as usual.
int host_symbols(Reader &r, uint32_t n, std::vector<uint32_t> &out, DcbSeqIndexLoc *raw_loc = nullptr) {
  if (n == 0) {
    out.clear();
    return DCB_OK;
  }
  const uint32_t scheme = r.u8();
  if (r.err) return r.err;
  int mbl = 5;
  if (scheme == 1) {
    mbl = (int)r.u8();
    if (r.err) return r.err;
    if (mbl < 1 || mbl > 18) return DCB_ERR_BITLEN;
  } else if (scheme != 0) {
    return DCB_ERR_SCHEME;
  }
  const int pb = dcb_rans_precision(mbl);
  const uint32_t prec = 1u << pb, lbase = 4u << pb;
  const uint64_t table_off = r.pos;
  const uint64_t ns = r.varint();
  if (r.err) return r.err;
  if (ns == 0) return DCB_ERR_NUM_SYMBOLS;
  if (ns > (r.len - r.pos) * 64u || ns > (1u << 20)) return DCB_ERR_EOF;
  std::vector<uint32_t> prob(ns, 0), cum(ns + 1, 0);
  for (uint64_t i = 0; i < ns; ++i) {
    const uint32_t pd = r.u8();
    if (r.err) return r.err;
    const uint32_t tok = pd & 3u;
    if (tok == 3u) {
      const uint32_t off = pd >> 2;
      if (i + off >= ns) return DCB_ERR_TABLE;
      i += off;
    } else {
      uint32_t pr = pd >> 2;
      for (uint32_t b = 0; b < tok; ++b) pr |= r.u8() << (8 * (b + 1) - 2);
      if (r.err) return r.err;
      prob[i] = pr;
    }
  }
  uint64_t c = 0;
  for (uint64_t i = 0; i < ns; ++i) { cum[i] = (uint32_t)c; c += prob[i]; if (c > prec) return DCB_ERR_TABLE; }
  if (c != prec) return DCB_ERR_TABLE;
  cum[ns] = prec;
  const uint64_t nb = r.varint();
  if (r.err) return r.err;
  if (r.len - r.pos < nb) return DCB_ERR_EOF;
  const uint8_t *buf = r.p + r.pos;
  r.pos += nb;
  if (nb < 1) return DCB_ERR_RANS_INIT;
  const uint32_t tg = (uint32_t)buf[nb - 1] >> 6;
  if (nb < tg + 1u) return DCB_ERR_RANS_INIT;
  uint32_t v = 0;
  for (uint32_t i = 0; i <= tg; ++i) v |= (uint32_t)buf[nb - 1 - tg + i] << (8 * i);
  v &= tg == 0 ? 0x3Fu : tg == 1 ? 0x3FFFu : tg == 2 ? 0x3FFFFFu : 0x3FFFFFFFu;
  uint32_t state = v + lbase;
  int64_t off = (int64_t)nb - (tg + 1);
  if (state >= lbase * 256u) return DCB_ERR_RANS_INIT;
  if (raw_loc && scheme == 1) {  // every check the decode makes is behind us: the symbols themselves cannot fail
    raw_loc->off = table_off;
    raw_loc->bytes = r.pos - table_off;
    raw_loc->mbl = mbl;
    raw_loc->located = true;
    return DCB_OK;
  }
  out.assign(n, 0);
  std::vector<uint32_t> lut(prec);
  for (uint64_t i = 0; i < ns; ++i)
    for (uint32_t j = cum[i]; j < cum[i + 1]; ++j) lut[j] = (uint32_t)i;
  auto read = [&]() {
    while (state < lbase && off > 0) state = state * 256u + buf[--off];
    const uint32_t q = state >> pb, rem = state & (prec - 1u), s = lut[rem];
    state = q * prob[s] + rem - cum[s];
    return s;
  };
  if (scheme == 1) {
    for (uint32_t i = 0; i < n; ++i) out[i] = read();
  } else {
    uint64_t bitpos = 0;
    const uint8_t *bits = r.p + r.pos;
    const uint64_t blen = r.len - r.pos;
    for (uint32_t i = 0; i < n; ++i) {
      const uint32_t bl = read() & 0xFFu;
      if (bl > 32) return DCB_ERR_TAG;
      uint32_t val = 0;
      for (uint32_t k = 0; k < bl; ++k, ++bitpos) {
        if ((bitpos >> 3) >= blen) return DCB_ERR_EOF;
        val |= (uint32_t)((bits[bitpos >> 3] >> (bitpos & 7)) & 1u) << k;
      }
      out[i] = val;
    }
    r.pos += (bitpos + 7) / 8;
  }
  return DCB_OK;
}

inline uint32_t c_next(uint32_t c) { return c == INV ? c : ((c + 1) % 3 != 0 ? c + 1 : c - 2); }
inline uint32_t c_prev(uint32_t c) { return c == INV ? c : (c % 3 != 0 ? c - 1 : c + 2); }

// corner table view: base table or an attribute's table (seam edges cut)
struct View {
  const std::vector<uint32_t> *opp, *c2v, *vleft;
  uint32_t n_vertices;
  uint32_t Opp(uint32_t c) const { return c == INV ? c : (*opp)[c]; }
  uint32_t Vertex(uint32_t c) const { return (c == INV || c >= c2v->size()) ? c : (*c2v)[c]; }
  uint32_t SwingRight(uint32_t c) const { return c_prev(Opp(c_prev(c))); }
  uint32_t SwingLeft(uint32_t c) const { return c_next(Opp(c_next(c))); }
  uint32_t RightCorner(uint32_t c) const { return c == INV ? INV : Opp(c_next(c)); }
  uint32_t LeftCorner(uint32_t c) const { return c == INV ? INV : Opp(c_prev(c)); }
  bool OnBoundary(uint32_t v) const {
    const uint32_t c = (*vleft)[v];
    return c == INV || SwingLeft(c) == INV;
  }
};

struct AttrTable {
  std::vector<uint8_t> edge_seam, vert_seam;
  std::vector<uint32_t> c2v, opp, vleft;
  uint32_t n_vertices = 0;
};

class EdgebreakerHost {
 public:
  std::vector<uint32_t> c2v, opp, vcorner;  // base corner table
  std::vector<uint8_t> is_vert_hole;
  std::vector<AttrTable> att;
  std::vector<uint32_t> faces;
  uint32_t n_points = 0;

  int Decode(const uint8_t *buf, uint64_t len, uint64_t &pos, int traversal_type);
  int BuildMaps(const uint8_t *dec_ids, int n_dec, std::vector<DcbHostMaps> &maps);

 private:
  View Base() const { return View{&opp, &c2v, &vcorner, (uint32_t)vcorner.size()}; }
  void BuildAttrTable(AttrTable &a);
  void AssignPoints();
  static void Traverse(const View &t, uint32_t n_faces, std::vector<uint32_t> &d2c, std::vector<int32_t> &v2d);
};

// MeshAttributeCornerTable.RecomputeVertices(null, null): :107-155
void EdgebreakerHost::BuildAttrTable(AttrTable &a) {
  const uint32_t nc = (uint32_t)c2v.size();
  a.vert_seam.assign(vcorner.size(), 0);
  a.opp.resize(nc);
  for (uint32_t c = 0; c < nc; ++c) {
    a.opp[c] = a.edge_seam[c] ? INV : opp[c];
    if (a.edge_seam[c]) {
      a.vert_seam[c2v[c_next(c)]] = 1;
      a.vert_seam[c2v[c_prev(c)]] = 1;
    }
  }
  a.c2v.assign(nc, INV);
  a.vleft.clear();
  const View av{&a.opp, &a.c2v, &a.vleft, 0};
  const View bv = Base();
  for (uint32_t v = 0; v < vcorner.size(); ++v) {
    const uint32_t c = vcorner[v];
    if (c == INV) continue;
    uint32_t first_vert = (uint32_t)a.vleft.size();
    uint32_t first_c = c, act;
    if (a.vert_seam[v]) {
      act = av.SwingLeft(first_c);
      while (act != INV) {
        first_c = act;
        act = av.SwingLeft(act);
        if (act == c) break;
      }
    }
    a.c2v[first_c] = first_vert;
    a.vleft.push_back(first_c);
    act = bv.SwingRight(first_c);
    while (act != INV && act != first_c) {
      if (a.edge_seam[c_next(act)]) {
        first_vert = (uint32_t)a.vleft.size();
        a.vleft.push_back(first_c);  // sic (:146)
      }
      a.c2v[act] = first_vert;
      act = bv.SwingRight(act);
    }
  }
  a.n_vertices = (uint32_t)a.vleft.size();
}

int EdgebreakerHost::Decode(const uint8_t *buf, uint64_t len, uint64_t &pos, int traversal_type) {
  if (traversal_type != 0 && traversal_type != 2) return DCB_ERR_UNSUPPORTED;
  Reader r{buf, len, pos};
  const uint64_t n_enc_verts = r.varint(), n_faces = r.varint();
  if (r.err) return r.err;
  if (n_faces > (1u << 28) || n_enc_verts > n_faces * 3) return DCB_ERR_CONNECTIVITY;
  // Counts that the buffer cannot plausibly back fail before anything is allocated from them (the corner table alone
  // is 24 bytes per face): Edgebreaker symbols cost at least a fraction of a bit each even in the valence coder's
  // best case, and every mesh carries attribute bytes on top.  Generous: 64 faces per byte of the whole buffer.
  if (n_faces > 65536 + 64 * len) return DCB_ERR_CONNECTIVITY;
  if (n_faces > 0 && n_enc_verts * (n_enc_verts - 1) / 2 < 3 * n_faces / 2) return DCB_ERR_CONNECTIVITY;
  const uint32_t n_attr_data = r.u8();
  const uint64_t n_symbols = r.varint();
  if (r.err) return r.err;
  if (n_faces < n_symbols || n_faces > n_symbols + n_symbols / 3) return DCB_ERR_CONNECTIVITY;
  const uint64_t n_split_symbols = r.varint();
  if (r.err) return r.err;
  if (n_split_symbols > n_symbols) return DCB_ERR_CONNECTIVITY;
  const uint32_t nc = (uint32_t)n_faces * 3;
  c2v.assign(nc, INV);
  opp.assign(nc, INV);
  vcorner.clear();
  const uint32_t max_verts = (uint32_t)(n_enc_verts + n_split_symbols);
  is_vert_hole.assign(max_verts ? max_verts : 1, 1);
  // topology splits
  const uint64_t n_splits = r.varint();
  if (r.err) return r.err;
  if (n_splits > n_faces) return DCB_ERR_CONNECTIVITY;
  std::vector<uint32_t> split_src(n_splits), split_id(n_splits);
  std::vector<uint8_t> split_edge(n_splits);
  if (n_splits > 0) {
    uint32_t last = 0;
    for (uint64_t i = 0; i < n_splits; ++i) {
      uint32_t d = (uint32_t)r.varint();
      split_src[i] = d + last;
      d = (uint32_t)r.varint();
      if (r.err) return r.err;
      if (d > split_src[i]) return DCB_ERR_CONNECTIVITY;
      split_id[i] = split_src[i] - d;
      last = split_src[i];
    }
    const uint64_t nbytes = (n_splits + 7) / 8;
    if (r.len - r.pos < nbytes) return DCB_ERR_EOF;
    for (uint64_t i = 0; i < n_splits; ++i) split_edge[i] = (buf[r.pos + (i >> 3)] >> (i & 7)) & 1u;
    r.pos += nbytes;
  }
  // traversal start
  const uint8_t *sym_bits = nullptr;
  uint64_t sym_len = 0, sym_bitpos = 0;
  if (traversal_type == 0) {
    const uint64_t tsz = r.varint();
    if (r.err) return r.err;
    if (r.len - r.pos < tsz) return DCB_ERR_EOF;
    sym_bits = buf + r.pos;
    sym_len = tsz;
    r.pos += tsz;
  }
  RabsBits start_face;
  int st = start_face.start(r);
  if (st) return st;
  std::vector<RabsBits> seams(n_attr_data);
  for (auto &s : seams)
    if ((st = s.start(r))) return st;
  std::vector<uint32_t> valence;
  std::vector<uint32_t> ctx_syms[6];
  int64_t ctx_count[6] = {0, 0, 0, 0, 0, 0};
  if (traversal_type == 2) {
    valence.assign(max_verts ? max_verts : 1, 0);
    for (int i = 0; i < 6; ++i) {
      const uint64_t n = r.varint();
      if (r.err) return r.err;
      if (n > n_faces) return DCB_ERR_CONNECTIVITY;
      if (n > 0) {
        if ((st = host_symbols(r, (uint32_t)n, ctx_syms[i]))) return st;
        ctx_count[i] = (int64_t)n;
      }
    }
  }
  int last_symbol = -1, active_context = -1;
  static const uint8_t kTopo[5] = {0, 1, 3, 5, 7};
  bool bit_err = false;
  auto next_symbol = [&]() -> uint32_t {
    if (traversal_type == 0) {
      auto bit = [&]() -> uint32_t {
        if ((sym_bitpos >> 3) >= sym_len) { bit_err = true; return 0; }
        const uint32_t b = (sym_bits[sym_bitpos >> 3] >> (sym_bitpos & 7)) & 1u;
        ++sym_bitpos;
        return b;
      };
      uint32_t s = bit();
      if (s == 0) return 0;
      const uint32_t b1 = bit(), b2 = bit();
      return s | ((b1 | (b2 << 1)) << 1);
    }
    if (active_context != -1) {
      const int64_t k = --ctx_count[active_context];
      if (k < 0) return 9;
      const uint32_t id = ctx_syms[active_context][k];
      if (id > 4) return 9;
      last_symbol = kTopo[id];
    } else {
      last_symbol = 7;
    }
    return (uint32_t)last_symbol;
  };
  auto new_corner = [&](uint32_t corner) {
    if (traversal_type != 2) return;
    const uint32_t vc = c2v[corner], vn = c2v[c_next(corner)], vp = c2v[c_prev(corner)];
    switch (last_symbol) {
      case 0: case 1: valence[vn] += 1; valence[vp] += 1; break;
      case 5: valence[vc] += 1; valence[vn] += 1; valence[vp] += 2; break;
      case 3: valence[vc] += 1; valence[vn] += 2; valence[vp] += 1; break;
      case 7: valence[vc] += 2; valence[vn] += 2; valence[vp] += 2; break;
      default: break;
    }
    const int av = (int)valence[vn];
    active_context = (av < 2 ? 2 : (av > 7 ? 7 : av)) - 2;
  };
  auto add_vertex = [&]() { vcorner.push_back(INV); return (uint32_t)vcorner.size() - 1; };
  auto set_opp = [&](uint32_t a, uint32_t b) { opp[a] = b; opp[b] = a; };

  std::vector<uint32_t> stack, tkey, tval, invalid_verts;
  int64_t split_top = (int64_t)n_splits - 1;
  const bool remove_invalid = n_attr_data == 0;
  uint32_t num_faces = 0;
  for (uint64_t sid = 0; sid < n_symbols; ++sid) {
    const uint32_t face = num_faces++;
    bool check_split = false;
    const uint32_t sym = next_symbol();
    if (bit_err) return DCB_ERR_EOF;
    const uint32_t corner = 3 * face;
    if (sym == 0) {  // C
      if (stack.empty()) return DCB_ERR_CONNECTIVITY;
      const uint32_t ca = stack.back();
      const uint32_t vx = c2v[c_next(ca)];
      if (vx >= vcorner.size() || vcorner[vx] == INV) return DCB_ERR_CONNECTIVITY;
      const uint32_t cb = c_next(vcorner[vx]);
      if (ca == cb || opp[ca] != INV || opp[cb] != INV) return DCB_ERR_CONNECTIVITY;
      set_opp(ca, corner + 1);
      set_opp(cb, corner + 2);
      const uint32_t va_prev = c2v[c_prev(ca)], vb_next = c2v[c_next(cb)];
      if (vx == va_prev || vx == vb_next) return DCB_ERR_CONNECTIVITY;
      c2v[corner] = vx; c2v[corner + 1] = vb_next; c2v[corner + 2] = va_prev;
      if (va_prev != INV) vcorner[va_prev] = corner + 2;
      is_vert_hole[vx] = 0;
      stack.back() = corner;
    } else if (sym == 5 || sym == 3) {  // R / L
      if (stack.empty()) return DCB_ERR_CONNECTIVITY;
      const uint32_t ca = stack.back();
      if (opp[ca] != INV) return DCB_ERR_CONNECTIVITY;
      uint32_t oc, cl, cr;
      if (sym == 5) { oc = corner + 2; cl = corner + 1; cr = corner; }
      else { oc = corner + 1; cl = corner; cr = corner + 2; }
      set_opp(oc, ca);
      const uint32_t nv = add_vertex();
      if (vcorner.size() > max_verts) return DCB_ERR_CONNECTIVITY;
      c2v[oc] = nv;
      vcorner[nv] = oc;
      const uint32_t vr = c2v[c_prev(ca)];
      c2v[cr] = vr;
      if (vr != INV) vcorner[vr] = cr;
      c2v[cl] = c2v[c_next(ca)];
      stack.back() = corner;
      check_split = true;
    } else if (sym == 1) {  // S
      if (stack.empty()) return DCB_ERR_CONNECTIVITY;
      const uint32_t cb = stack.back();
      stack.pop_back();
      for (size_t k = 0; k < tkey.size(); ++k)
        if (tkey[k] == (uint32_t)sid) { stack.push_back(tval[k]); break; }
      if (stack.empty()) return DCB_ERR_CONNECTIVITY;
      const uint32_t ca = stack.back();
      if (ca == cb || opp[ca] != INV || opp[cb] != INV) return DCB_ERR_CONNECTIVITY;
      set_opp(ca, corner + 2);
      set_opp(cb, corner + 1);
      const uint32_t vp = c2v[c_prev(ca)];
      c2v[corner] = vp;
      c2v[corner + 1] = c2v[c_next(ca)];
      const uint32_t vb_prev = c2v[c_prev(cb)];
      c2v[corner + 2] = vb_prev;
      if (vb_prev != INV) vcorner[vb_prev] = corner + 2;
      uint32_t cn = c_next(cb);
      const uint32_t vn = c2v[cn];
      if (vp >= vcorner.size() || vn >= vcorner.size()) return DCB_ERR_CONNECTIVITY;
      if (traversal_type == 2) valence[vp] += valence[vn];
      vcorner[vp] = vcorner[vn];
      const View bv = Base();
      const uint32_t first = cn;
      while (cn != INV) {
        c2v[cn] = vp;
        cn = bv.SwingLeft(cn);
        if (cn == first) return DCB_ERR_CONNECTIVITY;
      }
      vcorner[vn] = INV;
      if (remove_invalid) invalid_verts.push_back(vn);
      stack.back() = corner;
    } else if (sym == 7) {  // E
      const uint32_t v0 = add_vertex(), v1 = add_vertex(), v2 = add_vertex();
      if (vcorner.size() > max_verts) return DCB_ERR_CONNECTIVITY;
      c2v[corner] = v0; c2v[corner + 1] = v1; c2v[corner + 2] = v2;
      vcorner[v0] = corner; vcorner[v1] = corner + 1; vcorner[v2] = corner + 2;
      stack.push_back(corner);
      check_split = true;
    } else {
      return DCB_ERR_CONNECTIVITY;
    }
    new_corner(stack.back());
    if (check_split) {
      const uint32_t enc_sid = (uint32_t)(n_symbols - sid - 1);
      for (;;) {
        if (split_top < 0) break;
        if (split_src[split_top] > enc_sid) return DCB_ERR_CONNECTIVITY;
        if (split_src[split_top] != enc_sid) break;
        const uint32_t edge = split_edge[split_top], enc_split = split_id[split_top];
        --split_top;
        const uint32_t top = stack.back();
        const uint32_t nac = edge == 1 ? c_next(top) : c_prev(top);
        const uint32_t dec_split = (uint32_t)(n_symbols - enc_split - 1);
        size_t k = 0;
        for (; k < tkey.size(); ++k)
          if (tkey[k] == dec_split) { tval[k] = nac; break; }
        if (k == tkey.size()) { tkey.push_back(dec_split); tval.push_back(nac); }
      }
    }
  }
  if (vcorner.size() > max_verts) return DCB_ERR_CONNECTIVITY;
  while (!stack.empty()) {  // start faces
    const uint32_t corner = stack.back();
    stack.pop_back();
    if (start_face.bit() & 1u) {
      if (num_faces >= n_faces) return DCB_ERR_CONNECTIVITY;
      const uint32_t vn = c2v[c_next(corner)];
      if (vn >= vcorner.size() || vcorner[vn] == INV) return DCB_ERR_CONNECTIVITY;
      const uint32_t cb = c_next(vcorner[vn]);
      const uint32_t vx = c2v[c_next(cb)];
      if (vx >= vcorner.size() || vcorner[vx] == INV) return DCB_ERR_CONNECTIVITY;
      const uint32_t cc = c_next(vcorner[vx]);
      if (corner == cb || corner == cc || cb == cc) return DCB_ERR_CONNECTIVITY;
      if (opp[corner] != INV || opp[cb] != INV || opp[cc] != INV) return DCB_ERR_CONNECTIVITY;
      const uint32_t vp = c2v[c_next(cc)];
      const uint32_t ncn = 3 * num_faces++;
      set_opp(ncn, corner);
      set_opp(ncn + 1, cb);
      set_opp(ncn + 2, cc);
      c2v[ncn] = vx; c2v[ncn + 1] = vp; c2v[ncn + 2] = vn;
      for (int k = 0; k < 3; ++k)
        if (c2v[ncn + k] < max_verts) is_vert_hole[c2v[ncn + k]] = 0;
    }
  }
  if (num_faces != n_faces) return DCB_ERR_CONNECTIVITY;
  uint32_t num_vertices = (uint32_t)vcorner.size();
  {
    const View bv = Base();
    for (uint32_t iv : invalid_verts) {
      uint32_t src = num_vertices - 1;
      while (vcorner[src] == INV) src = --num_vertices - 1;
      if (src < iv) continue;
      const uint32_t start = vcorner[src];
      uint32_t c = start;
      bool left = true;
      while (c != INV) {
        if (c2v[c] != src) return DCB_ERR_CONNECTIVITY;
        c2v[c] = iv;
        if (left) {
          c = bv.SwingLeft(c);
          if (c == INV) { c = bv.SwingRight(start); left = false; }
          else if (c == start) c = INV;
        } else {
          c = bv.SwingRight(c);
        }
      }
      vcorner[iv] = vcorner[src];
      vcorner[src] = INV;
      is_vert_hole[iv] = is_vert_hole[src];
      is_vert_hole[src] = 0;
      num_vertices--;
    }
  }
  n_points = num_vertices;
  // attribute seams
  att.assign(n_attr_data, AttrTable{});
  for (auto &a : att) a.edge_seam.assign(nc, 0);
  if (n_attr_data > 0) {
    for (uint32_t ci = 0; ci < nc; ci += 3) {
      const uint32_t corners[3] = {ci, c_next(ci), c_prev(ci)};
      for (int c = 0; c < 3; ++c) {
        const uint32_t oc = opp[corners[c]];
        if (oc == INV) {
          for (auto &a : att) a.edge_seam[corners[c]] = 1;
          continue;
        }
        if (oc / 3 < ci / 3) continue;
        for (uint32_t i = 0; i < n_attr_data; ++i)
          if (seams[i].bit()) { att[i].edge_seam[corners[c]] = 1; att[i].edge_seam[oc] = 1; }
      }
    }
    for (auto &a : att) BuildAttrTable(a);
  }
  AssignPoints();
  pos = r.pos;
  return DCB_OK;
}

// AssignPointsToCorners: :537-638
void EdgebreakerHost::AssignPoints() {
  const uint32_t nc = (uint32_t)c2v.size();
  faces.assign(nc, 0);
  if (att.empty()) {
    for (uint32_t c = 0; c < nc; ++c) faces[c] = c2v[c];
    return;
  }
  const View bv = Base();
  uint32_t np = 0;
  for (uint32_t v = 0; v < vcorner.size(); ++v) {
    uint32_t c = vcorner[v];
    if (c == INV) continue;
    uint32_t dedup_first = c;
    if (!is_vert_hole[v]) {
      for (auto &a : att) {
        if (!a.vert_seam[v]) continue;
        const uint32_t vid = a.c2v[c];
        uint32_t act = bv.SwingRight(c);
        bool found = false;
        while (act != c && act != INV) {
          if (a.c2v[act] != vid) { dedup_first = act; found = true; break; }
          act = bv.SwingRight(act);
        }
        if (found) break;
      }
    }
    c = dedup_first;
    faces[c] = np++;
    uint32_t prev_c = c;
    c = bv.SwingRight(c);
    while (c != INV && c != dedup_first) {
      bool seam = false;
      for (auto &a : att)
        if (a.c2v[c] != a.c2v[prev_c]) { seam = true; break; }
      faces[c] = seam ? np++ : faces[prev_c];
      prev_c = c;
      c = bv.SwingRight(c);
    }
  }
  n_points = np;
}

// MeshTraversalSequencer.GenerateSequenceInternal + DepthFirstTraverser.TraverseFromCorner + the observer
void EdgebreakerHost::Traverse(const View &t, uint32_t n_faces, std::vector<uint32_t> &d2c, std::vector<int32_t> &v2d) {
  std::vector<uint8_t> fvis(n_faces ? n_faces : 1, 0), vvis(t.n_vertices ? t.n_vertices : 1, 0);
  std::vector<uint32_t> stk;
  auto visit = [&](uint32_t v, uint32_t c) { vvis[v] = 1; v2d[v] = (int32_t)d2c.size(); d2c.push_back(c); };
  for (uint32_t f = 0; f < n_faces; ++f) {
    uint32_t corner = 3 * f;
    if (fvis[f]) continue;
    stk.clear();
    stk.push_back(corner);
    const uint32_t nv = t.Vertex(c_next(corner)), pv = t.Vertex(c_prev(corner));
    if (nv >= t.n_vertices || pv >= t.n_vertices) continue;
    if (!vvis[nv]) visit(nv, c_next(corner));
    if (!vvis[pv]) visit(pv, c_prev(corner));
    while (!stk.empty()) {
      corner = stk.back();
      uint32_t face = corner / 3;
      if (corner == INV || fvis[face]) { stk.pop_back(); continue; }
      for (;;) {
        fvis[face] = 1;
        const uint32_t v = t.Vertex(corner);
        if (v >= t.n_vertices) { stk.clear(); break; }
        if (!vvis[v]) {
          const bool on_b = t.OnBoundary(v);
          visit(v, corner);
          if (!on_b) {
            corner = t.RightCorner(corner);
            face = corner / 3;
            continue;
          }
        }
        const uint32_t rc = t.RightCorner(corner), lc = t.LeftCorner(corner);
        const bool rvis = rc == INV || fvis[rc / 3], lvis = lc == INV || fvis[lc / 3];
        if (rvis) {
          if (lvis) { stk.pop_back(); break; }
          corner = lc; face = lc / 3;
        } else {
          if (lvis) { corner = rc; face = rc / 3; }
          else { stk.back() = lc; stk.push_back(rc); break; }
        }
      }
    }
  }
}

int EdgebreakerHost::BuildMaps(const uint8_t *dec_ids, int n_dec, std::vector<DcbHostMaps> &maps) {
  maps.assign((size_t)n_dec, DcbHostMaps{});
  bool pos_used = false;
  std::vector<uint8_t> att_used(att.size(), 0);
  const uint32_t n_faces = (uint32_t)c2v.size() / 3;
  for (int d = 0; d < n_dec; ++d) {
    const int att_id = (int8_t)dec_ids[3 * d];
    const int dec_type = dec_ids[3 * d + 1], trav = dec_ids[3 * d + 2];
    if (trav >= 2) return DCB_ERR_CONNECTIVITY;
    if (att_id >= 0) {
      if ((size_t)att_id >= att.size() || att_used[att_id]) return DCB_ERR_CONNECTIVITY;
      att_used[att_id] = 1;
    } else {
      if (pos_used) return DCB_ERR_CONNECTIVITY;
      pos_used = true;
    }
    DcbHostMaps &m = maps[d];
    View t = Base();
    uint32_t n_map_verts = (uint32_t)vcorner.size();
    if (dec_type == 0) {  // vertex attribute: base corner table
      if (trav != 0) return DCB_ERR_UNSUPPORTED;
      if (att_id >= 0 && att[att_id].n_vertices > n_map_verts) n_map_verts = att[att_id].n_vertices;
      m.opposite = opp;
      m.corner_to_vertex = c2v;
    } else {  // corner attribute: the attribute's own corner table
      if (trav != 0 || att_id < 0) return DCB_ERR_CONNECTIVITY;
      const AttrTable &a = att[att_id];
      t = View{&a.opp, &a.c2v, &a.vleft, a.n_vertices};
      n_map_verts = a.n_vertices > vcorner.size() ? a.n_vertices : (uint32_t)vcorner.size();
      m.opposite = a.opp;
      m.corner_to_vertex = a.c2v;
    }
    m.vertex_to_data.assign(n_map_verts, 0);
    Traverse(t, n_faces, m.data_to_corner, m.vertex_to_data);
  }
  return DCB_OK;
}

}  // namespace

int dcb_host_edgebreaker(const uint8_t *buf, uint64_t len, uint64_t conn_off, uint64_t *attr_section_off,
                         uint32_t *n_points, std::vector<DcbHostMaps> *maps, std::vector<uint32_t> *faces) {
  // conn_off: first byte after the header (and metadata), i.e. the traversal-type byte (DracoDecoder.cs:80)
  if (conn_off >= len) return DCB_ERR_EOF;
  uint64_t pos = conn_off;
  const int traversal_type = buf[pos++];
  EdgebreakerHost eb;
  int st = eb.Decode(buf, len, pos, traversal_type);
  if (st) return st;
  // ATTRIBUTES: u8 n_dec, then n_dec x (att_data_id, decoder_type, traversal_method)
  if (pos >= len) return DCB_ERR_EOF;
  const int n_dec = buf[pos];
  if (len - pos - 1 < (uint64_t)3 * n_dec) return DCB_ERR_EOF;
  st = eb.BuildMaps(buf + pos + 1, n_dec, *maps);
  if (st) return st;
  *attr_section_off = pos;
  *n_points = eb.n_points;
  if (faces) faces->swap(eb.faces);
  return DCB_OK;
}

// ---------------------------------------------------------------------------------------------
// Sequential mesh connectivity (MeshSequentialDecoder.cs:8-118), v2.2: varint faces, varint points, u8 method, then
// either entropy-coded index differences (method 0, the symbol streams of SymbolDecoding.cs) or plain indices whose
// width follows the point count (method 1).  Host work like the Edgebreaker connectivity: the attributes behind it
// are sequential (LinearSequencer) and decode through the point-cloud kernels, no maps needed.
// Index differences: symbol >> 1 with the sign in bit 0, ODD = negative -- the bitstream's rule; the C# tests the
// bit the other way round (:97) and cannot decode an ordinary mesh (SURVEY Appendix B).  Its range checks are kept:
// an index may neither drop below zero (:99) nor pass int.MaxValue (:107).
int dcb_host_sequential(const uint8_t *buf, uint64_t len, uint64_t conn_off, uint64_t *attr_section_off, uint32_t *n_points,
                        std::vector<uint32_t> *faces, DcbSeqIndexLoc *loc) {
  Reader r{buf, len, conn_off};
  const uint64_t n_faces = r.varint();
  const uint64_t points = r.varint();
  const uint32_t method = r.u8();
  if (r.err) return r.err;
  if (n_faces > (1u << 28) || points > 0xFFFFFFFFull) return DCB_ERR_CONNECTIVITY;
  const uint64_t n_idx = 3 * n_faces;
  // counts the data cannot back fail this buffer before they size anything (as for the Edgebreaker counts)
  if (n_idx > 65536 + 4096 * (len - r.pos)) return DCB_ERR_CONNECTIVITY;
  std::vector<uint32_t> idx;
  if (method == 0) {
    if (loc) {
      loc->ckpt.clear();
      loc->n_idx = n_idx;
      loc->width = -1;
    }
    const int st = host_symbols(r, (uint32_t)n_idx, idx, loc && n_idx ? loc : nullptr);
    if (st) return st;
    if (loc && loc->located) {
      *attr_section_off = r.pos;
      *n_points = (uint32_t)points;
      return DCB_OK;
    }
    int64_t cur = 0;
    for (uint64_t i = 0; i < n_idx; ++i) {
      const int64_t step = (int64_t)(idx[i] >> 1);
      cur += (idx[i] & 1u) ? -step : step;
      if (cur < 0 || cur > 0x7FFFFFFFll) return DCB_ERR_CONNECTIVITY;
      idx[i] = (uint32_t)cur;
    }
  } else if (method == 1) {
    // bytes per index: 1, 2, varint (0) or 4
    const int width = points < 256 ? 1 : points < 65536 ? 2 : points < (1u << 21) ? 0 : 4;
    if (width && (len - r.pos) / (uint64_t)width < n_idx) return DCB_ERR_EOF;
    if (!width && len - r.pos < n_idx) return DCB_ERR_EOF;  // a varint is at least one byte
    if (loc) {
      // locate only: fixed widths by arithmetic; varints by their terminator bytes (bit 7 clear), with Reader::varint's
      // framing -- the run may not leave the buffer and a varint ends within 10 bytes
      loc->ckpt.clear();
      loc->n_idx = n_idx;
      loc->off = r.pos;
      loc->width = width;
      if (width) {
        r.pos += (uint64_t)width * n_idx;
      } else {
        // whole chunks branch-free (terminators counted, the longest continuation run tracked) while they cannot hold
        // the last index; the chunk that does, byte by byte to the exact end
        uint64_t ended = 0, run = 0;
        while (ended < n_idx) {
          if (r.pos >= len) return DCB_ERR_EOF;
          loc->ckpt.push_back(ended);
          const uint64_t n = std::min<uint64_t>(DCB_VARINT_CHUNK, len - r.pos);
          const uint8_t *c = buf + r.pos;
          uint64_t cnt = 0, worst = 0;
          for (uint64_t i = 0; i < n; ++i) {
            const uint64_t cont = c[i] >> 7;
            run = cont ? run + 1 : 0;
            worst = run > worst ? run : worst;
            cnt += cont ^ 1u;
          }
          if (ended + cnt < n_idx && worst < 10 && n == DCB_VARINT_CHUNK) {
            ended += cnt;
            r.pos += n;
            continue;
          }
          run = 0;  // redo this chunk exactly: the run in front of it ended at a terminator or is carried below
          for (uint64_t q = r.pos; q > loc->off && (buf[q - 1] & 0x80u); --q) ++run;
          for (uint64_t i = 0; i < n && ended < n_idx; ++i) {
            if (c[i] & 0x80u) {
              if (++run == 10) return DCB_ERR_EOF;
            } else {
              run = 0;
              ++ended;
            }
            ++r.pos;
          }
        }
      }
      loc->bytes = r.pos - loc->off;
      loc->located = true;
      *attr_section_off = r.pos;
      *n_points = (uint32_t)points;
      return DCB_OK;
    }
    idx.resize((size_t)n_idx);
    for (uint64_t i = 0; i < n_idx; ++i) {
      if (width == 0) {
        idx[i] = (uint32_t)r.varint();
      } else {
        uint32_t v = 0;
        for (int k = 0; k < width; ++k) v |= (uint32_t)buf[r.pos + k] << (8 * k);
        r.pos += (uint64_t)width;
        idx[i] = v;
      }
    }
    if (r.err) return r.err;
  } else {
    return DCB_ERR_CONNECTIVITY;  // :81
  }
  *attr_section_off = r.pos;
  *n_points = (uint32_t)points;
  if (faces) faces->swap(idx);
  return DCB_OK;
}
