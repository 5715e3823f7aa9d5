// Static tables of one env batch, built on the host from a pgw_spec (see tables.h).
#include "tables.h"

#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace pgw {
namespace {

int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Appends `bytes` at the next multiple of `align`; returns the offset relative to `base`.
int append(std::vector<unsigned char>& blob, const void* src, size_t bytes, size_t align, size_t base = 0) {
  const size_t off = (blob.size() + align - 1) / align * align;
  blob.resize(off + bytes, 0);
  if (bytes) memcpy(blob.data() + off, src, bytes);
  return (int)(off - base);
}

template <typename T>
int append(std::vector<unsigned char>& blob, const std::vector<T>& v, size_t align, size_t base = 0) {
  return append(blob, v.data(), v.size() * sizeof(T), align, base);
}

void pad_to(std::vector<unsigned char>& blob, size_t align) {
  blob.resize((blob.size() + align - 1) / align * align, 0);
}

// entries of the complex [nb][nb] Zbb and [nn][nb] Znb
double2 cplx(const double* m, size_t i) { return make_double2(m[2 * i], m[2 * i + 1]); }
double2 Zbb(const pgw_feeder& f, int k, int j) { return cplx(f.zbb, (size_t)k * f.nb + j); }
double2 Znb(const pgw_feeder& f, int n, int k) { return cplx(f.znb, (size_t)n * f.nb + k); }

// v = hi + lo in FP16, both rounded through float32
void split16(double v, __half* hi, __half* lo) {
  *hi = __float2half_rn((float)v);
  *lo = __float2half_rn((float)(v - (double)__half2float(*hi)));
}

// Operand images of the split-TF32 tcgen05 kernel (powerflow_tc.cu), byte-exact as they sit in
// shared memory: canonical K-major no-swizzle UMMA layout, element (row, k) at
//   (row/8)*3072 + (k/4)*128 + (row%8)*16 + (k%4)*4,   K = 96 = [hi | hi | lo] of B.
void build_tc_tables(const pgw_spec& s, FeederTables& out) {
  const pgw_feeder& f = *s.feeder;
  PfParams& p = out.base;
  const int nb = f.nb, nn = f.nn, A = s.num_agents;
  const int NB = kTcNb, K3 = kTcK3, nnp8 = round_up(nn, 8), n2 = 2 * nnp8;
  auto hi_of = [](double v) {
    float x = (float)v;
    uint32_t u;
    memcpy(&u, &x, 4);
    u &= 0xFFFFE000u;
    memcpy(&x, &u, 4);
    return x;
  };
  auto image = [&](int rows, const std::vector<double>& b /* [rows][32] */) {
    std::vector<unsigned char> img((size_t)rows * K3 * 4, 0);
    for (int r = 0; r < rows; ++r)
      for (int k = 0; k < 32; ++k) {
        const double v = b[(size_t)r * 32 + k];
        const float hi = hi_of(v), lo = (float)(v - (double)hi);
        const float part[3] = {hi, hi, lo};
        for (int q = 0; q < 3; ++q) {
          const int kc = q * 32 + k;
          const size_t off = (size_t)(r / 8) * 3072 + (size_t)(kc / 4) * 128 + (r % 8) * 16 + (kc % 4) * 4;
          memcpy(img.data() + off, &part[q], 4);
        }
      }
    return img;
  };
  // D[e][n] = sum_k X[e][k] B[n][k],  X = [Re i (16) | Im i (16)],  D = [Re du (16) | Im du (16)]
  std::vector<double> b1((size_t)32 * 32, 0.0), b2((size_t)n2 * 32, 0.0);
  for (int k = 0; k < nb; ++k)
    for (int j = 0; j < nb; ++j) {
      const double2 z = Zbb(f, k, j);
      b1[(size_t)k * 32 + j] = -z.x;            // Re du_k -= Zr Re i_j
      b1[(size_t)k * 32 + NB + j] = z.y;        //           + Zi Im i_j
      b1[(size_t)(NB + k) * 32 + j] = -z.y;     // Im du_k -= Zi Re i_j
      b1[(size_t)(NB + k) * 32 + NB + j] = -z.x;  //         - Zr Im i_j
    }
  for (int n = 0; n < nn; ++n)                  // rows interleaved: 2n = Re dv_n, 2n+1 = Im dv_n
    for (int k = 0; k < nb; ++k) {
      const double2 z = Znb(f, n, k);
      b2[(size_t)(2 * n) * 32 + k] = -z.x;
      b2[(size_t)(2 * n) * 32 + NB + k] = z.y;
      b2[(size_t)(2 * n + 1) * 32 + k] = -z.y;
      b2[(size_t)(2 * n + 1) * 32 + NB + k] = -z.x;
    }
  std::vector<unsigned char>& blob = out.tc_blob;
  append(blob, image(32, b1), 128);
  p.tc_off_b2 = append(blob, image(n2, b2), 128);
  std::vector<float> u0f(2 * NB, 0.f), wf(2 * nnp8, 0.f), vlf(NB, 0.95f), vhf(NB, 1.05f);
  std::vector<double> shd(NB, 0.0);
  std::vector<int32_t> bl16(NB, 0), bm16(NB, 1), slot(A), node(A);
  for (int k = 0; k < NB; ++k) { u0f[2 * k] = 1.f; }
  for (int k = 0; k < nb; ++k) {
    u0f[2 * k] = (float)f.u0[2 * k]; u0f[2 * k + 1] = (float)f.u0[2 * k + 1];
    vlf[k] = (float)f.vminpu[k]; vhf[k] = (float)f.vmaxpu[k]; shd[k] = f.branch_share[k];
    bl16[k] = f.branch_load[k]; bm16[k] = f.branch_model[k];
  }
  for (int n = 0; n < nn; ++n) { wf[2 * n] = (float)f.w[2 * n]; wf[2 * n + 1] = (float)f.w[2 * n + 1]; }
  for (int a = 0; a < A; ++a) { slot[a] = s.agents[a].load_slot; node[a] = s.agents[a].bus_node; }
  p.tc_off_u0 = append(blob, u0f, 128);
  p.tc_off_w = append(blob, wf, 128);
  p.tc_off_share = append(blob, shd, 128);
  p.tc_off_vlo = append(blob, vlf, 128);
  p.tc_off_vhi = append(blob, vhf, 128);
  p.tc_off_bload = append(blob, bl16, 128);
  p.tc_off_bmodel = append(blob, bm16, 128);
  p.tc_off_slot = append(blob, slot, 128);
  p.tc_off_node = append(blob, node, 128);
  pad_to(blob, 128);
  p.tc_blob_bytes = (int)blob.size();
  p.tc_n2 = n2; p.tc_nnp8 = nnp8;
}

// Operand images and tables of the FP16 tcgen05 kernel (powerflow_tc2.cu) for a tile of nch
// chunks of 8 load branches, and the fused step kernel's section behind them (step_fused.cu).
void build_tc2_tables(const pgw_spec& s, int nch, FeederTables& out) {
  const pgw_feeder& f = *s.feeder;
  Tc2Params& t = out.base.tc2;
  const int nb = f.nb, nn = f.nn, A = s.num_agents;
  const double punit = f.penalty_unit;
  // Images byte-exact as they sit in shared memory: canonical K-major no-swizzle UMMA tiles,
  // element (row, k) of an image with K columns at  (row/8)*SBO + (k/8)*128 + (row%8)*16 + (k%8)*2,
  // SBO = (K/8)*128.  Row / column order: 16c + j = Re (j < 8) or Im (j >= 8) of item 8c + (j % 8).
  const int N = 16 * nch, NBP = 8 * nch;
  const size_t sbo = (size_t)(N / 8) * 128, part = (size_t)(N / 8) * sbo;
  auto pos = [](int item, bool im) { return 16 * (item / 8) + (item % 8) + (im ? 8 : 0); };
  // Nodes whose voltage IS a load-branch voltage up to a real factor c (a wye load between
  // the node and ground: row n of Znb = c x row k of Zbb and w[n] = c u0[k], c = the ratio
  // of the two voltage bases) need no expansion: |v_n| = c |u_k|.
  std::vector<int32_t> dnode(NBP, -1), xnode;
  std::vector<float> dscale(NBP, 0.f);
  std::vector<double> dscale64(NBP, 0.0);
  {
    std::vector<char> taken(nb, 0);
    for (int n = 0; n < nn; ++n) {
      int hit = -1;
      double cr = 0.0;
      for (int k = 0; k < nb && hit < 0; ++k) {
        if (taken[k]) continue;
        const double ur = f.u0[2 * k], ui = f.u0[2 * k + 1], wr = f.w[2 * n], wi = f.w[2 * n + 1];
        const double den = ur * ur + ui * ui;
        if (den <= 0.0) continue;
        const double c = (wr * ur + wi * ui) / den;
        if (!(c > 0.0)) continue;
        double err = std::hypot(wr - c * ur, wi - c * ui), ref = std::hypot(wr, wi);
        for (int j = 0; j < nb; ++j) {
          const double2 a = Znb(f, n, j), b = Zbb(f, k, j);
          err = std::fmax(err, std::hypot(a.x - c * b.x, a.y - c * b.y));
          ref = std::fmax(ref, std::hypot(a.x, a.y));
        }
        if (err <= 1e-10 * ref) { hit = k; cr = c; }
      }
      if (hit >= 0) { taken[hit] = 1; dnode[hit] = n; dscale[hit] = (float)cr; dscale64[hit] = cr; }
      else xnode.push_back(n);
    }
  }
  auto branch_of = [&](int nd) {                  // the load branch whose wye node is nd, or -1
    for (int k = 0; k < nb; ++k)
      if (nd >= 0 && dnode[k] == nd) return k;
    return -1;
  };
  const int nx = (int)xnode.size(), ncc = (nx + NBP - 1) / NBP;
  xnode.resize((size_t)std::max(ncc, 1) * NBP, -1);
  auto zx = [&](int slot, int k) { return Znb(f, xnode[slot], k); };   // Znb of the expansion slots
  auto zb = [&](int k, int j) { return Zbb(f, k, j); };
  // real-ified operator rows:  D[pos(out)] = sum_k X[pos(k)] * M[pos(out)][pos(k)]
  auto realify = [&](int item0, int nitems, auto&& zget) {
    std::vector<double> m((size_t)N * N, 0.0);
    for (int r = 0; r < NBP; ++r) {
      const int item = item0 + r;
      if (item >= nitems) break;
      for (int k = 0; k < nb; ++k) {
        const double2 z = zget(item, k);
        m[(size_t)pos(r, false) * N + pos(k, false)] = -z.x;   // Re out -= Zr Re i
        m[(size_t)pos(r, false) * N + pos(k, true)] = z.y;     //         + Zi Im i
        m[(size_t)pos(r, true) * N + pos(k, false)] = -z.y;    // Im out -= Zi Re i
        m[(size_t)pos(r, true) * N + pos(k, true)] = -z.x;     //         - Zr Im i
      }
    }
    return m;
  };
  // the power of two that takes the largest entry into [8192, 16384)
  auto scale_for = [](double mx) {
    return mx > 0.0 ? std::ldexp(1.0, (int)std::floor(std::log2(16384.0 / mx))) : 1.0;
  };
  auto images = [&](const std::vector<double>& m, double scale, unsigned char* dst) {
    for (int r = 0; r < N; ++r)
      for (int k = 0; k < N; ++k) {
        __half hi, lo;
        split16(m[(size_t)r * N + k] * scale, &hi, &lo);
        const size_t off = (size_t)(r / 8) * sbo + (size_t)(k / 8) * 128 + (r % 8) * 16 + (k % 8) * 2;
        memcpy(dst + off, &hi, 2);
        memcpy(dst + part + off, &lo, 2);
      }
  };
  double mx1 = 0.0, mx2 = 0.0;
  for (size_t i = 0; i < 2 * (size_t)nb * nb; ++i) mx1 = std::fmax(mx1, std::fabs(f.zbb[i]));
  for (size_t i = 0; i < 2 * (size_t)nn * nb; ++i) mx2 = std::fmax(mx2, std::fabs(f.znb[i]));
  const double sb1 = scale_for(mx1), sb2 = scale_for(mx2), xs = 2048.0;
  std::vector<unsigned char>& blob = out.tc2_blob;
  blob.assign((size_t)(1 + ncc) * 2 * part, 0);
  images(realify(0, nb, zb), sb1, blob.data());
  for (int cc = 0; cc < ncc; ++cc)
    images(realify(cc * NBP, nx, zx), sb2, blob.data() + (size_t)(1 + cc) * 2 * part);
  t.nch = nch; t.ncc = ncc; t.nx = nx; t.part_bytes = (int)part; t.off_zn = (int)(2 * part);
  t.off_tab = (int)blob.size();
  t.xscale = (float)xs; t.descale1 = (float)(1.0 / (sb1 * xs)); t.descale2 = (float)(1.0 / (sb2 * xs));
  // small feeders keep every Znb chunk resident (64 kB of images, accumulators 2 + cc)
  t.resident = ((2 + ncc) * N <= 512 && (size_t)ncc * 2 * part <= 64 * 1024) ? 1 : 0;
  t.tmem_cols = 32;
  while (t.tmem_cols < (t.resident ? 2 + ncc : 2) * N) t.tmem_cols *= 2;
  // cst = {Re u0, Im u0, vlo^2, vhi^2}, gh = (1, 0) -> 1/clamp(|u|^2), (0, 1) -> 1/|u| (model 5)
  std::vector<float> cst(4 * (size_t)NBP, 1.f), gh(2 * (size_t)NBP, 0.f), shf(NBP, 0.f), wf(2 * xnode.size(), 0.f);
  std::vector<int32_t> blp(NBP, 0), bag(NBP, -1), lptr(f.nl + 1, 0), lidx(A, 0), node(A);
  for (int k = 0; k < NBP; ++k) { cst[4 * k + 1] = 0.f; gh[2 * k] = 1.f; }
  for (int k = 0; k < nb; ++k) {
    cst[4 * k] = (float)f.u0[2 * k]; cst[4 * k + 1] = (float)f.u0[2 * k + 1];
    if (f.branch_model[k] == 5) {
      cst[4 * k + 2] = 1e-30f; cst[4 * k + 3] = 3e38f; gh[2 * k] = 0.f; gh[2 * k + 1] = 1.f;
      t.any_m5 = 1;
    } else if (f.branch_model[k] != 2) {
      cst[4 * k + 2] = (float)(f.vminpu[k] * f.vminpu[k]);
      cst[4 * k + 3] = (float)(f.vmaxpu[k] * f.vmaxpu[k]);
    }
    shf[k] = (float)(f.branch_share[k] * 1e-3);
    blp[k] = f.branch_load[k];
  }
  for (int sidx = 0; sidx < nx; ++sidx) {
    wf[2 * sidx] = (float)f.w[2 * xnode[sidx]]; wf[2 * sidx + 1] = (float)f.w[2 * xnode[sidx] + 1];
  }
  for (int a = 0; a < A; ++a) {
    node[a] = s.agents[a].bus_node;
    if (s.agents[a].load_slot >= 0) ++lptr[s.agents[a].load_slot + 1];
  }
  for (int l = 0; l < f.nl; ++l) lptr[l + 1] += lptr[l];
  {
    std::vector<int32_t> fill(lptr.begin(), lptr.end() - 1);
    for (int a = 0; a < A; ++a)                   // agent order inside a load slot
      if (s.agents[a].load_slot >= 0) lidx[fill[s.agents[a].load_slot]++] = a;
  }
  for (int k = 0; k < nb; ++k) {                  // the one agent on the branch's load, or -2
    const int l = blp[k], cnt = lptr[l + 1] - lptr[l];
    bag[k] = cnt == 0 ? -1 : (cnt == 1 ? lidx[lptr[l]] : -2);
  }
  for (int q = 0; q < NBP / 2; ++q) {            // pairs of branches (2q, 2q + 1)
    const int k0 = 2 * q, k1 = 2 * q + 1;
    out.tc2c.pa[q] = make_float4(cst[4 * k0], cst[4 * k1], cst[4 * k0 + 1], cst[4 * k1 + 1]);
    out.tc2c.pb[q] = make_float4(cst[4 * k0 + 2], cst[4 * k1 + 2], cst[4 * k0 + 3], cst[4 * k1 + 3]);
    out.tc2c.pc[q] = make_float4(gh[2 * k0], gh[2 * k1], gh[2 * k0 + 1], gh[2 * k1 + 1]);
  }
  const size_t tab = (size_t)t.off_tab;
  t.t_share = append(blob, shf, 16, tab);
  t.t_bload = append(blob, blp, 16, tab);
  t.t_bagent = append(blob, bag, 16, tab);
  t.t_w = append(blob, wf, 16, tab);
  t.t_xnode = append(blob, xnode, 16, tab);
  t.t_dnode = append(blob, dnode, 16, tab);
  t.t_dscale = append(blob, dscale, 16, tab);
  // FP64 polish (powerflow_tc2.cu): one full float64 sweep + one over the rows the rewards
  // and the agents read, on by default where the rewards read the fresh voltages
  t.polish_ok = nch == 2 ? 1 : 0;
  t.polish = (t.polish_ok && punit != 0.0) ? 1 : 0;
  t.tol = tc2_default_tol(f.tol, t.polish);
  t.polish_row = -1;
  if (t.polish_ok) {
    Tc2Polish& kp = out.tc2p;
    for (int j = 0; j < 16; ++j)
      for (int k = 0; k < 16; ++k) {
        kp.zT[j * 16 + k] = (j < nb && k < nb) ? Zbb(f, k, j) : make_double2(0.0, 0.0);
        kp.z32[j * 16 + k] = make_float2((float)(kp.zT[j * 16 + k].x / xs), (float)(kp.zT[j * 16 + k].y / xs));
      }
    for (int k = 0; k < 16; ++k) {
      const bool real = k < nb;
      kp.u0[k] = real ? make_double2(f.u0[2 * k], f.u0[2 * k + 1]) : make_double2(1.0, 0.0);
      kp.share[k] = real ? f.branch_share[k] * 1e-3 : 0.0;
      kp.model[k] = real ? f.branch_model[k] : 1;
      const bool z = real && f.branch_model[k] == 2;
      kp.vlo2[k] = z ? 1.0 : (real ? f.vminpu[k] * f.vminpu[k] : 0.9025);
      kp.vhi2[k] = z ? 1.0 : (real ? f.vmaxpu[k] * f.vmaxpu[k] : 1.1025);
      kp.dscale[k] = real ? dscale64[k] : 0.0;
    }
    kp.rows = 0u;
    for (int a = 0; a < A; ++a)
      if (branch_of(node[a]) >= 0) kp.rows |= 1u << branch_of(node[a]);
    if (punit != 0.0 && branch_of(f.penalty_node) >= 0) kp.rows |= 1u << branch_of(f.penalty_node);
    else if (punit != 0.0) t.polish_row = f.penalty_node;
  }
  t.t_lptr = append(blob, lptr, 16, tab);
  t.t_lidx = append(blob, lidx, 16, tab);
  t.t_anode = append(blob, node, 16, tab);
  {
    // up to two agents per branch whose bus node derives from it (vag); the others (more
    // than two on a node, or a bus that is not a wye-load node) go to the tail list
    std::vector<int32_t> vag(2 * (size_t)NBP, -1), vtail;
    for (int a = 0; a < A; ++a) {
      const int k = branch_of(node[a]);
      if (k >= 0 && vag[2 * k] < 0) vag[2 * k] = a;
      else if (k >= 0 && vag[2 * k + 1] < 0) vag[2 * k + 1] = a;
      else vtail.push_back(a);
    }
    t.ntail = (int)vtail.size();
    vtail.push_back(0);
    t.t_vag = append(blob, vag, 16, tab);
    t.t_vtail = append(blob, vtail, 16, tab);
  }
  pad_to(blob, 16);
  t.tab_bytes = (int)(blob.size() - tab);
  t.off_ftab = (int)blob.size(); t.ftab_bytes = 0; t.pen_slot = -1;
  if (!t.polish_ok) return;
  // the fused step kernel's own section
  const size_t ftab = (size_t)t.off_ftab;
  std::vector<int32_t> aslot(std::max(A, 1), -1);
  for (int a = 0; a < A; ++a) aslot[a] = branch_of(node[a]);
  if (punit != 0.0) t.pen_slot = branch_of(f.penalty_node);
  t.f_kc = append(blob, &out.tc2c, sizeof(out.tc2c), 16, ftab);
  t.f_kp = append(blob, &out.tc2p, sizeof(out.tc2p), 16, ftab);
  t.f_aslot = append(blob, aslot, 16, ftab);
  // B fragments of the fused kernel's mma.sync.m16n8k16 products: the realified operator
  // (rows: outputs, columns: the 16 branch currents) x scale, split into FP16 hi / lo as
  // images() does, with (Re, Im) interleaved per item along N (the outputs) and K (the
  // currents): n-tile j = outputs 4j .. 4j + 3.  In the order the registers take them:
  // [n-tile][lane][k-step][hi b0, hi b1, lo b0, lo b1], two 16-byte loads a lane.
  auto mma_frags = [&](std::vector<uint16_t>& bf, int ntiles, int nitems, double scale, auto&& zget) {
    const size_t base = bf.size();
    bf.resize(base + (size_t)ntiles * 32 * 2 * 4 * 2, 0);
    for (int j = 0; j < ntiles; ++j)
      for (int lane = 0; lane < 32; ++lane) {
        const int g = lane >> 2, tq = lane & 3;
        const int r = 4 * j + g / 2;               // output item of column 8j + g
        const bool im_out = (g & 1) != 0;
        for (int st = 0; st < 2; ++st)
          for (int reg = 0; reg < 2; ++reg)
            for (int ii = 0; ii < 2; ++ii) {       // the two halves: Re / Im of current q
              const int q = 8 * st + tq + 4 * reg;
              const double2 z = (r < nitems && q < nb) ? zget(r, q) : make_double2(0.0, 0.0);
              __half hi, lo;
              split16((im_out ? (ii ? -z.x : -z.y) : (ii ? z.y : -z.x)) * scale, &hi, &lo);
              const size_t o = base + ((((size_t)j * 32 + lane) * 2 + st) * 4 + reg) * 2 + ii;
              memcpy(&bf[o], &hi, 2);
              memcpy(&bf[o + 4], &lo, 2);
            }
      }
  };
  // f_xz: 4 n-tiles of the fixed point's drops (Zbb x sb1), then 4 per chunk of 16 slots of
  // the expansion's node voltages (Znb of the expansion slots x sb2)
  std::vector<uint16_t> bf;
  mma_frags(bf, 4, nb, sb1, zb);
  mma_frags(bf, 4 * ncc, nx, sb2, zx);
  t.f_xz = append(blob, bf, 16, ftab);
  pad_to(blob, 16);
  t.ftab_bytes = (int)(blob.size() - ftab);
}

}  // namespace

// Convergence threshold max|d drop| (p.u.) of the tcgen05 fixed point.  The float32 iteration cannot
// resolve less than ~1e-7.  Where the float64 polish follows (its two sweeps contract whatever the loop
// leaves behind by > 100x for the voltages the rewards read) the loop stops at 1e-6: one iteration
// less per solve, rewards and voltages unchanged within their bounds (measured over 2.3 M env-steps:
// worst reward error 0.093 of the bound against 0.089 at 1e-7, node voltages 2.3e-7 p.u. either way;
// tools/reward_margin.py).  OpenDSS's own convergence tolerance is 1e-4.
float tc2_default_tol(double solver_tol, int polish) {
  const double floor_tol = polish > 0 ? 1e-6 : 1e-7;
  return (float)(solver_tol > floor_tol ? solver_tol : floor_tol);
}

std::string validate_spec(const pgw_spec& s) {
  if (s.abi_version != PGW_ABI_VERSION) return "ABI version mismatch";
  if (s.num_envs <= 0 || s.num_agents <= 0 || s.num_components <= 0 || s.num_events <= 1)
    return "empty spec";
  if (s.dtab_stride % 2 || s.itab_stride % 4) return "event rows must be multiples of 16 bytes";
  if (s.num_agents > 65535) return "too many agents";
  for (int a = 0; a < s.num_agents; ++a) {
    const pgw_agent& ag = s.agents[a];
    if (ag.comp_begin < 0 || ag.comp_end > s.num_components || ag.comp_begin >= ag.comp_end)
      return "agent component range out of bounds";
    if (ag.load_slot >= 0 && (!s.feeder || ag.load_slot >= s.feeder->nl)) return "agent load slot out of range";
    if (ag.bus_node >= 0 && (!s.feeder || ag.bus_node >= s.feeder->nn)) return "agent bus node out of range";
  }
  for (int c = 0; c < s.num_components; ++c) {
    const pgw_component& k = s.components[c];
    if (k.type < PGW_STORAGE || k.type > PGW_HS_DEVICES) return "unknown component type (no CPU fallback exists)";
    if (k.obs_off < 0 || k.obs_off + k.obs_dim > s.obs_dim || k.act_off < 0 || k.act_off >= s.act_dim ||
        k.dpar_off < 0 || k.dpar_off > s.dpar_len || k.ipar_off < 0 || k.ipar_off > s.ipar_len)
      return "component offsets out of range";
    // rows each component kind reads and writes (layouts in include/pgw.h): a spec that is off
    // by a row must come back as PGW_ERR_INVALID, not as an out-of-bounds access on the device
    auto ip = [&](int i) { return k.ipar_off + i < s.ipar_len ? s.ipar[k.ipar_off + i] : -1; };
    const bool tel = (k.flags & PGW_F_TELEMETRY) != 0;
    int act = 1, obs_min = 1, sd = 0, si = 0, dw = 0, iw = 0;
    switch (k.type) {
      case PGW_STORAGE: sd = 1; break;
      case PGW_PV: obs_min = (k.flags & PGW_F_GRID_AWARE) ? 2 : 1; dw = 1; break;
      case PGW_EV: case PGW_HS_EV: {
        const int n = ip(0), words = ip(1), cap = ip(2);
        if (k.flags & PGW_F_EV_PER_ENV) {            // per-env rosters: window words behind the mask
          if (k.type != PGW_EV || n <= 0 || n > 256 || words != (n + 31) / 32)
            return "EV station with per-env rosters: stock station, 1..256 vehicles, ipar = n, ceil(n/32), 0";
          obs_min = 6; sd = n; si = words + n; dw = 2; iw = 0;
          break;
        }
        if (n <= 0 || words != (n + 31) / 32 || cap <= 0)
          return "EV station: ipar must hold n, ceil(n/32), list capacity";
        obs_min = k.type == PGW_EV ? 6 : 7;
        sd = n + (k.type == PGW_HS_EV ? 1 : 0); si = words; dw = 2 + 2 * cap; iw = 2 + 2 * cap;
        break;
      }
      case PGW_BUILDING: act = 6; sd = 6; dw = 17; break;
      case PGW_HS_BEGIN: act = 0; obs_min = 0; sd = 5; dw = 1; break;
      case PGW_HS_PV: dw = 1; break;
      case PGW_HS_STORAGE: obs_min = 2; sd = 2; break;
      case PGW_HS_DEVICES: {
        const int cols = ip(0);
        if (cols <= 0) return "devices: ipar must hold the column count";
        obs_min = cols; dw = 2 * cols;
        break;
      }
      default: break;
    }
    if (tel && k.type >= PGW_HS_PV) sd += PGW_HS_TEL_ROWS;
    if (k.act_off + act > s.act_dim) return "component action rows out of range";
    if (k.obs_dim < obs_min) return "component observation rows: fewer than the kind writes";
    if (k.sd_off < 0 || k.sd_off + sd > s.sd_rows || k.si_off < 0 || k.si_off + si > s.si_rows)
      return "component state rows out of range";
    if (k.dtab_off < 0 || k.dtab_off + dw > s.dtab_stride || k.itab_off < 0 || k.itab_off + iw > s.itab_stride)
      return "component event-row block out of range";
    if (!s.feeder && (k.flags & (PGW_F_GRID_AWARE | PGW_F_PV_VOLT_REWARD)))
      return "grid-aware component without a feeder";
    if (k.type == PGW_BUILDING && (k.flags & PGW_F_BUILDING_FAST) && k.obs_dim != 15)
      return "PGW_F_BUILDING_FAST requires the 15-entry observation set";
  }
  return "";
}

CompTables build_comp_tables(const pgw_spec& s, int cta_budget) {
  CompTables out;
  CompParams& p = out.base;
  const int A = s.num_agents, C = s.num_components;
  p.E = s.num_envs; p.A = A; p.e_lo = 0; p.e_hi = s.num_envs;
  p.dstride = s.dtab_stride; p.istride = s.itab_stride;
  for (int c = 0; c < C; ++c) {
    const pgw_component& k = s.components[c];
    if (k.type == PGW_HS_BEGIN) p.has_house = std::max(p.has_house, 1);
    if (k.type >= PGW_HS_PV && (k.flags & PGW_F_TELEMETRY)) p.has_house = 2;
    if (k.flags & PGW_F_EV_PER_ENV) p.ev_per_env = 1;
    if (k.type == PGW_BUILDING) {
      out.need_scratch_reset = true;                 // reset always takes the table-driven path
      if (!(k.flags & PGW_F_BUILDING_FAST)) out.need_scratch = true;
    }
  }
  // static component tables as one blob, staged to shared memory by every CTA
  std::vector<unsigned char>& blob = out.blob;
  append(blob, s.agents, (size_t)A * sizeof(pgw_agent), 16);
  p.off_comps = append(blob, s.components, (size_t)C * sizeof(pgw_component), 16);
  p.off_dpar = append(blob, s.dpar, (size_t)s.dpar_len * sizeof(double), 16);
  p.off_ipar = append(blob, s.ipar, (size_t)s.ipar_len * sizeof(int32_t), 16);
  pad_to(blob, 16);
  p.blob_bytes = (int)blob.size();
  // per-agent slices: components [begin, end), and the span of their parameter blocks (a
  // block ends where the next larger offset of any component starts)
  std::vector<int> dstart, istart;
  for (int c = 0; c < C; ++c) {
    dstart.push_back(s.components[c].dpar_off);
    istart.push_back(s.components[c].ipar_off);
  }
  dstart.push_back(s.dpar_len); istart.push_back(s.ipar_len);
  std::sort(dstart.begin(), dstart.end()); std::sort(istart.begin(), istart.end());
  auto block_end = [](const std::vector<int>& starts, int off) {
    return *std::upper_bound(starts.begin(), starts.end(), off);
  };
  std::vector<AgentSlice> sl(A);
  for (int a = 0; a < A; ++a) {
    const pgw_agent& ag = s.agents[a];
    int dlo = s.dpar_len, dhi = 0, ilo = s.ipar_len, ihi = 0;
    for (int c = ag.comp_begin; c < ag.comp_end; ++c) {
      const pgw_component& k = s.components[c];
      if (k.dpar_off < s.dpar_len) {
        dlo = std::min(dlo, k.dpar_off); dhi = std::max(dhi, block_end(dstart, k.dpar_off));
      }
      if (k.ipar_off < s.ipar_len) {
        ilo = std::min(ilo, k.ipar_off); ihi = std::max(ihi, block_end(istart, k.ipar_off));
      }
    }
    if (dhi <= dlo) dlo = dhi = 0;
    if (ihi <= ilo) ilo = ihi = 0;
    AgentSlice& x = sl[a];
    x.c_lo = ag.comp_begin; x.c_n = ag.comp_end - ag.comp_begin;
    x.d_lo = dlo / 2 * 2; x.d_n = round_up(dhi - x.d_lo, 2);
    x.i_lo = ilo / 4 * 4; x.i_n = round_up(ihi - x.i_lo, 4);
    x.pad0 = x.pad1 = 0;
    p.max_cn = std::max(p.max_cn, x.c_n);
    p.max_dn = std::max(p.max_dn, x.d_n);
    p.max_in = std::max(p.max_in, x.i_n);
  }
  // The budget is split over the agents in proportion to a cost estimate of their components
  // (rough time per 64-env block), every agent between 1 CTA and one CTA per 64-env block.
  const int blocks = (s.num_envs + 63) / 64;
  std::vector<double> w(A, 0.5);                 // ~us per env block: loop + latency floor
  double wsum = 0.0;
  for (int a = 0; a < A; ++a) {
    for (int c = s.agents[a].comp_begin; c < s.agents[a].comp_end; ++c) {
      const pgw_component& k = s.components[c];
      switch (k.type) {
        case PGW_BUILDING: w[a] += 2.0; break;
        case PGW_EV: case PGW_HS_EV: w[a] += 1.0 + 0.04 * s.ipar[k.ipar_off]; break;
        case PGW_STORAGE: w[a] += 0.8; break;
        case PGW_HS_BEGIN: case PGW_HS_STORAGE: case PGW_HS_DEVICES: w[a] += 1.0; break;
        default: w[a] += 0.5; break;
      }
    }
    wsum += w[a];
  }
  // water-filling: agents that reach one CTA per block give their surplus to the others
  std::vector<int> n(A, 0);
  {
    std::vector<char> capped(A, 0);
    double left = cta_budget, wleft = wsum;
    for (bool again = true; again;) {
      again = false;
      for (int a = 0; a < A; ++a)
        if (!capped[a] && left * w[a] / wleft >= blocks) {
          capped[a] = 1; n[a] = blocks; left -= blocks; wleft -= w[a]; again = true;
        }
    }
    for (int a = 0; a < A; ++a)
      if (!capped[a]) n[a] = std::max(1, std::min(blocks, (int)std::ceil(left * w[a] / wleft)));
  }
  std::vector<int> order(A);
  for (int a = 0; a < A; ++a) order[a] = a;
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return w[x] > w[y]; });
  // longest-processing-time-first: every CTA of the heaviest agent, then the next agent, ...
  // so that the long-running CTAs are all resident from the start and the light ones fill in
  // behind them (with round-robin emission half of an EV station's CTAs started a wave late)
  for (int a : order)
    for (int j = 0; j < n[a]; ++j) out.work.push_back(CtaWork{a, j, n[a], 0, sl[a]});
  p.num_ctas = (int)out.work.size();
  p.tickets = (unsigned int)p.num_ctas;
  return out;
}

int comp_staging_bytes(const CompParams& p) {
  return p.max_cn * (int)sizeof(pgw_component) + p.max_dn * 8 + p.max_in * 4 + p.dstride * 8 + p.istride * 4;
}

FeederTables build_feeder_tables(const pgw_spec& s, int tc2_nch) {
  FeederTables out;
  const pgw_feeder& f = *s.feeder;
  if (f.nb <= 0 || f.nn <= 0 || f.nl <= 0 || f.nb > 128 || f.max_iter <= 0)
    out.error = "feeder dimensions out of range (1..128 load branches)";
  else if (s.dtab_stride < 2 + 2 * f.nl)
    out.error = "event row too short for the feeder base loads";
  else if (f.penalty_unit != 0.0 && (f.penalty_node < 0 || f.penalty_node >= f.nn))
    out.error = "penalty node out of range";
  else
    for (int k = 0; k < f.nb && out.error.empty(); ++k)
      if (f.branch_load[k] < 0 || f.branch_load[k] >= f.nl) out.error = "branch load index out of range";
  if (!out.error.empty()) return out;
  PfParams& p = out.base;
  const int nb = f.nb, nn = f.nn, A = s.num_agents;
  p.E = s.num_envs; p.A = A; p.e_lo = 0; p.e_hi = s.num_envs;
  p.nb = nb; p.nn = nn; p.nl = f.nl; p.max_iter = f.max_iter; p.tol = f.tol;
  p.nbp = nb <= 16 ? 16 : round_up(nb, 32);
  p.nnp = round_up(nn, 2);
  p.penalty_node = f.penalty_node; p.pvlo = f.penalty_vlo; p.pvhi = f.penalty_vhi; p.punit = f.penalty_unit;
  p.dstride = s.dtab_stride;
  p.tc_tol = (float)(f.tol > 1e-7 ? f.tol : 1e-7);
  const int nbp = p.nbp, nnp = p.nnp;
  std::vector<double2> zt((size_t)nb * nbp, make_double2(0, 0)), u0(nbp, make_double2(1, 0)),
      znt((size_t)nb * nnp, make_double2(0, 0)), w(nnp, make_double2(0, 0));
  for (int k = 0; k < nb; ++k)
    for (int j = 0; j < nb; ++j) zt[(size_t)j * nbp + k] = Zbb(f, k, j);
  for (int k = 0; k < nb; ++k) u0[k] = make_double2(f.u0[2 * k], f.u0[2 * k + 1]);
  for (int n = 0; n < nn; ++n) {
    w[n] = make_double2(f.w[2 * n], f.w[2 * n + 1]);
    for (int k = 0; k < nb; ++k) znt[(size_t)k * nnp + n] = Znb(f, n, k);
  }
  std::vector<int32_t> bl(nbp, 0), bm(nbp, 1), slot(A), node(A);
  std::vector<double> bs(nbp, 0.0), vlo(nbp, 0.95), vhi(nbp, 1.05);
  for (int k = 0; k < nb; ++k) {
    bl[k] = f.branch_load[k]; bm[k] = f.branch_model[k]; bs[k] = f.branch_share[k];
    vlo[k] = f.vminpu[k]; vhi[k] = f.vmaxpu[k];
  }
  for (int a = 0; a < A; ++a) { slot[a] = s.agents[a].load_slot; node[a] = s.agents[a].bus_node; }
  std::vector<unsigned char>& blob = out.blob;
  append(blob, zt, 16);
  p.off_u0 = append(blob, u0, 16);
  p.off_znbT = append(blob, znt, 16);
  p.off_w = append(blob, w, 16);
  p.off_share = append(blob, bs, 16);
  p.off_vmin = append(blob, vlo, 16);
  p.off_vmax = append(blob, vhi, 16);
  p.off_bload = append(blob, bl, 16);
  p.off_bmodel = append(blob, bm, 16);
  p.off_slot = append(blob, slot, 16);
  p.off_node = append(blob, node, 16);
  pad_to(blob, 16);
  p.blob_bytes = (int)blob.size();
  p.stage_blob = p.blob_bytes <= 96 * 1024 ? 1 : 0;   // else read through L1/L2
  if (nb <= kTcNb && 32 + 2 * round_up(nn, 8) <= 128) build_tc_tables(s, out);
  if (tc2_nch > 0) build_tc2_tables(s, tc2_nch, out);
  return out;
}

}  // namespace pgw
