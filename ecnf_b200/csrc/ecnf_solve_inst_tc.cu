// Tensor-core (tcgen05 / TMEM) instantiations of engine A + their weight-image / tile-table preparation.
#include <algorithm>
#include <vector>

#include "ecnf_solve_tc.cuh"

namespace ecnf_solve_detail {

namespace {

// the compiled (U, H) pairs of the tensor-core engine
bool tc_shape(const ecnf_config& c, int& U, int& H) {
  U = c.mlp_units; H = c.n_hidden;
  return (U == 128 && H == 64) || (U == 64 && H == 32);
}
int sub_of(const ecnf_config& c) { return 128 / c.mlp_units; }

int pick_mrows(const ecnf_config& c, bool div) {
  return c.mlp_units == 128 ? tc_pick_mrows<128, 64>(c.n_frames, c.dim, div) : tc_pick_mrows<64, 32>(c.n_frames, c.dim, div);
}
TcSmemLayout layout_of(const ecnf_config& c, int MR) {
  return c.mlp_units == 128 ? make_tc_layout<128, 64>(c.n_frames, c.dim, MR) : make_tc_layout<64, 32>(c.n_frames, c.dim, MR);
}

// walks the images (3 L + 3 per block) in a fixed order; fills the offsets and (optionally) the prep items
int64_t walk_images(const ecnf_model* mdl, TcImages* img, std::vector<TcPrepItem>* items) {
  const ecnf_config& c = mdl->cfg;
  const int H = c.n_hidden, U = c.mlp_units, L = c.n_layers, SUB = sub_of(c);
  int64_t off = 0;
  auto add = [&](int64_t src_off, int ksub, int N) {
    const int64_t o = off;
    if (items) items->push_back(TcPrepItem{(int)src_off, (int)o, ksub, N, SUB, U});
    off += (int64_t)(SUB * ksub) * 512;   // hi | lo, 128 lanes x K/2 words each
    return (int)o;
  };
  for (int b = 0; b < c.n_blocks; ++b) {
    const EcnfBlockOffsets& po = mdl->off[b];
    TcImgBlock ib{};
    ib.Wd = add(po.Wd, H, H);
    ib.We0 = add(po.We[0], 2 * H, U);                 // rows [h_send | h_recv]; the |v|^2 row is applied by the epilogue
    for (int l = 1; l < L; ++l) ib.We[l] = add(po.We[l], U, U);
    for (int l = 0; l < L; ++l) ib.Wx[l] = add(po.Wx[l], U, U);
    ib.Wh0m = add(po.Wh[0], U, U);
    ib.Wh0h = add(po.Wh[0] + (int64_t)U * U, H, U);
    for (int l = 1; l < L; ++l) ib.Wh[l] = add(po.Wh[l], U, U);
    ib.WhL = add(po.Wh[L], U, H);
    if (img) img->blk[b] = ib;
  }
  return off;
}

// tile counts / offsets of the table kinds
TcTabs make_tabs(const ecnf_model* mdl, int MR, int ntan = 0) {   // ntan: 0 = n * dim (exact trace), 1 = Hutchinson
  if (ntan <= 0) ntan = mdl->cfg.n_frames * mdl->cfg.dim;
  TcTabs t{};
  int off = 0;
  for (int k = 0; k < TT_COUNT; ++k) {
    t.off[k] = off;
    t.cnt[k] = tc_pack(k, mdl->cfg.n_frames, mdl->cfg.dim, sub_of(mdl->cfg), MR, nullptr, ntan);
    off += t.cnt[k];
  }
  return t;
}
int64_t tables_bytes(const TcTabs& t) { return (int64_t)(t.off[TT_COUNT - 1] + t.cnt[TT_COUNT - 1]) * TC_TILE_WORDS * 4; }
int64_t images_bytes(const ecnf_model* mdl) { return (walk_images(mdl, nullptr, nullptr) + 255) & ~255LL; }

template <int U, int H, bool DIV, bool SAVE>
int launch_one(const KernelArgs& a, int grid, size_t smem, cudaStream_t st) {
  auto kern = ecnf_solve_tc_kernel<U, H, DIV, SAVE>;
  ECNF_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, TC_NT, smem, st>>>(a);
  ECNF_CHECK_CUDA(cudaGetLastError());
  return ECNF_OK;
}

}  // namespace

bool tc_eligible(const ecnf_model* mdl, bool div) {
  const ecnf_config& c = mdl->cfg;
  int U, H;
  if (!tc_shape(c, U, H) || c.n_layers < 1 || c.n_frames < 2) return false;
  const int D = c.n_frames * c.dim;
  if (div && 1 + D > 256) return false;                 // slot numbers are 8-bit in the chunk words
  if (c.n_frames * (c.n_frames - 1) > 1023) return false;
  const int MR = pick_mrows(c, div);
  if (MR < 8 && div) return false;
  if (!div && MR < c.n_frames) return false;            // primal-only edge tiles aggregate over all receivers at once
  return layout_of(c, MR).total_bytes + 1024 <= 227 * 1024;
}

int64_t tc_image_bytes(const ecnf_model* mdl) {
  // tables of both variants (with / without the divergence) have different window sizes: reserve for the larger
  const int64_t t1 = tables_bytes(make_tabs(mdl, pick_mrows(mdl->cfg, true)));
  const int64_t t0 = tables_bytes(make_tabs(mdl, pick_mrows(mdl->cfg, false)));
  return images_bytes(mdl) + (((t1 > t0 ? t1 : t0) + 255) & ~255LL);
}

int64_t tc_flops_per_eval(const ecnf_model* mdl) {
  const ecnf_config& c = mdl->cfg;
  const int MR = pick_mrows(c, true), SUB = sub_of(c);
  int64_t sumN[TT_COUNT];
  for (int k = 0; k < TT_COUNT; ++k) {
    const int cnt = tc_pack(k, c.n_frames, c.dim, SUB, MR, nullptr, c.n_frames * c.dim);
    std::vector<uint32_t> buf((size_t)cnt * TC_TILE_WORDS);
    tc_pack(k, c.n_frames, c.dim, SUB, MR, buf.data(), c.n_frames * c.dim);
    sumN[k] = 0;
    for (int t = 0; t < cnt; ++t) sumN[k] += buf[(size_t)t * TC_TILE_WORDS + 32 + TH_N];
  }
  auto layer = [](int64_t n_cols, int K) { return 3 * 2 * (int64_t)128 * n_cols * K; };   // hi*hi + lo*hi + hi*lo
  int64_t fl = 0;
  for (int b = 0; b < c.n_blocks; ++b) {
    const bool last = b == c.n_blocks - 1;
    fl += (last ? 1 : 2) * layer(sumN[b > 0 ? TT_NODE : TT_NODE1], SUB * c.n_hidden);
    fl += (2 * c.n_layers) * layer(sumN[last ? TT_LAST : (b == 0 ? TT_FIRST : TT_MID)], 128);
    if (!last) fl += (c.n_layers + 1) * layer(sumN[TT_NODE], 128);
  }
  return fl;
}

int tc_tile_table(const ecnf_model* mdl, int kind, uint32_t* out, int64_t cap_words) {
  const bool hutch = kind >= 8;      // kind + 8: the one-tangent (Hutchinson) variant of the table
  if (hutch) kind -= 8;
  if (kind < 0 || kind >= TT_COUNT) return 0;
  const ecnf_config& c = mdl->cfg;
  const int MR = pick_mrows(c, kind != TT_NODE1 && kind != TT_EDGE1);
  const int ntan = hutch ? 1 : c.n_frames * c.dim;
  const int cnt = tc_pack(kind, c.n_frames, c.dim, sub_of(c), MR, nullptr, ntan);
  if (out && (int64_t)cnt * TC_TILE_WORDS <= cap_words) tc_pack(kind, c.n_frames, c.dim, sub_of(c), MR, out, ntan);
  return cnt;
}

int launch_tc(const ecnf_model* mdl, KernelArgs& a, int grid, void* image_ws, bool div, bool save, cudaStream_t st) {
  const ecnf_config& c = mdl->cfg;
  std::vector<TcPrepItem> items;
  a.img.base = reinterpret_cast<const unsigned char*>(image_ws);
  walk_images(mdl, &a.img, &items);
  // up to 8 blocks x (3 L + 3) = 168 images: one prep launch per slice of at most TC_PREP_MAX of them
  for (size_t i0 = 0; i0 < items.size(); i0 += TC_PREP_MAX) {
    TcPrepList list{};
    list.count = (int)std::min(items.size() - i0, (size_t)TC_PREP_MAX);
    std::copy(items.begin() + i0, items.begin() + i0 + list.count, list.item);
    dim3 pgrid(16, list.count);
    tc_prep_kernel<<<pgrid, 256, 0, st>>>(mdl->d_params, reinterpret_cast<unsigned char*>(image_ws), list);
    ECNF_CHECK_CUDA(cudaGetLastError());
  }
  const int MR = pick_mrows(c, div);
  // Hutchinson (a.eps given): one tangent direction -- the tables of kinds TT_NODE / TT_MID with two rows per group
  const int ntan = (div && a.eps) ? 1 : c.n_frames * c.dim;
  a.tabs = make_tabs(mdl, MR, ntan);
  uint32_t* tab_ws = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(image_ws) + images_bytes(mdl));
  a.tabs.base = tab_ws;
  tc_tables_kernel<<<TT_COUNT, 32, 0, st>>>(tab_ws, c.n_frames, c.dim, sub_of(c), MR, ntan, a.tabs);
  ECNF_CHECK_CUDA(cudaGetLastError());
  a.lay = layout_of(c, MR);
  const size_t smem = (size_t)a.lay.total_bytes;
  if (save) {
    if (c.mlp_units == 128)
      return div ? launch_one<128, 64, true, true>(a, grid, smem, st) : launch_one<128, 64, false, true>(a, grid, smem, st);
    return div ? launch_one<64, 32, true, true>(a, grid, smem, st) : launch_one<64, 32, false, true>(a, grid, smem, st);
  }
  if (c.mlp_units == 128)
    return div ? launch_one<128, 64, true, false>(a, grid, smem, st) : launch_one<128, 64, false, false>(a, grid, smem, st);
  return div ? launch_one<64, 32, true, false>(a, grid, smem, st) : launch_one<64, 32, false, false>(a, grid, smem, st);
}

}  // namespace ecnf_solve_detail
