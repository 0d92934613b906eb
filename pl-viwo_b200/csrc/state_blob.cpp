// Encoder and checked decoder of the tracker state blob (state_blob.h).
#include "state_blob.h"

#include <cstring>

namespace plviwo {

static constexpr uint32_t kStateMagic = 0x504c5657u;
static constexpr uint32_t kStateVersion = 1;

StateHeader state_header(int w, int h, uint64_t currid, uint64_t line_currid, int n_pts, int n_lines, const PointsOnLines &pol,
                         bool has_image, bool has_mask) {
  StateHeader hd;
  std::memset(&hd, 0, sizeof(hd));
  hd.magic = kStateMagic;
  hd.version = kStateVersion;
  hd.w = w;
  hd.h = h;
  hd.currid = currid;
  hd.line_currid = line_currid;
  hd.n_pts = n_pts;
  hd.n_lines = n_lines;
  hd.has_image = has_image ? 1 : 0;
  hd.has_mask = has_image && has_mask ? 1 : 0;
  for (const auto &m : pol) hd.n_pol_entries += (int32_t)m.size();
  return hd;
}

StateLayout state_layout(const StateHeader &hd) {
  StateLayout at;
  const size_t img = (size_t)hd.w * hd.h;
  at.pts = sizeof(StateHeader);
  at.ids = at.pts + (size_t)hd.n_pts * 2 * sizeof(float);
  at.lines = at.ids + (size_t)hd.n_pts * sizeof(uint64_t);
  at.line_ids = at.lines + (size_t)hd.n_lines * 4 * sizeof(float);
  at.pol_sizes = at.line_ids + (size_t)hd.n_lines * sizeof(uint64_t);
  at.pol = at.pol_sizes + (size_t)hd.n_lines * sizeof(int32_t);
  at.image = at.pol + (size_t)hd.n_pol_entries * (sizeof(int32_t) + sizeof(double));
  at.mask = at.image + (hd.has_image ? img : 0);
  at.size = at.mask + (hd.has_image && hd.has_mask ? img : 0);
  return at;
}

void state_write(void *buf, const StateHeader &hd, const void *pts, const void *ids, const void *lines, const void *line_ids,
                 const PointsOnLines &pol) {
  uint8_t *p = static_cast<uint8_t *>(buf);
  auto put = [&](const void *src, size_t n) {
    if (n) std::memcpy(p, src, n);
    p += n;
  };
  put(&hd, sizeof(hd));
  put(pts, (size_t)hd.n_pts * 2 * sizeof(float));
  put(ids, (size_t)hd.n_pts * sizeof(uint64_t));
  put(lines, (size_t)hd.n_lines * 4 * sizeof(float));
  put(line_ids, (size_t)hd.n_lines * sizeof(uint64_t));
  for (const auto &m : pol) {
    const int32_t k = (int32_t)m.size();
    put(&k, sizeof(k));
  }
  for (const auto &m : pol)
    for (const auto &kv : m) {
      const int32_t k = kv.first;
      put(&k, sizeof(k));
      put(&kv.second, sizeof(double));
    }
}

const char *state_read(const void *buf, size_t n_bytes, int w, int h, StateView &v) {
  if (!buf || n_bytes < sizeof(StateHeader)) return "set_state: blob shorter than a state header";
  v.base = static_cast<const uint8_t *>(buf);
  std::memcpy(&v.hd, v.base, sizeof(v.hd));
  const StateHeader &hd = v.hd;
  if (hd.magic != kStateMagic || hd.version != kStateVersion || hd.w != w || hd.h != h) return "set_state: foreign blob";
  if (hd.n_pts < 0 || hd.n_lines < 0 || hd.n_pol_entries < 0) return "set_state: negative counts";
  v.at = state_layout(hd);
  // a truncated or foreign buffer is rejected, not read past
  if (n_bytes < v.at.size) return "set_state: blob shorter than its header announces";
  std::vector<int32_t> sizes(hd.n_lines);
  if (hd.n_lines) std::memcpy(sizes.data(), v.base + v.at.pol_sizes, (size_t)hd.n_lines * sizeof(int32_t));
  long long tot = 0;
  for (int32_t k : sizes) {
    if (k < 0) return "set_state: negative line size";
    tot += k;
  }
  if (tot != hd.n_pol_entries) return "set_state: line sizes do not add up to the header's entry count";
  v.pol.assign(hd.n_lines, {});
  const uint8_t *p = v.base + v.at.pol;
  for (int i = 0; i < hd.n_lines; i++)
    for (int k = 0; k < sizes[i]; k++) {
      int32_t key;
      double val;
      std::memcpy(&key, p, sizeof(key));
      std::memcpy(&val, p + sizeof(key), sizeof(val));
      p += sizeof(key) + sizeof(val);
      v.pol[i][key] = val;
    }
  return nullptr;
}

}  // namespace plviwo
