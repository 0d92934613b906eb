// The tracker state blob of plviwo_fe_get_state / _set_state, also one stream's blob of plviwo_fe_group_get_state /
// _set_state.  After the header, in this order:
//   pts        n_pts x 2 float        pts_last
//   ids        n_pts x uint64         ids_last
//   lines      n_lines x 4 float      lines_last of the line tracker
//   line_ids   n_lines x uint64
//   pol_sizes  n_lines x int32        entries of each line's point map
//   pol        n_pol_entries x (int32 point id, double distance), line after line
//   image      w x h bytes            the last equalised level-0 image, if has_image
//   mask       w x h bytes            its mask, if has_image and has_mask
#pragma once
#include <cstddef>
#include <cstdint>
#include <map>
#include <vector>

namespace plviwo {

struct StateHeader {
  uint32_t magic, version;
  int32_t w, h;
  uint64_t currid, line_currid;
  int32_t n_pts, n_lines, has_image, has_mask;
  int32_t n_pol_entries, reserved;
};

// A line tracker's point map per line: point id -> distance, ascending ids (TrackLSD's std::map<int, double>).
using PointsOnLines = std::vector<std::map<int, double>>;

// Byte offsets of the sections of a blob and its total size.
struct StateLayout {
  size_t pts, ids, lines, line_ids, pol_sizes, pol, image, mask, size;
};

StateHeader state_header(int w, int h, uint64_t currid, uint64_t line_currid, int n_pts, int n_lines, const PointsOnLines &pol,
                         bool has_image, bool has_mask);
StateLayout state_layout(const StateHeader &hd);

// Writes the header and every section before the image into buf (state_layout(hd).size bytes); the caller copies the image
// and the mask to their offsets.  pts / ids hold hd.n_pts entries, lines / line_ids and pol hd.n_lines.
void state_write(void *buf, const StateHeader &hd, const void *pts, const void *ids, const void *lines, const void *line_ids,
                 const PointsOnLines &pol);

// A blob that passed state_read: sections are read at base + at.*, the point maps are decoded (of two entries of one line
// with the same point id the later wins).
struct StateView {
  StateHeader hd;
  StateLayout at;
  const uint8_t *base;
  PointsOnLines pol;
};
// Accepts a blob of this format for a w x h tracker that holds everything its header announces; otherwise returns the
// reason and leaves v unspecified.
const char *state_read(const void *buf, size_t n_bytes, int w, int h, StateView &v);

// A stereo rig's blob (plviwo_fe_stereo_get_state, plviwo_fe_stereo_group_get_state): this header, then the left and the right
// camera's blob of the format above (size[0] and size[1] bytes).  currid is the rig's id counter, shared by both cameras.
struct StereoStateHeader {
  uint32_t magic, version;
  uint64_t currid;
  uint64_t size[2];
};
constexpr uint32_t kStereoStateMagic = 0x504c5653u;   // 'PLVS'
constexpr uint32_t kStereoStateVersion = 1;

}  // namespace plviwo
