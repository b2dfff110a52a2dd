// tests/host_cpp/roadmap_check.cpp -- drives the C++ host mirror (include/artp_host.hpp) the way Planner's old-map chain
// and LazyPRMStarMinUpdate::clear() drive the reference: processors::computeChange on the new / old map, then
// LazyPRMStarMinUpdateMaintainer::update on the roadmap's validity flags.
//   roadmap_check --expect-no-gpu       : construction must fail loudly (no CPU fallback)
//   roadmap_check <in.bin> <out.bin>    : run the case in in.bin, write the results (see tests/test_roadmap_update_gpu.py)
#include <cstring>
#include <fstream>
#include <iostream>

#include "artp_host.hpp"

using namespace artp_host;

template <class T> static void rd(std::ifstream& f, T* p, size_t n) { f.read(reinterpret_cast<char*>(p), sizeof(T) * n); }
template <class T> static void wr(std::ofstream& f, const T* p, size_t n) { f.write(reinterpret_cast<const char*>(p), sizeof(T) * n); }

int main(int argc, char** argv) {
  auto params = std::make_shared<Params>();
  if (argc == 2 && !std::strcmp(argv[1], "--expect-no-gpu")) {
    try {
      auto h = std::make_shared<Handle>(params);
    } catch (const std::runtime_error& e) {
      std::cout << "failed loudly: " << e.what() << "\n";
      return 0;
    }
    std::cout << "a handle was created: a CUDA device is present\n";
    return 3;
  }
  if (argc != 3) { std::cerr << "usage\n"; return 2; }
  std::ifstream in(argv[1], std::ios::binary);
  int32_t hdr[6];   // rows_new, cols_new, rows_old, cols_old, n_vertices, n_edges
  double geo[6];    // res, new cx, cy, old cx, cy, height_change_for_update
  rd(in, hdr, 6);
  rd(in, geo, 6);
  auto map_new = std::make_shared<Map>(), map_old = std::make_shared<Map>();
  map_new->rows = hdr[0]; map_new->cols = hdr[1]; map_old->rows = hdr[2]; map_old->cols = hdr[3];
  map_new->resolution = map_old->resolution = geo[0];
  map_new->position_x = geo[1]; map_new->position_y = geo[2]; map_old->position_x = geo[3]; map_old->position_y = geo[4];
  for (Map* m : {map_new.get(), map_old.get()}) {
    const size_t ncell = static_cast<size_t>(m->rows) * m->cols;
    m->elevation.resize(ncell); m->traversability_thresholded.resize(ncell);
    rd(in, m->elevation.data(), ncell);
    rd(in, m->traversability_thresholded.data(), ncell);
  }
  const size_t nv = hdr[4], ne = hdr[5];
  std::vector<State> vertices(nv);
  std::vector<uint32_t> edges(2 * ne);
  std::vector<unsigned int> vvalid(nv), evalid(ne);
  rd(in, &vertices[0].x, 7 * nv);
  rd(in, edges.data(), 2 * ne);
  rd(in, vvalid.data(), nv);
  rd(in, evalid.data(), ne);

  auto handle = std::make_shared<Handle>(params);
  processors::computeChange(handle, map_new, map_old, static_cast<float>(geo[5]));   // planner.cpp:60-69 old-map chain
  LazyPRMStarMinUpdateMaintainer maintainer(handle);
  const std::vector<size_t> removed = maintainer.update(vertices, &vvalid, edges, &evalid);   // :123-135
  std::vector<uint8_t> at(nv);   // Map::getUpdatedAtPosition per vertex: 0 / 1, 2 = threw std::out_of_range
  for (size_t v = 0; v < nv; ++v) {
    try {
      at[v] = map_new->getUpdatedAtPosition(vertices[v].x, vertices[v].y) ? 1 : 0;
    } catch (const std::out_of_range&) {
      at[v] = 2;
    }
  }
  std::ofstream out(argv[2], std::ios::binary);
  wr(out, map_new->updated.data(), map_new->updated.size());
  wr(out, vvalid.data(), nv);
  wr(out, evalid.data(), ne);
  const uint64_t nr = removed.size();
  wr(out, &nr, 1);
  for (size_t v : removed) { const uint64_t x = v; wr(out, &x, 1); }
  wr(out, at.data(), nv);
  return 0;
}
