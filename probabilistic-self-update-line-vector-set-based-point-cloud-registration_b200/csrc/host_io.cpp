// host_io.cpp -- host-side helpers of the callers around the hot path (include/psulvsb_io.h):
// PLY vertex reader (positions, and colours on request), correspondence files.  (The pre-filter and reduced-set builder are device code: k7_prefilter.cu.)
// Plain C++17, no CUDA, no third-party dependency (the reference uses PCL/Eigen/tinyply here).
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <numeric>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/psulvsb_io.h"

namespace psulvsb {
int fail(int code, const std::string& msg);
}
using psulvsb::fail;

// ---------------------------------------------------------------------------------------------
// PLY
// ---------------------------------------------------------------------------------------------
namespace {

struct PlyProp {
  std::string name;
  int size = 0;        // bytes of a scalar property (0 for lists)
  char kind = 'f';     // 'f' float, 'i' signed int, 'u' unsigned int
  bool is_list = false;
  int list_count_size = 0, list_item_size = 0;
};
struct PlyElement {
  std::string name;
  long long count = 0;
  std::vector<PlyProp> props;
};
struct PlyHeader {
  int format = 0;  // 0 ascii, 1 binary LE, 2 binary BE
  std::vector<PlyElement> elements;
  std::streampos data_begin;
};

bool type_info(const std::string& t, int& size, char& kind) {
  if (t == "char" || t == "int8") { size = 1; kind = 'i'; return true; }
  if (t == "uchar" || t == "uint8") { size = 1; kind = 'u'; return true; }
  if (t == "short" || t == "int16") { size = 2; kind = 'i'; return true; }
  if (t == "ushort" || t == "uint16") { size = 2; kind = 'u'; return true; }
  if (t == "int" || t == "int32") { size = 4; kind = 'i'; return true; }
  if (t == "uint" || t == "uint32") { size = 4; kind = 'u'; return true; }
  if (t == "float" || t == "float32") { size = 4; kind = 'f'; return true; }
  if (t == "double" || t == "float64") { size = 8; kind = 'f'; return true; }
  return false;
}

int parse_header(std::ifstream& f, PlyHeader& h, std::string& err) {
  std::string line;
  if (!std::getline(f, line) || line.substr(0, 3) != "ply") {
    err = "not a PLY file";
    return 1;
  }
  while (std::getline(f, line)) {
    if (!line.empty() && line.back() == '\r') line.pop_back();
    std::istringstream iss(line);
    std::string tok;
    iss >> tok;
    if (tok == "format") {
      std::string fmt;
      iss >> fmt;
      if (fmt == "ascii") h.format = 0;
      else if (fmt == "binary_little_endian") h.format = 1;
      else if (fmt == "binary_big_endian") h.format = 2;
      else { err = "unknown PLY format " + fmt; return 1; }
    } else if (tok == "element") {
      PlyElement e;
      iss >> e.name >> e.count;
      h.elements.push_back(e);
    } else if (tok == "property") {
      if (h.elements.empty()) { err = "property before element"; return 1; }
      PlyProp p;
      std::string t;
      iss >> t;
      if (t == "list") {
        std::string ct, it;
        iss >> ct >> it >> p.name;
        p.is_list = true;
        char kc, ki;
        if (!type_info(ct, p.list_count_size, kc) || !type_info(it, p.list_item_size, ki)) { err = "bad list type"; return 1; }
        if (kc == 'f') { err = "list count type must be an integer type, got " + ct; return 1; }
      } else {
        iss >> p.name;
        if (!type_info(t, p.size, p.kind)) { err = "unknown property type " + t; return 1; }
      }
      h.elements.back().props.push_back(p);
    } else if (tok == "end_header") {
      h.data_begin = f.tellg();
      return 0;
    }
  }
  err = "no end_header";
  return 1;
}

template <typename T>
T load_scalar(const unsigned char* p, bool swap) {
  unsigned char b[sizeof(T)];
  for (size_t i = 0; i < sizeof(T); ++i) b[i] = swap ? p[sizeof(T) - 1 - i] : p[i];
  T v;
  std::memcpy(&v, b, sizeof(T));
  return v;
}

double scalar_as_double(const unsigned char* p, const PlyProp& pr, bool swap) {
  if (pr.kind == 'f') return pr.size == 4 ? (double)load_scalar<float>(p, swap) : load_scalar<double>(p, swap);
  if (pr.kind == 'i') {
    if (pr.size == 1) return (double)load_scalar<int8_t>(p, swap);
    if (pr.size == 2) return (double)load_scalar<int16_t>(p, swap);
    return (double)load_scalar<int32_t>(p, swap);
  }
  if (pr.size == 1) return (double)load_scalar<uint8_t>(p, swap);
  if (pr.size == 2) return (double)load_scalar<uint16_t>(p, swap);
  return (double)load_scalar<uint32_t>(p, swap);
}

unsigned long long list_count(const unsigned char* p, int size, bool swap) {
  if (size == 1) return load_scalar<uint8_t>(p, swap);
  if (size == 2) return load_scalar<uint16_t>(p, swap);
  return load_scalar<uint32_t>(p, swap);
}

// a colour channel's value: uchar / uint8 over 255, float / double as stored
double color_value(double v, const PlyProp& pr) { return pr.kind == 'u' ? v / 255.0 : v; }

// reads the vertex element; xyz == nullptr: only counts.  rgb != nullptr: the red, green and blue properties too
// (uchar / uint8, float or double; anything else, or a missing channel, is refused)
int ply_read(const char* path, float* xyz, double* rgb, long long capacity, long long* n_out) {
  if (!path || !n_out) return fail(PSULVSB_ERR_INVALID, "ply: NULL argument");
  std::ifstream f(path, std::ios::binary);
  if (!f.is_open()) return fail(PSULVSB_ERR_INVALID, std::string("ply: cannot open ") + path);
  PlyHeader h;
  std::string err;
  if (parse_header(f, h, err)) return fail(PSULVSB_ERR_INVALID, std::string("ply: ") + err + " in " + path);
  int vi = -1;
  for (size_t e = 0; e < h.elements.size(); ++e)
    if (h.elements[e].name == "vertex") vi = (int)e;
  if (vi < 0) return fail(PSULVSB_ERR_INVALID, std::string("ply: no vertex element in ") + path);
  const PlyElement& V = h.elements[(size_t)vi];
  *n_out = V.count;
  if (!xyz) return PSULVSB_OK;
  if (capacity < V.count) return fail(PSULVSB_ERR_CAPACITY, "ply: output buffer too small");
  int ix = -1, iy = -1, iz = -1;
  for (size_t p = 0; p < V.props.size(); ++p) {
    if (V.props[p].name == "x") ix = (int)p;
    if (V.props[p].name == "y") iy = (int)p;
    if (V.props[p].name == "z") iz = (int)p;
  }
  if (ix < 0 || iy < 0 || iz < 0) return fail(PSULVSB_ERR_INVALID, "ply: vertex element lacks x / y / z");
  int ic[3] = {-1, -1, -1};
  if (rgb) {
    static const char* const kChannel[3] = {"red", "green", "blue"};
    for (int k = 0; k < 3; ++k) {
      for (size_t p = 0; p < V.props.size(); ++p)
        if (V.props[p].name == kChannel[k]) ic[k] = (int)p;
      if (ic[k] < 0)
        return fail(PSULVSB_ERR_INVALID, std::string("ply: vertex element lacks ") + kChannel[k] + " in " + path);
      const PlyProp& pr = V.props[(size_t)ic[k]];
      if (pr.is_list || !((pr.kind == 'u' && pr.size == 1) || pr.kind == 'f'))
        return fail(PSULVSB_ERR_INVALID, std::string("ply: unsupported type of vertex property ") + kChannel[k] +
                                             " (uchar / uint8, float or double) in " + path);
    }
  }
  f.clear();
  f.seekg(h.data_begin);
  const bool host_le = [] { const uint16_t one = 1; return *reinterpret_cast<const unsigned char*>(&one) == 1; }();
  const bool swap = (h.format == 1 && !host_le) || (h.format == 2 && host_le);
  for (int e = 0; e <= vi; ++e) {
    const PlyElement& E = h.elements[(size_t)e];
    const bool is_vertex = e == vi;
    for (long long r = 0; r < E.count; ++r) {
      if (h.format == 0) {
        std::string line;
        do {
          if (!std::getline(f, line)) return fail(PSULVSB_ERR_INVALID, "ply: truncated ascii data");
        } while (line.find_first_not_of(" \t\r") == std::string::npos);
        if (!is_vertex) continue;
        std::istringstream iss(line);
        for (size_t p = 0; p < E.props.size(); ++p) {
          double v;
          if (!(iss >> v)) return fail(PSULVSB_ERR_INVALID, "ply: malformed ascii vertex line");
          if ((int)p == ix) xyz[3 * r + 0] = (float)v;
          if ((int)p == iy) xyz[3 * r + 1] = (float)v;
          if ((int)p == iz) xyz[3 * r + 2] = (float)v;
          if (rgb)
            for (int k = 0; k < 3; ++k)
              if ((int)p == ic[k]) rgb[3 * r + k] = color_value(v, E.props[p]);
        }
      } else {
        for (size_t p = 0; p < E.props.size(); ++p) {
          const PlyProp& pr = E.props[p];
          unsigned char buf[8];
          if (pr.is_list) {
            if (!f.read((char*)buf, pr.list_count_size)) return fail(PSULVSB_ERR_INVALID, "ply: truncated data");
            const unsigned long long c = list_count(buf, pr.list_count_size, swap);
            if (!f.seekg((std::streamoff)(c * (unsigned long long)pr.list_item_size), std::ios::cur))
              return fail(PSULVSB_ERR_INVALID, "ply: cannot skip a list property (truncated data)");
          } else {
            if (!f.read((char*)buf, pr.size)) return fail(PSULVSB_ERR_INVALID, "ply: truncated data");
            if (is_vertex) {
              if ((int)p == ix) xyz[3 * r + 0] = (float)scalar_as_double(buf, pr, swap);
              if ((int)p == iy) xyz[3 * r + 1] = (float)scalar_as_double(buf, pr, swap);
              if ((int)p == iz) xyz[3 * r + 2] = (float)scalar_as_double(buf, pr, swap);
              if (rgb)
                for (int k = 0; k < 3; ++k)
                  if ((int)p == ic[k]) rgb[3 * r + k] = color_value(scalar_as_double(buf, pr, swap), pr);
            }
          }
        }
      }
    }
  }
  return PSULVSB_OK;
}

bool is_single_integer(const std::string& line) {
  std::istringstream iss(line);
  long long v;
  std::string rest;
  if (!(iss >> v)) return false;
  return !(iss >> rest);
}

// src/dst == nullptr: only counts
int corr_read(const char* path, double* src, double* dst, long long capacity, long long* n_out) {
  if (!path || !n_out) return fail(PSULVSB_ERR_INVALID, "corr: NULL argument");
  std::ifstream f(path);
  if (!f.is_open()) return fail(PSULVSB_ERR_INVALID, std::string("corr: cannot open ") + path);
  std::string line;
  long long n = 0;
  bool first = true;
  while (std::getline(f, line)) {
    if (first) {
      first = false;
      if (is_single_integer(line)) continue;  // count header (teaser_cpp_ply.cc:236)
    }
    std::istringstream iss(line);
    double s1, s2, s3, t1, t2, t3;
    if (iss >> s1 >> s2 >> s3 >> t1 >> t2 >> t3) {
      if (src && dst) {
        if (n >= capacity) return fail(PSULVSB_ERR_CAPACITY, "corr: output buffer too small");
        src[3 * n + 0] = s1;
        src[3 * n + 1] = s2;
        src[3 * n + 2] = s3;
        dst[3 * n + 0] = t1;
        dst[3 * n + 1] = t2;
        dst[3 * n + 2] = t3;
      }
      ++n;
    }
  }
  *n_out = n;
  return PSULVSB_OK;
}

}  // namespace

extern "C" {

int psulvsb_ply_vertex_count(const char* path, long long* n) { return ply_read(path, nullptr, nullptr, 0, n); }
int psulvsb_ply_read_xyz(const char* path, float* xyz, long long capacity, long long* n) {
  if (!xyz) return fail(PSULVSB_ERR_INVALID, "psulvsb_ply_read_xyz: NULL output");
  return ply_read(path, xyz, nullptr, capacity, n);
}
int psulvsb_ply_read_xyz_rgb(const char* path, float* xyz, double* rgb, long long capacity, long long* n) {
  if (!xyz || !rgb) return fail(PSULVSB_ERR_INVALID, "psulvsb_ply_read_xyz_rgb: NULL output");
  return ply_read(path, xyz, rgb, capacity, n);
}
int psulvsb_corr_count(const char* path, long long* n) { return corr_read(path, nullptr, nullptr, 0, n); }
int psulvsb_corr_read(const char* path, double* src, double* dst, long long capacity, long long* n) {
  if (!src || !dst) return fail(PSULVSB_ERR_INVALID, "psulvsb_corr_read: NULL output");
  return corr_read(path, src, dst, capacity, n);
}
int psulvsb_gtmat_read(const char* path, double* T) {
  if (!path || !T) return fail(PSULVSB_ERR_INVALID, "psulvsb_gtmat_read: NULL argument");
  std::ifstream f(path);
  if (!f.is_open()) return fail(PSULVSB_ERR_INVALID, std::string("gtmat: cannot open ") + path);
  for (int r = 0; r < 4; ++r) {
    double a, b, c, d;
    if (!(f >> a >> b >> c >> d)) return fail(PSULVSB_ERR_INVALID, std::string("gtmat: fewer than 16 numbers in ") + path);
    T[0 * 4 + r] = a;
    T[1 * 4 + r] = b;
    T[2 * 4 + r] = c;
    T[3 * 4 + r] = d;
  }
  return PSULVSB_OK;
}
int psulvsb_gtlog_read(const char* path, int* pairs, long long capacity, long long* n) {
  if (!path || !n) return fail(PSULVSB_ERR_INVALID, "psulvsb_gtlog_read: NULL argument");
  std::ifstream f(path);
  if (!f.is_open()) return fail(PSULVSB_ERR_INVALID, std::string("gtlog: cannot open ") + path);
  std::string line;
  long long k = 0;
  while (std::getline(f, line)) {
    std::istringstream iss(line);
    int a, b, v;
    if (iss >> a >> b >> v) {
      if (pairs) {
        if (k >= capacity) return fail(PSULVSB_ERR_CAPACITY, "gtlog: output buffer too small");
        pairs[2 * k] = a;
        pairs[2 * k + 1] = b;
      }
      ++k;
    }
  }
  *n = k;
  return PSULVSB_OK;
}

}  // extern "C"
