// vlp16_synth.cpp — seeded synthetic Velodyne VLP-16 scans (SURVEY.md §8d sensor model).
//
// Test / bench input generator, host only.  16 lasers at -15..+15 deg (step 2), A azimuth
// columns over 360 deg, sensor at the origin, level ground plane at z = -1.8 m in the levelled
// frame, max range 100 m, no-return rays dropped, range noise N(0, 0.02 m), 1 % dropout.
// The sensor frame is tilted by (roll, pitch) w.r.t. the levelled frame, so that the pipeline's
// rotateCloud (reference src:159-167) levels the ground again.  Points come out in firing order
// (column-major, lasers interleaved as on the real device), as float4 {x,y,z,intensity=0}.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#include "../../include/fe_b200.h"

namespace {

struct Rng {  // splitmix64-seeded xoshiro256**
  uint64_t s[4];
  static uint64_t splitmix(uint64_t& x) {
    uint64_t z = (x += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  }
  explicit Rng(uint64_t seed) { for (int i = 0; i < 4; i++) s[i] = splitmix(seed); }
  static uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
  uint64_t next() {
    uint64_t r = rotl(s[1] * 5, 7) * 9, t = s[1] << 17;
    s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t; s[3] = rotl(s[3], 45);
    return r;
  }
  double uni() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
  double uni(double a, double b) { return a + (b - a) * uni(); }
  int randint(int a, int b) { return a + (int)(uni() * (double)(b - a + 1)); }  // inclusive
  double normal() {
    double u1 = uni(), u2 = uni();
    if (u1 < 1e-300) u1 = 1e-300;
    return sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
  }
};

const double kGroundZ = -1.8;
const double kMaxRange = 100.0;

struct Cyl { double x, y, r, z0, z1; };
struct Box { double cx, cy, hx, hy, yaw_c, yaw_s, z0, z1; };
struct Sph { double x, y, z, r; };

struct Scene {
  std::vector<Cyl> cyl;
  std::vector<Box> box;
  std::vector<Sph> sph;
};

void add_pole(Scene& sc, Rng& g, double x, double y, bool trunk) {
  Cyl c;
  c.x = x; c.y = y;
  c.r = trunk ? g.uni(0.15, 0.25) : g.uni(0.06, 0.12);
  c.z0 = kGroundZ;
  c.z1 = kGroundZ + (trunk ? g.uni(3.0, 6.0) : 4.0);
  sc.cyl.push_back(c);
}

void random_xy(Rng& g, double rmin, double rmax, double& x, double& y) {
  // uniform in range/azimuth, restricted to the default crop's footprint (x>=2, |y|<=28)
  for (;;) {
    double r = g.uni(rmin, rmax), a = g.uni(-1.45, 1.45);
    x = r * cos(a); y = r * sin(a);
    if (x >= 2.0 && x <= 72.0 && fabs(y) <= 28.0) return;
  }
}

void add_wall(Scene& sc, Rng& g, double rmin, double rmax, bool car) {
  Box b;
  random_xy(g, rmin, rmax, b.cx, b.cy);
  double yaw = g.uni(0.0, 3.141592653589793);
  b.yaw_c = cos(yaw); b.yaw_s = sin(yaw);
  if (car) { b.hx = 2.0; b.hy = 0.9; b.z0 = kGroundZ; b.z1 = kGroundZ + 1.5; }
  else { b.hx = 0.5 * g.uni(4.0, 15.0); b.hy = 0.15; b.z0 = kGroundZ; b.z1 = kGroundZ + g.uni(2.0, 4.0); }
  // keep the sensor outside the box
  double dx = -b.cx, dy = -b.cy;
  double lx = b.yaw_c * dx + b.yaw_s * dy, ly = -b.yaw_s * dx + b.yaw_c * dy;
  if (fabs(lx) < b.hx + 1.0 && fabs(ly) < b.hy + 1.0) return;
  sc.box.push_back(b);
}

void build_scene(int config, Rng& g, Scene& sc) {
  double x, y;
  if (config == 1) {  // a few poles / trees
    for (int i = 0; i < 5; i++) { random_xy(g, 5.0, 40.0, x, y); add_pole(sc, g, x, y, false); }
    for (int i = 0; i < 3; i++) { random_xy(g, 5.0, 40.0, x, y); add_pole(sc, g, x, y, true); }
  } else if (config == 3) {  // dense urban
    int np = g.randint(30, 60);
    for (int i = 0; i < np; i++) { random_xy(g, 4.0, 60.0, x, y); add_pole(sc, g, x, y, g.uni() < 0.3); }
    int nb = g.randint(10, 20);
    for (int i = 0; i < nb; i++) add_wall(sc, g, 6.0, 60.0, g.uni() < 0.5);
    int ns = g.randint(20, 40);
    for (int i = 0; i < ns; i++) {
      Sph s; random_xy(g, 4.0, 50.0, s.x, s.y); s.r = g.uni(0.2, 0.5); s.z = kGroundZ + s.r * g.uni(0.5, 1.0);
      sc.sph.push_back(s);
    }
  } else if (config == 4) {  // descriptor-heavy: hundreds of poles on a jittered lattice
    int n = g.randint(200, 400);
    double x0 = 3.0, x1 = 72.0, y0 = -28.0, y1 = 28.0;
    double s = sqrt((x1 - x0) * (y1 - y0) / (double)n);
    int placed = 0;
    for (double yy = y0 + 0.5 * s; yy < y1 && placed < n; yy += s)
      for (double xx = x0 + 0.5 * s; xx < x1 && placed < n; xx += s) {
        add_pole(sc, g, xx + g.uni(-0.3, 0.3) * s, yy + g.uni(-0.3, 0.3) * s, false);
        placed++;
      }
  } else {  // config 2 / 5: 3-12 poles or trunks, 0-4 walls
    int np = g.randint(3, 12);
    for (int i = 0; i < np; i++) { random_xy(g, 4.0, 25.0, x, y); add_pole(sc, g, x, y, g.uni() < 0.3); }
    int nw = g.randint(0, 4);
    for (int i = 0; i < nw; i++) add_wall(sc, g, 10.0, 50.0, false);
  }
}

inline void add_cols(std::vector<std::vector<int> >& cols, int A, double az_c, double half, int id) {
  if (half >= 3.14159) { for (int a = 0; a < A; a++) cols[a].push_back(id); return; }
  const double step = 6.283185307179586 / (double)A;
  int a0 = (int)floor((az_c - half) / step), a1 = (int)ceil((az_c + half) / step);
  for (int a = a0; a <= a1; a++) cols[((a % A) + A) % A].push_back(id);
}

uint64_t scene_seed(int config, uint64_t scan_index) {
  return (uint64_t)config * 0x100000001B3ull + scan_index * 0x9E3779B97F4A7C15ull + 12345u;
}

// The scene `sc` as the sensor at pose = (x, y, yaw) of the scene frame sees it: every object moved by
// R(-yaw) * (world - (x, y)).  The ground plane does not move.  At the identity pose every coordinate comes out
// bit for bit as it went in (x*1 + y*0 == x).
Scene posed(const Scene& sc, const double* pose) {
  const double c = cos(pose[2]), s = sin(pose[2]);
  auto move = [&](double& x, double& y) {
    const double dx = x - pose[0], dy = y - pose[1];
    x = c * dx + s * dy;
    y = -s * dx + c * dy;
  };
  Scene o = sc;
  for (Cyl& k : o.cyl) move(k.x, k.y);
  for (Sph& k : o.sph) move(k.x, k.y);
  for (Box& k : o.box) {
    move(k.cx, k.cy);
    const double yc = k.yaw_c * c + k.yaw_s * s, ys = k.yaw_s * c - k.yaw_c * s;  // yaw - pose yaw
    k.yaw_c = yc;
    k.yaw_s = ys;
  }
  return o;
}

// Renders the scene `sc`, given in the sensor's levelled frame: roll, pitch, range noise and dropout are drawn from g.
int64_t render_scan(int config, const Scene& sc, Rng& g, int A, fe_point_t* out, double* roll_pitch) {
  double roll, pitch;
  if (config == 1) { roll = 0.02; pitch = -0.015; }
  else { roll = g.uni(-0.05, 0.05); pitch = g.uni(-0.05, 0.05); }
  roll_pitch[0] = roll; roll_pitch[1] = pitch;
  // levelled = Ry(pitch) * Rx(roll) * sensor
  const double cr = cos(roll), sr = sin(roll), cp = cos(pitch), sp = sin(pitch);
  const double M[3][3] = {{cp, sp * sr, sp * cr}, {0.0, cr, -sr}, {-sp, cp * sr, cp * cr}};

  // per-column candidate lists (azimuth culling in the sensor frame, padded for the tilt)
  const int nc = (int)sc.cyl.size(), nb = (int)sc.box.size(), ns = (int)sc.sph.size();
  std::vector<std::vector<int> > cols(A);
  const double pad = 0.12;
  for (int i = 0; i < nc; i++) {
    double d = hypot(sc.cyl[i].x, sc.cyl[i].y);
    double half = d > sc.cyl[i].r ? asin(std::min(1.0, sc.cyl[i].r / d)) + pad : 4.0;
    add_cols(cols, A, atan2(sc.cyl[i].y, sc.cyl[i].x), half, i);
  }
  for (int i = 0; i < nb; i++) {
    double rb = hypot(sc.box[i].hx, sc.box[i].hy), d = hypot(sc.box[i].cx, sc.box[i].cy);
    double half = d > rb ? asin(std::min(1.0, rb / d)) + pad : 4.0;
    add_cols(cols, A, atan2(sc.box[i].cy, sc.box[i].cx), half, nc + i);
  }
  for (int i = 0; i < ns; i++) {
    double d = hypot(sc.sph[i].x, sc.sph[i].y);
    double half = d > sc.sph[i].r ? asin(std::min(1.0, sc.sph[i].r / d)) + pad : 4.0;
    add_cols(cols, A, atan2(sc.sph[i].y, sc.sph[i].x), half, nc + nb + i);
  }

  static const int kLaserDeg[16] = {-15, 1, -13, 3, -11, 5, -9, 7, -7, 9, -5, 11, -3, 13, -1, 15};
  double cel[16], sel[16];
  for (int k = 0; k < 16; k++) {
    double e = (double)kLaserDeg[k] * 0.017453292519943295;
    cel[k] = cos(e); sel[k] = sin(e);
  }
  int64_t n = 0;
  for (int a = 0; a < A; a++) {
    const double az = 6.283185307179586 * (double)a / (double)A;
    const double ca = cos(az), sa = sin(az);
    const std::vector<int>& cand = cols[a];
    for (int k = 0; k < 16; k++) {
      const double ds[3] = {cel[k] * ca, cel[k] * sa, sel[k]};
      const double dx = M[0][0] * ds[0] + M[0][1] * ds[1] + M[0][2] * ds[2];
      const double dy = M[1][0] * ds[0] + M[1][1] * ds[1] + M[1][2] * ds[2];
      const double dz = M[2][0] * ds[0] + M[2][1] * ds[1] + M[2][2] * ds[2];
      double t = 1e30;
      if (dz < -1e-9) t = kGroundZ / dz;
      for (size_t ci = 0; ci < cand.size(); ci++) {
        int id = cand[ci];
        if (id < nc) {
          const Cyl& c = sc.cyl[id];
          double A2 = dx * dx + dy * dy;
          double B = -(dx * c.x + dy * c.y);
          double C = c.x * c.x + c.y * c.y - c.r * c.r;
          double disc = B * B - A2 * C;
          if (disc <= 0.0 || A2 < 1e-18) continue;
          double tt = (-B - sqrt(disc)) / A2;
          if (tt <= 0.0 || tt >= t) continue;
          double z = tt * dz;
          if (z < c.z0 || z > c.z1) continue;
          t = tt;
        } else if (id < nc + nb) {
          const Box& b = sc.box[id - nc];
          // ray in box frame
          double ox = -(b.yaw_c * b.cx + b.yaw_s * b.cy), oy = -(-b.yaw_s * b.cx + b.yaw_c * b.cy);
          double lx = b.yaw_c * dx + b.yaw_s * dy, ly = -b.yaw_s * dx + b.yaw_c * dy;
          double t0 = 0.0, t1 = t;
          const double o3[3] = {ox, oy, 0.0}, d3[3] = {lx, ly, dz};
          const double lo[3] = {-b.hx, -b.hy, b.z0}, hi[3] = {b.hx, b.hy, b.z1};
          bool miss = false;
          for (int ax = 0; ax < 3 && !miss; ax++) {
            if (fabs(d3[ax]) < 1e-12) { if (o3[ax] < lo[ax] || o3[ax] > hi[ax]) miss = true; continue; }
            double ta = (lo[ax] - o3[ax]) / d3[ax], tb = (hi[ax] - o3[ax]) / d3[ax];
            if (ta > tb) std::swap(ta, tb);
            t0 = std::max(t0, ta); t1 = std::min(t1, tb);
            if (t0 > t1) miss = true;
          }
          if (miss || t0 <= 0.0 || t0 >= t) continue;
          t = t0;
        } else {
          const Sph& s = sc.sph[id - nc - nb];
          double B = -(dx * s.x + dy * s.y + dz * s.z);
          double C = s.x * s.x + s.y * s.y + s.z * s.z - s.r * s.r;
          double disc = B * B - C;
          if (disc <= 0.0) continue;
          double tt = -B - sqrt(disc);
          if (tt <= 0.0 || tt >= t) continue;
          t = tt;
        }
      }
      // the noise / dropout draws are made for every ray so that the stream does not depend on hits
      double noise = 0.02 * g.normal();
      bool drop = g.uni() < 0.01;
      if (t > kMaxRange || drop) continue;
      double r = t + noise;
      if (r < 0.3) continue;
      out[n].x = (float)(r * ds[0]);
      out[n].y = (float)(r * ds[1]);
      out[n].z = (float)(r * ds[2]);
      out[n].intensity = 0.0f;
      n++;
    }
  }
  return n;
}

int64_t generate_scan(int config, uint64_t scan_index, int A, fe_point_t* out, double* roll_pitch) {
  Rng g(scene_seed(config, scan_index));
  Scene sc;
  build_scene(config, g, sc);
  return render_scan(config, sc, g, A, out, roll_pitch);
}

// Runs scan(i, out_slot, roll_pitch + 2i) for i in [0, n_scans) on n_threads threads and packs the scans into `out`
// in order.  Returns 0, or 3 if cap_points is too small.
template <class F>
int generate_scans(int n_scans, int A, int n_threads, fe_point_t* out, int64_t cap_points, int64_t* scan_offsets,
                   double* roll_pitch, const F& scan) {
  const int64_t slot = 16LL * A;
  if (n_threads < 1) n_threads = 1;
  std::vector<int64_t> counts(n_scans, 0);
  // generate in blocks so that temporary memory stays bounded; each block's scans are produced
  // into per-scan slots and then compacted in order
  const int block = 256;
  std::vector<fe_point_t> tmp((size_t)slot * (size_t)std::min(block, std::max(n_scans, 1)));
  int64_t total = 0;
  scan_offsets[0] = 0;
  for (int b0 = 0; b0 < n_scans; b0 += block) {
    const int nb = std::min(block, n_scans - b0);
    std::atomic<int> next(0);
    auto worker = [&]() {
      for (;;) {
        int i = next.fetch_add(1);
        if (i >= nb) break;
        counts[b0 + i] = scan(b0 + i, tmp.data() + (size_t)i * slot, roll_pitch + 2 * (b0 + i));
      }
    };
    if (n_threads == 1) worker();
    else {
      std::vector<std::thread> th;
      for (int t = 0; t < n_threads; t++) th.emplace_back(worker);
      for (auto& t : th) t.join();
    }
    for (int i = 0; i < nb; i++) {
      int64_t c = counts[b0 + i];
      if (total + c > cap_points) return 3;
      memcpy(out + total, tmp.data() + (size_t)i * slot, (size_t)c * sizeof(fe_point_t));
      total += c;
      scan_offsets[b0 + i + 1] = total;
    }
  }
  return 0;
}

}  // namespace

extern "C" {

int fes_default_azimuth_steps(int config) { return config == 3 ? 7200 : 1800; }

// Generates scans [scan_index_base, scan_index_base + n_scans) of `config` (1..5, BASELINE.json
// configs) into `out` (capacity cap_points; 16*A*n_scans always suffices), CSR offsets into
// scan_offsets[n_scans+1], roll/pitch into roll_pitch[2*n_scans].  Returns 0, or 3 if cap_points
// is too small.
int fes_generate(int config, int64_t scan_index_base, int n_scans, int azimuth_steps, int n_threads,
                 fe_point_t* out, int64_t cap_points, int64_t* scan_offsets, double* roll_pitch) {
  const int A = azimuth_steps > 0 ? azimuth_steps : fes_default_azimuth_steps(config);
  const int cfg = config == 5 ? 2 : config;
  return generate_scans(n_scans, A, n_threads, out, cap_points, scan_offsets, roll_pitch,
                        [&](int i, fe_point_t* o, double* rp) {
                          return generate_scan(cfg, (uint64_t)(scan_index_base + i), A, o, rp);
                        });
}

// One scene seen from n_scans sensor poses: the scene of fes_generate's scan `scene_index` (same seed, same
// build_scene), rendered from poses[3s .. 3s+2] = (x, y, yaw) of the scene frame, in metres and radians.  Scan 0 draws
// roll, pitch and noise from the scene's generator where build_scene left it, exactly as fes_generate does, so scan 0
// at pose (0, 0, 0) is fes_generate's scan `scene_index` byte for byte.  Scan s >= 1 draws them from a generator of its
// own, seeded by (config, scene_index, s).  Outputs and return value as fes_generate.
int fes_generate_poses(int config, int64_t scene_index, int n_scans, int azimuth_steps, int n_threads,
                       const double* poses, fe_point_t* out, int64_t cap_points, int64_t* scan_offsets,
                       double* roll_pitch) {
  const int A = azimuth_steps > 0 ? azimuth_steps : fes_default_azimuth_steps(config);
  const int cfg = config == 5 ? 2 : config;
  const uint64_t seed = scene_seed(cfg, (uint64_t)scene_index);
  Rng g0(seed);
  Scene sc;
  build_scene(cfg, g0, sc);
  return generate_scans(n_scans, A, n_threads, out, cap_points, scan_offsets, roll_pitch,
                        [&](int i, fe_point_t* o, double* rp) {
                          Rng g = g0;
                          if (i > 0) g = Rng(seed ^ ((uint64_t)i * 0xD1B54A32D192ED03ull));
                          return render_scan(cfg, posed(sc, poses + 3 * i), g, A, o, rp);
                        });
}

}  // extern "C"
