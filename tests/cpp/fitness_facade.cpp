// fitness_facade.cpp — compile-and-run check of NanoGICP::getFitnessScore in the drop-in facade: a scan-to-scan
// registration with a host target, the same with the target assembled on the device by KeyframeStore::setTarget, and
// a handle without a target (PCL-style message, DBL_MAX).
// Input : [int32 n_tgt][n_tgt*8 float][int32 n_src][n_src*8 float][double max_range]   (pcl::PointXYZI records)
// Output: one JSON line per case with the final transformation (column-major) and getFitnessScore() /
//         getFitnessScore(max_range), printed with 17 significant digits.
#include <cstdio>
#include <string>
#include <vector>

#include <nano_gicp/nano_gicp.hpp>

typedef pcl::PointXYZI PointType;
typedef nano_gicp::NanoGICP<PointType, PointType> Gicp;

static bool read_cloud(FILE* f, pcl::PointCloud<PointType>::Ptr& c) {
  int n = 0;
  if (std::fread(&n, 4, 1, f) != 1 || n < 0) return false;
  c.reset(new pcl::PointCloud<PointType>);
  c->resize((size_t)n);
  return std::fread(c->points.data(), sizeof(PointType), (size_t)n, f) == (size_t)n;
}

static void configure(Gicp& g) {   // cfg/params.yaml S2S values
  g.setCorrespondenceRandomness(10);
  g.setMaxCorrespondenceDistance(1.0);
  g.setMaximumIterations(32);
  g.setTransformationEpsilon(0.01);
}

static void print_case(const char* name, Gicp& g, double max_range) {
  const Eigen::Matrix4f T = g.getFinalTransformation();
  std::printf("{\"case\": \"%s\", \"T\": [", name);
  for (int i = 0; i < 16; i++) std::printf("%s%.9g", i ? ", " : "", T.data()[i]);
  const double s = g.getFitnessScore();
  const double sr = g.getFitnessScore(max_range);
  std::printf("], \"score\": %.17g, \"score_r\": %.17g}\n", s, sr);
}

int main(int argc, char** argv) {
  if (argc < 2) { std::fprintf(stderr, "usage: %s clouds.bin\n", argv[0]); return 2; }
  FILE* f = std::fopen(argv[1], "rb");
  if (!f) { std::perror("open"); return 2; }
  pcl::PointCloud<PointType>::Ptr tgt, src;
  double max_range = 0.0;
  if (!read_cloud(f, tgt) || !read_cloud(f, src) || std::fread(&max_range, 8, 1, f) != 1) return 2;
  std::fclose(f);

  Gicp gicp;
  if (!gicp.handle()) return 3;   // no GPU: fail loudly
  configure(gicp);
  gicp.setInputTarget(tgt);
  gicp.setInputSource(src);
  pcl::PointCloud<PointType> aligned;
  gicp.align(aligned);
  print_case("host_target", gicp, max_range);

  // the same target assembled on the device: keyframe = the target cloud with its covariances
  Gicp keyer, dev;
  configure(keyer);
  configure(dev);
  keyer.setInputSource(tgt);
  keyer.calculateSourceCovariances();
  nano_gicp::KeyframeStore store;
  store.push(keyer);
  store.setTarget(dev, std::vector<int>{0});
  dev.setInputSource(src);
  dev.align(aligned);
  print_case("kfstore_target", dev, max_range);

  Gicp lonely;
  lonely.setInputSource(src);
  std::printf("{\"case\": \"no_target\", \"score\": %.17g}\n", lonely.getFitnessScore());
  return 0;
}
