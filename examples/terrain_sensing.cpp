// World::rayTest against the terrain the robot collides with: vertical rays on a random HeightMap against HeightMap::getHeight, a
// slanted ray on a Ground against the closed form, and the refusal of closestOnly = false.  One line per check; non-zero exit on failure.
#include <cmath>
#include <cstdio>
#include <random>
#include <stdexcept>
#include <string>
#include <vector>
#include "raisim/World.hpp"

int main(int argc, char** argv) {
  std::string urdf = argc > 1 ? argv[1] : "raisimlib_b200/rsc/anymal_c_like.urdf";
  int failures = 0;
  {
    raisim::World world;
    world.addArticulatedSystem(urdf);
    const size_t xs = 97, ys = 81;
    std::mt19937 gen(7);
    std::uniform_real_distribution<double> u(-0.3, 0.3);
    std::vector<double> h(xs * ys);
    for (double& z : h) z = u(gen);
    raisim::HeightMap* hm = world.addHeightMap(xs, ys, 9.6, 8.0, 1.5, -0.5, h);
    std::uniform_real_distribution<double> px(1.5 - 4.7, 1.5 + 4.7), py(-0.5 - 3.9, -0.5 + 3.9);
    double worst = 0; int misses = 0;
    for (int k = 0; k < 200; k++) {
      const double x = px(gen), y = py(gen);
      const auto& hits = world.rayTest({x, y, 2.0}, {0.0, 0.0, -1.0}, 5.0);
      if (hits.size() != 1) { misses++; continue; }
      const raisim::Vec<3> p = hits[0].getPosition();
      // float32 ray arithmetic over a 2 m drop: ~1e-6 m; the height map holds float32 heights on both sides
      worst = std::fmax(worst, std::fabs(p[2] - hm->getHeight(x, y)));
      worst = std::fmax(worst, std::fabs(hits[0].getDistance() - (2.0 - hm->getHeight(x, y))));
    }
    const bool ok = misses == 0 && worst < 2e-5;
    std::printf("vertical rayTest vs HeightMap::getHeight: 200 rays, %d misses, max |dz| %.2e m  %s\n", misses, worst, ok ? "ok" : "FAIL");
    failures += !ok;
  }
  {
    raisim::World world;
    world.addArticulatedSystem(urdf);
    world.addGround(0.25);
    const double o[3] = {0.3, -1.2, 1.75}, d[3] = {2.0, 1.0, -3.0};     // not normalised: rayTest normalises
    const double n = std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    const double t = (0.25 - o[2]) / (d[2] / n);
    const auto& hits = world.rayTest({o[0], o[1], o[2]}, {d[0], d[1], d[2]}, 10.0);
    double err = 1.0;
    if (hits.size() == 1) {
      const raisim::Vec<3> p = hits[0].getPosition(), nm = hits[0].getNormal();
      err = std::fabs(hits[0].getDistance() - t);
      for (int k = 0; k < 3; k++) err = std::fmax(err, std::fabs(p[k] - (o[k] + t * d[k] / n)));
      err = std::fmax(err, std::fabs(nm[0]) + std::fabs(nm[1]) + std::fabs(nm[2] - 1.0));
      if (hits[0].getPairIndex() != 0) err = 1.0;
    }
    const auto& none = world.rayTest({o[0], o[1], o[2]}, {d[0], d[1], d[2]}, 0.9 * t);       // too short to reach the plane
    const bool ok = err < 1e-6 && none.size() == 0;
    std::printf("slanted rayTest on a Ground vs closed form: t = %.6f, max error %.2e, short ray %s  %s\n", t, err, none.size() ? "hit" : "missed", ok ? "ok" : "FAIL");
    failures += !ok;
    bool threw = false;
    try { world.rayTest({0.0, 0.0, 1.0}, {0.0, 0.0, -1.0}, 2.0, false); } catch (const std::runtime_error&) { threw = true; }
    std::printf("rayTest(closestOnly = false) refused: %s  %s\n", threw ? "yes" : "no", threw ? "ok" : "FAIL");
    failures += !threw;
  }
  return failures ? 1 : 0;
}
