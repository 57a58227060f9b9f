// ExpectedDistance -c center_mask.nii[.gz] -w weight.nii[.gz] [-m region_mask.nii[.gz]] [-p/--inside-positive bool]
// Prints, on one line, the weight-weighted mean of the signed distance to the contour of the center mask
// (!= 0), over the voxels where the region mask is != 0 (every voxel without -m): for a probability map
// from a classifier, how far from the structure that probability sits, in the units of the images'
// spacing, negative inside it unless -p (ExpectedDistanceFromCenterToInterestPoint.h,
// ife_cuda_expected_signed_distance).  Masks are read as unsigned short, the weight image as float;
// the three images must have one geometry.  The value is printed with 17 significant digits.
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <string>
#include <vector>

#include "ife/Context.h"
#include "ife/IO/NiftiIO.h"
#include "ife/Statistics/ExpectedDistanceFromCenterToInterestPoint.h"
#include "ife/Util/CmdLine.h"

const std::string VERSION("0.1");

static ife::Image<unsigned char>::Pointer ReadBinaryMask(const std::string& path) {
  auto m16 = ife::nifti::Read<unsigned short>(path);
  auto m = ife::Image<unsigned char>::New();
  m->SetGeometry(m16->GetGeometry());
  m->Allocate();
  const unsigned short* p = m16->GetBufferPointer();
  unsigned char* q = m->GetBufferPointer();
  for (size_t i = 0; i < m16->GetGeometry().voxels(); ++i) q[i] = p[i] != 0 ? 1 : 0;
  return m;
}

static bool SameGeometry(const ife::Geometry& a, const ife::Geometry& b) {
  return a.size == b.size && a.spacing == b.spacing && a.origin == b.origin;
}

int main(int argc, char* argv[]) {
  ife::CmdLine cmd("Probability-weighted mean signed distance to the contour of a mask.", VERSION);
  cmd.add("c", "center", "Path to center mask.", true, "", "path");
  cmd.add("w", "weight", "Path to weight (probability) image.", true, "", "path");
  cmd.add("m", "region", "Path to region mask restricting the mean (default: every voxel).", false, "", "path");
  cmd.add("p", "inside-positive", "Positive distances inside the center mask, negative outside.", false, "0", "boolean");
  int rc;
  if (!cmd.parse(argc, argv, &rc)) return rc;
  const std::string centerPath(cmd.value("center")), weightPath(cmd.value("weight")), regionPath(cmd.value("region"));
  bool insidePositive = false;
  if (!ife::CmdLine::to_bool(cmd.value("inside-positive"), &insidePositive)) {
    cmd.error("Couldn't read argument value from string '" + cmd.value("inside-positive") + "'", "-p", &rc);
    return rc;
  }

  try {
    auto center = ReadBinaryMask(centerPath);
    auto weight = ife::nifti::Read<float>(weightPath);
    ife::Image<unsigned char>::Pointer region;
    if (!regionPath.empty()) region = ReadBinaryMask(regionPath);
    if (!SameGeometry(center->GetGeometry(), weight->GetGeometry()) ||
        (region && !SameGeometry(center->GetGeometry(), region->GetGeometry())))
      throw std::runtime_error("the input images' geometries differ");
    const double e = ife::ExpectedDistanceFromCenterToInterestPoint(*center, *weight, region.get(), insidePositive);
    std::printf("%.17g\n", e);
  } catch (std::exception& e) {
    std::cerr << "Failed to process." << std::endl
              << "Center: " << centerPath << std::endl
              << "Weight: " << weightPath << std::endl
              << "ExceptionObject: " << e.what() << std::endl;
    return EXIT_FAILURE;
  }
  return EXIT_SUCCESS;
}
