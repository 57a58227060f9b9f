// SignedDistanceMap -i mask.nii[.gz] -o out.nii[.gz] [-p/--inside-positive bool] [-q/--squared bool]
//                   [-b/--background value]
// The signed Euclidean distance of every voxel to the contour of the object (mask != background), in
// the units of the image's spacing, written as float with the mask's header: negative inside the
// object unless -p, zero on its inner layer (SignedMaurerDistanceMapImageFilter; ife_cuda_signed_distance_map
// states the semantics).  The mask is read as unsigned short.
// The default is NOT squared, because a map in millimetres is what a tool user expects; this differs
// from the filter's ITK default (SquaredDistance on).
#include <cstdlib>
#include <iostream>
#include <string>

#include "ife/Context.h"
#include "ife/Filters/SignedMaurerDistanceMapImageFilter.h"
#include "ife/IO/NiftiIO.h"
#include "ife/Util/CmdLine.h"

const std::string VERSION("0.1");

int main(int argc, char* argv[]) {
  ife::CmdLine cmd("Signed Euclidean distance map of a mask.", VERSION);
  cmd.add("i", "input", "Path to input mask.", true, "", "path");
  cmd.add("o", "output", "Path to output distance map (float).", true, "", "path");
  cmd.add("p", "inside-positive", "Positive distances inside the object, negative outside.", false, "0", "boolean");
  cmd.add("q", "squared", "Write the squared distance.", false, "0", "boolean");
  cmd.add("b", "background", "Mask value of the background; every other value is the object.", false, "0", "unsigned short");
  int rc;
  if (!cmd.parse(argc, argv, &rc)) return rc;
  const std::string inPath(cmd.value("input")), outPath(cmd.value("output"));
  bool insidePositive = false, squared = false;
  if (!ife::CmdLine::to_bool(cmd.value("inside-positive"), &insidePositive)) {
    cmd.error("Couldn't read argument value from string '" + cmd.value("inside-positive") + "'", "-p", &rc);
    return rc;
  }
  if (!ife::CmdLine::to_bool(cmd.value("squared"), &squared)) {
    cmd.error("Couldn't read argument value from string '" + cmd.value("squared") + "'", "-q", &rc);
    return rc;
  }
  long background = 0;
  if (!ife::CmdLine::convert(cmd.value("background"), &background) || background < 0 || background > 65535) {
    cmd.error("Background must be an integer in [0, 65535], not '" + cmd.value("background") + "'", "-b", &rc);
    return rc;
  }

  try {
    auto mask = ife::nifti::Read<unsigned short>(inPath);
    auto filter = ife::SignedMaurerDistanceMapImageFilter<ife::Image<unsigned short> >::New();
    filter->SetInput(mask.get());
    filter->SetBackgroundValue((unsigned short)background);
    filter->SetInsideIsPositive(insidePositive);
    filter->SetSquaredDistance(squared);
    filter->Update();
    ife::nifti::Write(outPath, *filter->GetOutput());
  } catch (std::exception& e) {
    std::cerr << "Failed to process." << std::endl
              << "Input: " << inPath << std::endl
              << "Output: " << outPath << std::endl
              << "ExceptionObject: " << e.what() << std::endl;
    return EXIT_FAILURE;
  }
  return EXIT_SUCCESS;
}
