// Host-side mirror of itk::SignedMaurerDistanceMapImageFilter as recalled: SetInput / Update /
// GetOutput, the signed Euclidean distance of every voxel to the contour of the object
// (input != background value), computed on the GPU by ife_cuda_signed_distance_map
// (include/ife_cuda.h states the contour rule, the sign and the arithmetic).
// Defaults are ITK's: InsideIsPositive off, SquaredDistance ON, UseImageSpacing on, background 0.
// The input is an unsigned char or unsigned short image; it is binarised on the host (!= background)
// unless it already is uint8 with background 0.
#ifndef IFE_B200_SIGNED_MAURER_DISTANCE_MAP_IMAGE_FILTER_H
#define IFE_B200_SIGNED_MAURER_DISTANCE_MAP_IMAGE_FILTER_H
#include <memory>
#include <type_traits>
#include <vector>

#include "ife/Context.h"
#include "ife/Image.h"

namespace ife {

// The uint8 mask (!= background) the C ABI takes: the image's own buffer when it already is one,
// else a binarised copy in `scratch`.
template <typename TPixel>
const unsigned char* BinaryMaskBuffer(const Image<TPixel>& image, TPixel background, std::vector<unsigned char>& scratch) {
  static_assert(std::is_same<TPixel, unsigned char>::value || std::is_same<TPixel, unsigned short>::value,
                "masks are unsigned char or unsigned short images");
  if (std::is_same<TPixel, unsigned char>::value && background == 0)
    return reinterpret_cast<const unsigned char*>(image.GetBufferPointer());
  const size_t n = image.GetGeometry().voxels();
  const TPixel* p = image.GetBufferPointer();
  scratch.resize(n);
  for (size_t i = 0; i < n; ++i) scratch[i] = p[i] != background ? 1 : 0;
  return scratch.data();
}

template <typename TInputImage = Image<unsigned char>, typename TOutputImage = Image<float> >
class SignedMaurerDistanceMapImageFilter {
public:
  typedef SignedMaurerDistanceMapImageFilter Self;
  typedef std::shared_ptr<Self> Pointer;
  typedef TInputImage InputImageType;
  typedef TOutputImage OutputImageType;
  typedef typename TInputImage::PixelType InputPixelType;
  static_assert(std::is_same<typename TOutputImage::PixelType, float>::value, "the distance map is float");
  static Pointer New() { return Pointer(new Self()); }

  void SetInput(const InputImageType* image) { m_Image = image; }
  void SetInsideIsPositive(bool b) { m_InsideIsPositive = b; }
  bool GetInsideIsPositive() const { return m_InsideIsPositive; }
  void SetSquaredDistance(bool b) { m_Squared = b; }
  bool GetSquaredDistance() const { return m_Squared; }
  void SetUseImageSpacing(bool b) { m_UseImageSpacing = b; }
  bool GetUseImageSpacing() const { return m_UseImageSpacing; }
  void SetBackgroundValue(InputPixelType v) { m_Background = v; }
  InputPixelType GetBackgroundValue() const { return m_Background; }

  void Update() {
    if (!m_Image) throw ExceptionObject(IFE_E_INVALID, "SignedMaurerDistanceMapImageFilter: input not set");
    m_Image->UpdateSource();
    const Geometry& g = m_Image->GetGeometry();
    std::vector<unsigned char> scratch;
    const unsigned char* mask = BinaryMaskBuffer(*m_Image, m_Background, scratch);
    m_Output->SetGeometry(g);
    m_Output->Allocate();
    const double unit[3] = {1.0, 1.0, 1.0};
    const int flags = (m_InsideIsPositive ? IFE_SDM_INSIDE_POSITIVE : 0) | (m_Squared ? IFE_SDM_SQUARED : 0);
    CudaContext& c = CudaContext::Instance();
    c.Check(ife_cuda_signed_distance_map(c.Handle(), mask, m_Output->GetBufferPointer(), g.size.data(),
                                         m_UseImageSpacing ? g.spacing.data() : unit, flags, IFE_MEM_HOST));
  }
  void UpdateLargestPossibleRegion() { Update(); }
  OutputImageType* GetOutput() { return m_Output.get(); }

private:
  SignedMaurerDistanceMapImageFilter() : m_Output(OutputImageType::New()) { m_Output->SetSource([this]() { this->Update(); }); }
  const InputImageType* m_Image = nullptr;
  bool m_InsideIsPositive = false;
  bool m_Squared = true;
  bool m_UseImageSpacing = true;
  InputPixelType m_Background = InputPixelType();
  typename OutputImageType::Pointer m_Output;
};

}  // namespace ife
#endif
