// Segment lists from Python: an (S, 2) array of 64-bit integers (numpy uint64 / int64, or a CPU torch int64 tensor),
// row = (device pointer, byte length).  Read in place through the buffer protocol: no Python object per segment.
#pragma once
#include <pybind11/pybind11.h>

#include <cstring>
#include <stdexcept>

#include "common/types.h"

namespace bb::py_segments {

struct SegmentArray {
  pybind11::buffer_info info;  // keeps the exporting array alive and its memory in place
  const DeviceSegment* data = nullptr;
  size_t count = 0;
};

// True for objects read_segments() takes (anything but an int, a list or a tuple).
inline bool is_segment_array(const pybind11::handle& obj) {
  return !pybind11::isinstance<pybind11::int_>(obj) && !pybind11::isinstance<pybind11::list>(obj) &&
         !pybind11::isinstance<pybind11::tuple>(obj);
}

inline SegmentArray read_segments(const pybind11::handle& obj) {
  namespace py = pybind11;
  py::object src = py::reinterpret_borrow<py::object>(obj);
  if (!py::isinstance<py::buffer>(src)) {
    if (!py::hasattr(src, "numpy")) throw py::type_error("segments: an (S, 2) uint64 / int64 array or CPU tensor");
    if (py::hasattr(src, "is_cuda") && src.attr("is_cuda").cast<bool>()) throw py::type_error("segments: the table must be a CPU tensor");
    src = src.attr("numpy")();  // CPU torch tensor: zero-copy numpy view
  }
  SegmentArray a;
  a.info = py::reinterpret_borrow<py::buffer>(src).request();
  const std::string& f = a.info.format;
  const bool int64 = a.info.itemsize == 8 && (f == "Q" || f == "q" || f == "L" || f == "l" || f == "<Q" || f == "<q" || f == "<l" || f == "<L");
  if (!int64 || a.info.ndim != 2 || a.info.shape[1] != 2) throw py::value_error("segments: expected an (S, 2) array of 64-bit integers");
  if (a.info.shape[0] > 0 && (a.info.strides[1] != 8 || a.info.strides[0] != 16))
    throw py::value_error("segments: the array must be C-contiguous");
  a.data = static_cast<const DeviceSegment*>(a.info.ptr);
  a.count = static_cast<size_t>(a.info.shape[0]);
  static_assert(sizeof(DeviceSegment) == 16);
  return a;
}

}  // namespace bb::py_segments
