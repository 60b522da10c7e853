// ros_lite.hpp -- the handful of ROS1 message types the two nodes exchange, as plain structs with the ROS1
// wire (de)serialisation, so the node classes in nodes.hpp compile and run without a ROS installation.
// Field order and types follow the message definitions the reference uses:
//   std_msgs/Header, sensor_msgs/Image, sensor_msgs/PointField, sensor_msgs/PointCloud2, and sensor_msgs/LaserScan
//   (pointcloud_to_laserscan's output, which the point cloud node can publish next to its cloud)
//   (src/disparity_to_point_cloud.cpp:46-92, src/depth_map_fusion.cpp:46-136).
// With a real ROS1 the ros1_shim/ sources use the genuine sensor_msgs types instead; the layouts are identical.
#pragma once
#include <cstdint>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace ros_lite {

struct Time {
  uint32_t sec = 0, nsec = 0;
};

struct Header {
  uint32_t seq = 0;
  Time stamp;
  std::string frame_id;
};

namespace sensor_msgs {

struct Image {
  Header header;
  uint32_t height = 0, width = 0;
  std::string encoding;
  uint8_t is_bigendian = 0;
  uint32_t step = 0;
  std::vector<uint8_t> data;
};
using ImagePtr = std::shared_ptr<Image>;
using ImageConstPtr = std::shared_ptr<const Image>;

struct PointField {
  enum : uint8_t { INT8 = 1, UINT8, INT16, UINT16, INT32, UINT32, FLOAT32, FLOAT64 };
  std::string name;
  uint32_t offset = 0;
  uint8_t datatype = 0;
  uint32_t count = 0;
};

struct PointCloud2 {
  Header header;
  uint32_t height = 0, width = 0;
  std::vector<PointField> fields;
  uint8_t is_bigendian = 0;
  uint32_t point_step = 0, row_step = 0;
  std::vector<uint8_t> data;
  uint8_t is_dense = 0;
};

struct LaserScan {
  Header header;
  float angle_min = 0, angle_max = 0, angle_increment = 0, time_increment = 0, scan_time = 0, range_min = 0,
        range_max = 0;
  std::vector<float> ranges, intensities;
};

}  // namespace sensor_msgs

// ---- ROS1 serialisation: little endian, strings and arrays prefixed by a uint32 length --------------------
class Writer {
 public:
  std::vector<uint8_t> buf;
  void u8(uint8_t v) { buf.push_back(v); }
  void u32(uint32_t v) {
    uint8_t b[4];
    std::memcpy(b, &v, 4);
    buf.insert(buf.end(), b, b + 4);
  }
  void str(const std::string &s) {
    u32(static_cast<uint32_t>(s.size()));
    buf.insert(buf.end(), s.begin(), s.end());
  }
  void bytes(const std::vector<uint8_t> &d) {
    u32(static_cast<uint32_t>(d.size()));
    buf.insert(buf.end(), d.begin(), d.end());
  }
  void f32(float v) {
    uint8_t b[4];
    std::memcpy(b, &v, 4);
    buf.insert(buf.end(), b, b + 4);
  }
  void floats(const std::vector<float> &d) {
    u32(static_cast<uint32_t>(d.size()));
    for (float v : d) f32(v);
  }
  void header(const Header &h) {
    u32(h.seq), u32(h.stamp.sec), u32(h.stamp.nsec), str(h.frame_id);
  }
};

class Reader {
 public:
  Reader(const uint8_t *p, size_t n) : p_(p), end_(p + n) {}
  uint8_t u8() {
    need(1);
    return *p_++;
  }
  uint32_t u32() {
    need(4);
    uint32_t v;
    std::memcpy(&v, p_, 4);
    p_ += 4;
    return v;
  }
  std::string str() {
    const uint32_t n = u32();
    need(n);
    std::string s(reinterpret_cast<const char *>(p_), n);
    p_ += n;
    return s;
  }
  std::vector<uint8_t> bytes() {
    const uint32_t n = u32();
    need(n);
    std::vector<uint8_t> d(p_, p_ + n);
    p_ += n;
    return d;
  }
  float f32() {
    const uint32_t b = u32();
    float v;
    std::memcpy(&v, &b, 4);
    return v;
  }
  std::vector<float> floats() {
    const uint32_t n = u32();
    need(static_cast<size_t>(n) * 4);
    std::vector<float> d(n);
    for (auto &v : d) v = f32();
    return d;
  }
  Header header() {
    Header h;
    h.seq = u32(), h.stamp.sec = u32(), h.stamp.nsec = u32(), h.frame_id = str();
    return h;
  }
  bool done() const { return p_ == end_; }

 private:
  void need(size_t n) {
    if (static_cast<size_t>(end_ - p_) < n) throw std::runtime_error("ros_lite: truncated message");
  }
  const uint8_t *p_, *end_;
};

inline std::vector<uint8_t> serialize(const sensor_msgs::Image &m) {
  Writer w;
  w.header(m.header);
  w.u32(m.height), w.u32(m.width), w.str(m.encoding), w.u8(m.is_bigendian), w.u32(m.step), w.bytes(m.data);
  return std::move(w.buf);
}
inline sensor_msgs::Image deserialize_image(const uint8_t *p, size_t n) {
  Reader r(p, n);
  sensor_msgs::Image m;
  m.header = r.header();
  m.height = r.u32(), m.width = r.u32(), m.encoding = r.str(), m.is_bigendian = r.u8(), m.step = r.u32();
  m.data = r.bytes();
  return m;
}
inline std::vector<uint8_t> serialize(const sensor_msgs::PointCloud2 &m) {
  Writer w;
  w.header(m.header);
  w.u32(m.height), w.u32(m.width);
  w.u32(static_cast<uint32_t>(m.fields.size()));
  for (const auto &f : m.fields) w.str(f.name), w.u32(f.offset), w.u8(f.datatype), w.u32(f.count);
  w.u8(m.is_bigendian), w.u32(m.point_step), w.u32(m.row_step), w.bytes(m.data), w.u8(m.is_dense);
  return std::move(w.buf);
}
inline sensor_msgs::PointCloud2 deserialize_pointcloud2(const uint8_t *p, size_t n) {
  Reader r(p, n);
  sensor_msgs::PointCloud2 m;
  m.header = r.header();
  m.height = r.u32(), m.width = r.u32();
  const uint32_t nf = r.u32();
  for (uint32_t i = 0; i < nf; ++i) {
    sensor_msgs::PointField f;
    f.name = r.str(), f.offset = r.u32(), f.datatype = r.u8(), f.count = r.u32();
    m.fields.push_back(f);
  }
  m.is_bigendian = r.u8(), m.point_step = r.u32(), m.row_step = r.u32(), m.data = r.bytes(), m.is_dense = r.u8();
  return m;
}
inline std::vector<uint8_t> serialize(const sensor_msgs::LaserScan &m) {
  Writer w;
  w.header(m.header);
  w.f32(m.angle_min), w.f32(m.angle_max), w.f32(m.angle_increment), w.f32(m.time_increment), w.f32(m.scan_time);
  w.f32(m.range_min), w.f32(m.range_max), w.floats(m.ranges), w.floats(m.intensities);
  return std::move(w.buf);
}
inline sensor_msgs::LaserScan deserialize_laserscan(const uint8_t *p, size_t n) {
  Reader r(p, n);
  sensor_msgs::LaserScan m;
  m.header = r.header();
  m.angle_min = r.f32(), m.angle_max = r.f32(), m.angle_increment = r.f32(), m.time_increment = r.f32();
  m.scan_time = r.f32(), m.range_min = r.f32(), m.range_max = r.f32();
  m.ranges = r.floats(), m.intensities = r.floats();
  return m;
}

}  // namespace ros_lite
