// d2pc_offline -- roscore-free harness for the node classes of include/d2pc_b200/nodes.hpp.
//
//   d2pc_offline wire   <out.bin>
//       CPU only: serialises a small hand-made PointCloud2 and Image with ros_lite (self-test of the wire code).
//   d2pc_offline params <launch file> <name>...
//       CPU only: loads the launch file into a Bus and prints one line per name: "<name> number <value>" (%.17g),
//       "<name> string <value>" or "<name> missing" (the launch-file loader's number / string rule).
//   d2pc_offline node1  <launch file> <w> <h> <in.raw> <out.bin> [sec nsec]
//       BASELINE config 1/2 shape: one mono8 frame published on the node's (remapped) input topic; the
//       PointCloud2 received on the (remapped) output topic is written in ROS1 wire format.
//   d2pc_offline node1scan <launch file> <w> <h> <in.raw> <cloud.bin> <scan.bin>
//       node1 with the /scan subscriber too (scan_enable in the launch file): the PointCloud2 (an empty file when
//       none was published) and the LaserScan in ROS1 wire format.
//   d2pc_offline fusion <fusion launch> <w> <h> <d1.raw> <d2.raw> <s1.raw> <s2.raw> <fused.bin> [<cloud.bin> [<debug dir>]]
//       BASELINE config 5 shape: four mono8 frames into DepthMapFusion; the fused Image is written, and when
//       <cloud.bin> is given it is also fed to a Disparity2PCloud node whose /disparity is remapped to
//       /fused_depth_map.  With <debug dir> the six debug topics are subscribed too and the last message of
//       each is written there in wire format (cropped_depth_1.bin, ..., gradient.bin).
//   d2pc_offline fusion-seq <fusion launch> <w> <h> <script.txt> <out.bin>
//       An arbitrary callback sequence into one DepthMapFusion node: every script line is
//       "<which> <frame.raw> <sec> <nsec>" with which = 1 /disparity_1, 2 /disparity_2, 3 /matching_score_1,
//       4 /matching_score_2.  Every message the node publishes on any of its seven topics is appended to <out.bin>
//       in publish order as {u32 topic length, topic, u32 wire length, ROS1 wire bytes}.  This is how the state the
//       node keeps BETWEEN callbacks is tested (src/depth_map_fusion.cpp:77, :113, :118-121: after a fused publish the
//       cached score 1 is min(score 1, score 2) until the next MatchingScoreCb1).
//
// It touches the GPU only through the C ABI (libd2pc_b200.so).
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <map>
#include <string>
#include <vector>

#include "d2pc_b200/nodes.hpp"

namespace sm = ros_lite::sensor_msgs;

static std::vector<uint8_t> read_file(const std::string &path, size_t expect) {
  std::ifstream in(path, std::ios::binary);
  std::vector<uint8_t> d((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
  if (!in.good() && d.empty()) throw std::runtime_error("cannot read " + path);
  if (expect && d.size() != expect) throw std::runtime_error(path + ": unexpected size");
  return d;
}
static void write_file(const std::string &path, const std::vector<uint8_t> &d) {
  std::ofstream out(path, std::ios::binary);
  out.write(reinterpret_cast<const char *>(d.data()), (std::streamsize)d.size());
}
static sm::ImagePtr make_image(const std::vector<uint8_t> &px, uint32_t w, uint32_t h, uint32_t sec, uint32_t nsec) {
  auto m = std::make_shared<sm::Image>();
  m->header.seq = 0;
  m->header.stamp.sec = sec;
  m->header.stamp.nsec = nsec;
  m->header.frame_id = "camera";
  m->height = h, m->width = w, m->encoding = "mono8", m->is_bigendian = 0, m->step = w;
  m->data = px;
  return m;
}

int main(int argc, char **argv) {
  try {
    const std::string mode = argc > 1 ? argv[1] : "";
    if (mode == "wire" && argc == 3) {
      sm::PointCloud2 c;
      c.header.seq = 7, c.header.stamp.sec = 11, c.header.stamp.nsec = 13, c.header.frame_id = "/camera_optical_frame";
      c.height = 1, c.width = 2;
      const char *names[3] = {"x", "y", "z"};
      for (uint32_t i = 0; i < 3; ++i) c.fields.push_back({names[i], 4 * i, sm::PointField::FLOAT32, 1});
      c.point_step = 16, c.row_step = 32;
      for (int i = 0; i < 32; ++i) c.data.push_back((uint8_t)i);
      auto bytes = ros_lite::serialize(c);
      auto back = ros_lite::deserialize_pointcloud2(bytes.data(), bytes.size());
      if (ros_lite::serialize(back) != bytes) throw std::runtime_error("PointCloud2 round trip differs");
      sm::Image im = *make_image({1, 2, 3, 4, 5, 6}, 3, 2, 5, 6);
      auto ib = ros_lite::serialize(im);
      auto im2 = ros_lite::deserialize_image(ib.data(), ib.size());
      if (ros_lite::serialize(im2) != ib || im2.encoding != "mono8") throw std::runtime_error("Image round trip differs");
      sm::LaserScan sc;
      sc.header = c.header;
      sc.angle_min = -1.5f, sc.angle_max = 1.5f, sc.angle_increment = 0.75f, sc.scan_time = 0.25f, sc.range_max = 9.f;
      sc.ranges = {1.f, 2.f, 3.f, 4.f};
      auto sb = ros_lite::serialize(sc);
      auto sc2 = ros_lite::deserialize_laserscan(sb.data(), sb.size());
      if (ros_lite::serialize(sc2) != sb || sb.size() != 16 + 21 + 28 + 4 + 16 + 4)
        throw std::runtime_error("LaserScan round trip differs");
      write_file(argv[2], bytes);
      return 0;
    }
    if (mode == "node1scan" && argc == 8) {
      const uint32_t w = (uint32_t)std::atoi(argv[3]), h = (uint32_t)std::atoi(argv[4]);
      d2pc_b200::Bus bus;
      if (!bus.load_launch_file(argv[2])) throw std::runtime_error(std::string("cannot read ") + argv[2]);
      d2pc::Disparity2PCloud node(bus);
      std::vector<uint8_t> cloud, scan;
      bus.subscribe_cloud("/point_cloud", 1, [&](const sm::PointCloud2 &c) { cloud = ros_lite::serialize(c); });
      bus.subscribe_scan("/scan", 1, [&](const sm::LaserScan &s) { scan = ros_lite::serialize(s); });
      bus.publish(bus.resolve("/disparity"), make_image(read_file(argv[5], (size_t)w * h), w, h, 3, 4));
      if (scan.empty()) throw std::runtime_error("no scan was published");
      write_file(argv[6], cloud);
      write_file(argv[7], scan);
      return 0;
    }
    if (mode == "params" && argc >= 3) {
      d2pc_b200::Bus bus;
      if (!bus.load_launch_file(argv[2])) throw std::runtime_error(std::string("cannot read ") + argv[2]);
      for (int i = 3; i < argc; ++i) {
        double v = 0.0;
        std::string str;
        if (bus.get_param(argv[i], v))
          std::printf("%s number %.17g\n", argv[i], v);
        else if (bus.get_param(argv[i], str))
          std::printf("%s string %s\n", argv[i], str.c_str());
        else
          std::printf("%s missing\n", argv[i]);
      }
      return 0;
    }
    if (mode == "node1" && argc >= 7) {
      const uint32_t w = (uint32_t)std::atoi(argv[3]), h = (uint32_t)std::atoi(argv[4]);
      const uint32_t sec = argc > 7 ? (uint32_t)std::strtoul(argv[7], nullptr, 10) : 0;
      const uint32_t nsec = argc > 8 ? (uint32_t)std::strtoul(argv[8], nullptr, 10) : 0;
      d2pc_b200::Bus bus;
      if (!bus.load_launch_file(argv[2])) throw std::runtime_error(std::string("cannot read ") + argv[2]);
      d2pc::Disparity2PCloud node(bus);
      std::vector<uint8_t> got;
      bus.subscribe_cloud("/point_cloud", 1, [&](const sm::PointCloud2 &c) { got = ros_lite::serialize(c); });
      bus.publish(bus.resolve("/disparity"), make_image(read_file(argv[5], (size_t)w * h), w, h, sec, nsec));
      if (got.empty()) throw std::runtime_error("no point cloud was published");
      write_file(argv[6], got);
      return 0;
    }
    if (mode == "fusion" && argc >= 10) {
      const uint32_t w = (uint32_t)std::atoi(argv[3]), h = (uint32_t)std::atoi(argv[4]);
      d2pc_b200::Bus bus;
      if (!bus.load_launch_file(argv[2])) throw std::runtime_error(std::string("cannot read ") + argv[2]);
      depth_map_fusion::DepthMapFusion fusion(bus);
      std::vector<uint8_t> fused_bytes, cloud_bytes;
      sm::ImageConstPtr fused;
      bus.subscribe_image("/fused_depth_map", 5, [&](const sm::ImageConstPtr &m) {
        fused = m;
        fused_bytes = ros_lite::serialize(*m);
      });
      // the reference would start node 1 with <remap from="/disparity" to="/fused_depth_map"/>
      std::unique_ptr<d2pc_b200::Bus> bus1;
      std::unique_ptr<d2pc::Disparity2PCloud> node1;
      if (argc > 10) {
        bus1.reset(new d2pc_b200::Bus());
        bus1->remap("/disparity", "/fused_depth_map");
        node1.reset(new d2pc::Disparity2PCloud(*bus1));
        bus1->subscribe_cloud("/point_cloud", 1, [&](const sm::PointCloud2 &c) { cloud_bytes = ros_lite::serialize(c); });
      }
      std::map<std::string, std::vector<uint8_t>> debug;
      if (argc > 11)
        for (const char *t : {"cropped_depth_1", "cropped_depth_2", "cropped_score_1", "cropped_score_2", "combined_score",
                              "gradient"})
          bus.subscribe_image(std::string("/") + t, 5,
                              [&debug, t](const sm::ImageConstPtr &m) { debug[t] = ros_lite::serialize(*m); });
      // arrival order of the reference's typical use: scores, map 1, then map 2 triggers the fused publish
      bus.publish(bus.resolve("/matching_score_1"), make_image(read_file(argv[7], (size_t)w * h), w, h, 1, 0));
      bus.publish(bus.resolve("/matching_score_2"), make_image(read_file(argv[8], (size_t)w * h), w, h, 1, 0));
      bus.publish(bus.resolve("/disparity_1"), make_image(read_file(argv[5], (size_t)w * h), w, h, 1, 0));
      bus.publish(bus.resolve("/disparity_2"), make_image(read_file(argv[6], (size_t)w * h), w, h, 2, 500));
      if (fused_bytes.empty()) throw std::runtime_error("no fused depth map was published");
      write_file(argv[9], fused_bytes);
      if (node1) {
        bus1->publish("/fused_depth_map", fused);
        if (cloud_bytes.empty()) throw std::runtime_error("no point cloud was published");
        write_file(argv[10], cloud_bytes);
      }
      if (argc > 11) {
        if (debug.size() != 6) throw std::runtime_error("a debug topic was not published");
        for (const auto &kv : debug) write_file(std::string(argv[11]) + "/" + kv.first + ".bin", kv.second);
      }
      return 0;
    }
    if (mode == "fusion-seq" && argc == 7) {
      const uint32_t w = (uint32_t)std::atoi(argv[3]), h = (uint32_t)std::atoi(argv[4]);
      d2pc_b200::Bus bus;
      if (!bus.load_launch_file(argv[2])) throw std::runtime_error(std::string("cannot read ") + argv[2]);
      depth_map_fusion::DepthMapFusion fusion(bus);
      std::vector<uint8_t> log;
      auto put32 = [&log](uint32_t v) {
        for (int i = 0; i < 4; ++i) log.push_back((uint8_t)(v >> (8 * i)));
      };
      for (const char *t : {"cropped_depth_1", "cropped_depth_2", "cropped_score_1", "cropped_score_2", "combined_score",
                            "gradient", "fused_depth_map"}) {
        const std::string topic = std::string("/") + t;
        bus.subscribe_image(topic, 5, [&log, &put32, topic](const sm::ImageConstPtr &m) {
          const std::vector<uint8_t> wire = ros_lite::serialize(*m);
          put32((uint32_t)topic.size());
          log.insert(log.end(), topic.begin(), topic.end());
          put32((uint32_t)wire.size());
          log.insert(log.end(), wire.begin(), wire.end());
        });
      }
      const char *inputs[5] = {"", "/disparity_1", "/disparity_2", "/matching_score_1", "/matching_score_2"};
      std::ifstream script(argv[5]);
      if (!script) throw std::runtime_error(std::string("cannot read ") + argv[5]);
      int which;
      std::string path;
      uint32_t sec, nsec, seq = 0;
      while (script >> which >> path >> sec >> nsec) {
        if (which < 1 || which > 4) throw std::runtime_error("fusion-seq: which must be 1..4");
        auto m = make_image(read_file(path, (size_t)w * h), w, h, sec, nsec);
        m->header.seq = seq++;
        bus.publish(bus.resolve(inputs[which]), m);
      }
      write_file(argv[6], log);
      return 0;
    }
    std::fprintf(stderr, "usage: see the header of tools/d2pc_offline.cpp\n");
    return 2;
  } catch (const std::exception &e) {
    std::fprintf(stderr, "d2pc_offline: %s\n", e.what());
    return 1;
  }
}
