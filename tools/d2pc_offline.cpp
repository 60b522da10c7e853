// d2pc_offline -- roscore-free harness for the node classes of include/d2pc_b200/nodes.hpp.
//
//   d2pc_offline wire   <out.bin>
//       CPU only: serialises a small hand-made PointCloud2 and Image with ros_lite (self-test of the wire code).
//   d2pc_offline wire-octomap <out.bin>
//       CPU only: a small hand-made octomap_msgs/Octomap through ros_lite's serialize / deserialize; its wire bytes.
//   d2pc_offline wire-grid <out.bin>
//       CPU only: a small hand-made nav_msgs/OccupancyGrid through ros_lite's serialize / deserialize; its wire bytes.
//   d2pc_offline params <launch file> <name>...
//       CPU only: loads the launch file into a Bus and prints one line per name: "<name> number <value>" (%.17g),
//       "<name> string <value>" or "<name> missing" (the launch-file loader's number / string rule).
//   d2pc_offline node1settings <launch file>
//       CPU only: the point cloud node's settings as read from the launch file (d2pc_b200::read_cloud_settings), one
//       "<field> <value>" line per field of d2pc_b200::CloudSettings (numbers %.17g, arrays as <field>.<index>).
//   d2pc_offline node1  <launch file> <w> <h> <in.raw> <out.bin> [sec nsec]
//       BASELINE config 1/2 shape: one mono8 frame published on the node's (remapped) input topic; the
//       PointCloud2 received on the (remapped) output topic is written in ROS1 wire format.
//   d2pc_offline node1scan <launch file> <w> <h> <in.raw> <cloud.bin> <scan.bin>
//       node1 with the /scan subscriber too (scan_enable in the launch file): the PointCloud2 (an empty file when
//       none was published) and the LaserScan in ROS1 wire format.
//   d2pc_offline node1map <launch file> <w> <h> <cloud.bin> <centres.bin> <in.raw> [<in.raw> ...]
//       node1 with the map on (map_enable in the launch file), one frame per <in.raw> stamped (3 + i, 4): the last
//       PointCloud2 (an empty file when none was published) and the last /octomap_point_cloud_centers cloud.
//   d2pc_offline node1octomap <launch file> <w> <h> <cloud.bin> <centres.bin> <full.bin> <binary.bin> <in.raw>...
//       node1map with /octomap_full and /octomap_binary subscribed too: the last message of each (an empty file when
//       none was published); a path of "-" leaves that topic without a subscriber.  With map_enable 0 in the launch file nothing is subscribed but /point_cloud, and the
//       harness fails if the node advertised any octomap topic.
//   d2pc_offline node1projmap <launch file> <w> <h> <cloud.bin> <grid.bin> <count.txt> <in.raw> [<in.raw> ...]
//       node1 with the map on and /projected_map subscribed: the last PointCloud2 and the last OccupancyGrid (an empty
//       file when none was published), and the number of grids published.  With map_enable 0 in the launch file
//       only /point_cloud is subscribed, and the harness fails if the node advertised /projected_map.
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
    if (mode == "node1map" && argc >= 8) {
      const uint32_t w = (uint32_t)std::atoi(argv[3]), h = (uint32_t)std::atoi(argv[4]);
      d2pc_b200::Bus bus;
      if (!bus.load_launch_file(argv[2])) throw std::runtime_error(std::string("cannot read ") + argv[2]);
      d2pc::Disparity2PCloud node(bus);
      std::vector<uint8_t> cloud, centres;
      int n_centres = 0;
      bus.subscribe_cloud("/point_cloud", 1, [&](const sm::PointCloud2 &c) { cloud = ros_lite::serialize(c); });
      bus.subscribe_cloud("/octomap_point_cloud_centers", 1, [&](const sm::PointCloud2 &c) {
        centres = ros_lite::serialize(c);
        ++n_centres;
      });
      for (int i = 7; i < argc; ++i)  // frame i - 7 stamped (3 + i - 7, 4)
        bus.publish(bus.resolve("/disparity"), make_image(read_file(argv[i], (size_t)w * h), w, h, 3 + (i - 7), 4));
      if (n_centres != argc - 7) throw std::runtime_error("not one centres cloud per frame");
      write_file(argv[5], cloud);
      write_file(argv[6], centres);
      return 0;
    }
    if (mode == "wire-octomap" && argc == 3) {
      ros_lite::octomap_msgs::Octomap m;
      m.header.seq = 7, m.header.stamp.sec = 11, m.header.stamp.nsec = 13, m.header.frame_id = "/map";
      m.binary = 1, m.id = "OcTree", m.resolution = 0.05;
      m.data = {0, -128, 0x3F, -1, 1};
      auto bytes = ros_lite::serialize(m);
      auto back = ros_lite::deserialize_octomap(bytes.data(), bytes.size());
      if (ros_lite::serialize(back) != bytes || back.id != "OcTree" || back.data.size() != 5)
        throw std::runtime_error("Octomap round trip differs");
      write_file(argv[2], bytes);
      return 0;
    }
    if (mode == "node1octomap" && argc >= 10) {
      const uint32_t w = (uint32_t)std::atoi(argv[3]), h = (uint32_t)std::atoi(argv[4]);
      d2pc_b200::Bus bus;
      if (!bus.load_launch_file(argv[2])) throw std::runtime_error(std::string("cannot read ") + argv[2]);
      d2pc::Disparity2PCloud node(bus);
      bool map_on = false;
      for (const auto &a : bus.advertised()) map_on = map_on || a.topic == "/octomap_point_cloud_centers";
      std::vector<uint8_t> cloud, centres, full, binary;
      bus.subscribe_cloud("/point_cloud", 1, [&](const sm::PointCloud2 &c) { cloud = ros_lite::serialize(c); });
      if (map_on) {
        bus.subscribe_cloud("/octomap_point_cloud_centers", 1,
                            [&](const sm::PointCloud2 &c) { centres = ros_lite::serialize(c); });
        if (std::string(argv[7]) != "-")
          bus.subscribe_octomap("/octomap_full", 1,
                                [&](const ros_lite::octomap_msgs::Octomap &m) { full = ros_lite::serialize(m); });
        if (std::string(argv[8]) != "-")
          bus.subscribe_octomap("/octomap_binary", 1,
                                [&](const ros_lite::octomap_msgs::Octomap &m) { binary = ros_lite::serialize(m); });
      } else {
        for (const auto &a : bus.advertised())
          if (a.topic.find("octomap") != std::string::npos) throw std::runtime_error("map off, " + a.topic + " advertised");
      }
      for (int i = 9; i < argc; ++i)  // frame i - 9 stamped (3 + i - 9, 4)
        bus.publish(bus.resolve("/disparity"), make_image(read_file(argv[i], (size_t)w * h), w, h, 3 + (i - 9), 4));
      write_file(argv[5], cloud);
      write_file(argv[6], centres);
      if (std::string(argv[7]) != "-") write_file(argv[7], full);
      if (std::string(argv[8]) != "-") write_file(argv[8], binary);
      return 0;
    }
    if (mode == "wire-grid" && argc == 3) {
      ros_lite::nav_msgs::OccupancyGrid m;
      m.header.seq = 7, m.header.stamp.sec = 11, m.header.stamp.nsec = 13, m.header.frame_id = "/map";
      m.info.map_load_time.sec = 17, m.info.map_load_time.nsec = 19;
      m.info.resolution = 0.05f, m.info.width = 3, m.info.height = 2;
      m.info.origin.position.x = -1.25, m.info.origin.position.y = 2.5, m.info.origin.position.z = 0.125;
      m.info.origin.orientation.w = 1.0;
      m.data = {-1, 0, 100, 100, 0, -1};
      auto bytes = ros_lite::serialize(m);
      auto back = ros_lite::deserialize_grid(bytes.data(), bytes.size());
      if (ros_lite::serialize(back) != bytes || back.info.width != 3 || back.data.size() != 6)
        throw std::runtime_error("OccupancyGrid round trip differs");
      write_file(argv[2], bytes);
      return 0;
    }
    if (mode == "node1projmap" && argc >= 9) {
      const uint32_t w = (uint32_t)std::atoi(argv[3]), h = (uint32_t)std::atoi(argv[4]);
      d2pc_b200::Bus bus;
      if (!bus.load_launch_file(argv[2])) throw std::runtime_error(std::string("cannot read ") + argv[2]);
      d2pc::Disparity2PCloud node(bus);
      bool map_on = false;
      for (const auto &a : bus.advertised()) map_on = map_on || a.topic == "/octomap_point_cloud_centers";
      std::vector<uint8_t> cloud, grid;
      int grids = 0;
      bus.subscribe_cloud("/point_cloud", 1, [&](const sm::PointCloud2 &c) { cloud = ros_lite::serialize(c); });
      if (map_on) {
        bus.subscribe_grid("/projected_map", 1, [&](const ros_lite::nav_msgs::OccupancyGrid &m) {
          grid = ros_lite::serialize(m);
          ++grids;
        });
      } else {
        for (const auto &a : bus.advertised())
          if (a.topic == "/projected_map") throw std::runtime_error("map off, " + a.topic + " advertised");
      }
      for (int i = 8; i < argc; ++i)  // frame i - 8 stamped (3 + i - 8, 4)
        bus.publish(bus.resolve("/disparity"), make_image(read_file(argv[i], (size_t)w * h), w, h, 3 + (i - 8), 4));
      write_file(argv[5], cloud);
      write_file(argv[6], grid);
      const std::string count = std::to_string(grids) + "\n";
      write_file(argv[7], std::vector<uint8_t>(count.begin(), count.end()));
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
    if (mode == "node1settings" && argc == 3) {
      d2pc_b200::Bus bus;
      if (!bus.load_launch_file(argv[2])) throw std::runtime_error(std::string("cannot read ") + argv[2]);
      const d2pc_b200::CloudSettings s = d2pc_b200::read_cloud_settings(bus);
      auto put = [](const std::string &name, double v) { std::printf("%s %.17g\n", name.c_str(), v); };
      auto put_n = [&put](const std::string &name, const float *v, int n) {
        for (int i = 0; i < n; ++i) put(name + "." + std::to_string(i), v[i]);
      };
#define D2PC_PUT(field) put(#field, s.field)
      D2PC_PUT(config.fx), D2PC_PUT(config.fy), D2PC_PUT(config.cx), D2PC_PUT(config.cy), D2PC_PUT(config.baseline);
      D2PC_PUT(voxel_on), D2PC_PUT(voxel.leaf_x), D2PC_PUT(voxel.leaf_y), D2PC_PUT(voxel.leaf_z);
      D2PC_PUT(voxel.min_points_per_voxel), D2PC_PUT(voxel.limit_field), D2PC_PUT(voxel.limit_min);
      D2PC_PUT(voxel.limit_max), D2PC_PUT(ror_radius), D2PC_PUT(ror_min_neighbors), D2PC_PUT(crop_box.enabled);
      put_n("crop_box.min_pt", s.crop_box.min_pt, 3), put_n("crop_box.max_pt", s.crop_box.max_pt, 3);
      put_n("crop_box.transform", s.crop_box.transform, 12);
      D2PC_PUT(transform.enabled), put_n("transform.matrix", s.transform.matrix, 12);
      D2PC_PUT(scan.enabled), D2PC_PUT(scan.min_height), D2PC_PUT(scan.max_height), D2PC_PUT(scan.angle_min);
      D2PC_PUT(scan.angle_max), D2PC_PUT(scan.angle_increment), D2PC_PUT(scan.scan_time), D2PC_PUT(scan.range_min);
      D2PC_PUT(scan.range_max), D2PC_PUT(scan.use_inf), D2PC_PUT(scan.inf_epsilon), D2PC_PUT(scan.keep_cloud);
      D2PC_PUT(map.enabled), D2PC_PUT(map.resolution), D2PC_PUT(map.prob_hit), D2PC_PUT(map.prob_miss);
      D2PC_PUT(map.clamp_min), D2PC_PUT(map.clamp_max), D2PC_PUT(map.occupancy_thres), D2PC_PUT(map.max_range);
      D2PC_PUT(map.max_bricks), D2PC_PUT(map.keep_cloud), D2PC_PUT(projected_map.occupancy_min_z);
      D2PC_PUT(projected_map.occupancy_max_z), D2PC_PUT(projected_map.min_x_size), D2PC_PUT(projected_map.min_y_size);
      D2PC_PUT(publish_cloud);
#undef D2PC_PUT
      std::printf("frame_id %s\n", s.frame_id.c_str());
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
