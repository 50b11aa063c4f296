// TEST INFRASTRUCTURE, used only by tests/golden/make_reference_map_golden.py.  The reference's laserMapping.cpp driven by
// oracle/ref_drivers/ref_mapping.cc (included as it is), plus read access to what the node publishes at the end of a frame
// (laserMapping.cpp:803-848): the stand-in bus of oracle/ref_shim keeps the last message and a count per topic.
#include "../../oracle/ref_drivers/ref_mapping.cc"

extern "C" {

// the last cloud published on `topic` (/laser_cloud_surround, /laser_cloud_map, /velodyne_cloud_registered): number of points
// (-1 if none yet), up to cap of them into out
int ref_map_cloud(const char* topic, float* out, int cap) {
  ros::shim::Bus& b = ros::shim::Bus::get();
  auto it = b.last.find(topic);
  if (it == b.last.end()) return -1;
  const sensor_msgs::PointCloud2& m = *std::static_pointer_cast<const sensor_msgs::PointCloud2>(it->second);
  const int n = (int)(m.xyzi.size() / 4);
  if (out) std::memcpy(out, m.xyzi.data(), sizeof(float) * 4 * (size_t)(n < cap ? n : cap));
  return n;
}

// number of messages published on `topic` so far
long ref_map_published(const char* topic) {
  ros::shim::Bus& b = ros::shim::Bus::get();
  auto it = b.count.find(topic);
  return it == b.count.end() ? 0 : it->second;
}

}  // extern "C"
