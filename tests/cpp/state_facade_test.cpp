// Checkpoint / resume through the C++ facade: StateOptions rejects a damaged blob without a device; with one, a handle
// created from StateOptions(blob) loads the blob, and saving it again gives the same bytes. Without a usable device the
// constructor fails with CTICP_ERR_NO_DEVICE: exit 42.
#include <cstdio>
#include <vector>

#include "ct_icp_b200/odometry.hpp"

int main() {
    try {
        ct_icp::Odometry::StateOptions(std::vector<uint8_t>(16, 0));
        std::printf("a 16-byte blob was accepted\n");
        return 1;
    } catch (const ct_icp::CticpFailure &e) {
        if (e.code != CTICP_ERR_INVALID_ARGUMENT) {
            std::printf("unexpected status %d: %s\n", e.code, e.what());
            return 1;
        }
    }
    try {
        ct_icp::OdometryOptions options;
        options.init_num_frames = 5;
        options.map_options.capacity_voxels = 2048;
        ct_icp::Odometry a(options);
        const std::vector<uint8_t> blob = a.SaveState();
        ct_icp::OdometryOptions restored = ct_icp::Odometry::StateOptions(blob);
        if (restored.init_num_frames != 5 || restored.map_options.capacity_voxels != 2048) {
            std::printf("StateOptions did not return the saved options\n");
            return 1;
        }
        restored.map_options.capacity_voxels = 8192;   // sizes the tables only
        ct_icp::Odometry b(restored);
        b.LoadState(blob);
        std::vector<uint8_t> again = b.SaveState();
        if (again.size() != blob.size()) {
            std::printf("blob sizes differ: %zu vs %zu\n", again.size(), blob.size());
            return 1;
        }
        std::printf("STATE FACADE OK (%zu bytes)\n", blob.size());
        return 0;
    } catch (const ct_icp::CticpFailure &e) {
        std::printf("%s\n", e.what());
        return e.code == CTICP_ERR_NO_DEVICE ? 42 : 1;
    }
}
