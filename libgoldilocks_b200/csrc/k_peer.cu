// k_peer.cu -- explicit kernel instantiations (see launch.cuh): decaf peer sets
#include "launch.cuh"
INSTANTIATE_SM(SlotDecafPeer)
INSTANTIATE_PLAIN(LaneDecafPeerDecode)
INSTANTIATE_PLAIN(LaneDecafPeerKeys)
