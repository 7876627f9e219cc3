// k_x448.cu -- explicit kernel instantiations (see launch.cuh)
#include "launch.cuh"
INSTANTIATE_SM(SlotX448)
INSTANTIATE_SM(SlotX448Peer)
INSTANTIATE_SM(SlotX448PeerLookup)
INSTANTIATE_PLAIN(LaneX448PeerLookup)
INSTANTIATE_PLAIN(LaneX448PeerLift)
