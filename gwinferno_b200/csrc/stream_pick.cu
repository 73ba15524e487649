// dispatch to the per-dimension-count instantiation units
#include "stream_cta.cuh"
namespace gwi {
stream_fn pick_stream_ns0(int nd, int nlin, bool g2, bool param, bool maxonly);
stream_fn pick_stream_ns1(int nd, int nlin, bool g2, bool param, bool maxonly);
stream_fn pick_stream_ns2(int nd, int nlin, bool g2, bool param, bool maxonly);
stream_fn pick_stream_ns3(int nd, int nlin, bool g2, bool param, bool maxonly);
stream_fn pick_stream_ns4(int nd, int nlin, bool g2, bool param, bool maxonly);
stream_fn pick_stream_ns5(int nd, int nlin, bool g2, bool param, bool maxonly);
stream_fn pick_stream_ns6(int nd, int nlin, bool g2, bool param, bool maxonly);
stream_fn pick_stream_ns7(int nd, int nlin, bool g2, bool param, bool maxonly);
stream_fn pick_stream_ns8(int nd, int nlin, bool g2, bool param, bool maxonly);

stream_fn pick_stream_kernel(int ns, int ndeep, int nlin, bool g2, bool param, bool maxonly) {
  switch (ns) {
    case 0: return pick_stream_ns0(ndeep, nlin, g2, param, maxonly);
    case 1: return pick_stream_ns1(ndeep, nlin, g2, param, maxonly);
    case 2: return pick_stream_ns2(ndeep, nlin, g2, param, maxonly);
    case 3: return pick_stream_ns3(ndeep, nlin, g2, param, maxonly);
    case 4: return pick_stream_ns4(ndeep, nlin, g2, param, maxonly);
    case 5: return pick_stream_ns5(ndeep, nlin, g2, param, maxonly);
    case 6: return pick_stream_ns6(ndeep, nlin, g2, param, maxonly);
    case 7: return pick_stream_ns7(ndeep, nlin, g2, param, maxonly);
    case 8: return pick_stream_ns8(ndeep, nlin, g2, param, maxonly);
  }
  return nullptr;
}

stream_fn pick_stream_cta_ns1(int nd, int nlin);
stream_fn pick_stream_cta_ns2(int nd, int nlin);
stream_fn pick_stream_cta_ns3(int nd, int nlin);
stream_fn pick_stream_cta_ns4(int nd, int nlin);
stream_fn pick_stream_cta_ns5(int nd, int nlin);
stream_fn pick_stream_cta_ns6(int nd, int nlin);
stream_fn pick_stream_cta_ns7(int nd, int nlin);
stream_fn pick_stream_cta_ns8(int nd, int nlin);

stream_fn pick_stream_cta_kernel(int ns, int ndeep, int nlin) {
  switch (ns) {
    case 1: return pick_stream_cta_ns1(ndeep, nlin);
    case 2: return pick_stream_cta_ns2(ndeep, nlin);
    case 3: return pick_stream_cta_ns3(ndeep, nlin);
    case 4: return pick_stream_cta_ns4(ndeep, nlin);
    case 5: return pick_stream_cta_ns5(ndeep, nlin);
    case 6: return pick_stream_cta_ns6(ndeep, nlin);
    case 7: return pick_stream_cta_ns7(ndeep, nlin);
    case 8: return pick_stream_cta_ns8(ndeep, nlin);
  }
  return nullptr;
}
stream_fn pick_stream_cta_max_kernel() { return (stream_fn)stream_cta_max_kernel<0>; }
}  // namespace gwi
