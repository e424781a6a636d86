// rtrb_trace_fast_launch.cuh — the FAST64 kernels of every class build (rtrb_trace.cuh, "build policies").  The
// kernels carry their class as a namespace: rtrb_fast (generic), rtrb_fast_lean, rtrb_fast_l1 (one light) and
// rtrb_fast_l1n (one light, no Monte-Carlo rays).  Each rtrb_trace_fast_*.cu translation unit instantiates one
// (class, work-stack capacity) pair, so `make -j` compiles them in parallel; rtrb_trace_fast.cu launches them.
#pragma once
#include <type_traits>

#include "rtrb_launch.h"
#include "rtrb_trace_fast.cuh"

// One class build's kernels for one work-stack capacity (1: the stackless depth-1 kernels), indexed
// [count_detail][use_bvh], and the class they were compiled for.  pass: progressive-frame passes (generic build only,
// nullptr elsewhere).
struct FastKernels {
  bool one_light, lean, no_mc;
  int capacity;
  TraceKernel pre[2][2], extra[2][2], pass[2][2];
};

namespace rtrb_fast { using Pol = rtrb::Generic;
#include "rtrb_trace_fast_build.cuh"
}
namespace rtrb_fast_lean { using Pol = rtrb::Lean;
#include "rtrb_trace_fast_build.cuh"
}
namespace rtrb_fast_l1 { using Pol = rtrb::OneLight;
#include "rtrb_trace_fast_build.cuh"
}
namespace rtrb_fast_l1n { using Pol = rtrb::OneLightNoMc;
#include "rtrb_trace_fast_build.cuh"
}

// The builds, one object each (rtrb_trace_fast_{d1,d1lean,t10,t10_l1,t10_l1n,t32,t32_l1,t32_l1n,t128}.cu): the lean
// build has depth-1 kernels only, the one-light builds ray-tree kernels only (the depth-1 frames of their classes run
// the generic build).
namespace rtrb_fast { extern const FastKernels d1, t10, t32, t128; }
namespace rtrb_fast_lean { extern const FastKernels d1; }
namespace rtrb_fast_l1 { extern const FastKernels t10, t32; }
namespace rtrb_fast_l1n { extern const FastKernels t10, t32; }
