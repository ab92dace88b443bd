// reference_prior.cu — the reference's prior policy as a program (include/swarm_prior_api.cuh).
//
// robotPolicy of cus_gym/gym/envs/customized_envs/envs_cplus/src/AssemblyEnv.cpp (CPP:1121-1196), called by
// calculateActionPrior (CPP:1061-1118) for every agent.  It is the template for generated priors: the arithmetic is the
// reference's, in its order, so the prior it gives equals the simulator's built-in one bit for bit.
#include "swarm_prior_api.cuh"

__device__ void robot_policy(const swarm_agent &a, double out[2]) {
    double fx = 0.0, fy = 0.0;

    // attraction to the target: the agent's own position when it is in the shape, else the nearest cell (CPP:1102, 1136-1148)
    const double tx = a.in_shape ? a.x : a.cell_x;
    const double ty = a.in_shape ? a.y : a.cell_y;
    const double dirx = tx - a.x, diry = ty - a.y;                  // CPP:1142
    const double dist = sqrt(dirx * dirx + diry * diry);            // CPP:1143-1144
    if (dist > 0) {                                                 // CPP:1145-1148
        fx += 2.0 * dirx / dist;
        fy += 2.0 * diry / dist;
    }

    // repulsion from listed neighbours closer than r_avoid, and their mean velocity (CPP:1151-1180)
    double avx = 0.0, avy = 0.0;
    for (int q = 0; q < a.count; ++q) {
        const int j = a.neighbor(q);
        const swarm_xy pj = a.pos(j), vj = a.vel(j);
        const double ddx = a.x - pj.x, ddy = a.y - pj.y;            // CPP:1162
        const double dn = sqrt(ddx * ddx + ddy * ddy);              // CPP:1163
        if (dn > 0 && dn < a.r_avoid) {                             // CPP:1166-1174
            const double ux = ddx / dn, uy = ddy / dn;
            const double factor = 3.0 * (a.r_avoid / dn - 1.0);
            fx += factor * ux;
            fy += factor * uy;
        }
        avx += vj.x;                                                // CPP:1177-1178
        avy += vj.y;
    }
    if (a.count > 0) {                                              // CPP:1183-1189: velocity alignment
        avx /= a.count;
        avy /= a.count;
        fx += 2.0 * (avx - a.vx);
        fy += 2.0 * (avy - a.vy);
    }

    // clamp(f, -1, 1) = std::max(-1, std::min(f, 1)) (CPP:11-14, 1192-1193)
    const double cx = (1.0 < fx) ? 1.0 : fx, cy = (1.0 < fy) ? 1.0 : fy;
    out[0] = (-1.0 < cx) ? cx : -1.0;
    out[1] = (-1.0 < cy) ? cy : -1.0;
}
