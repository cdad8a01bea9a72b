/*
 * ref_shim.cpp -- TEST INFRASTRUCTURE: exposes the reference's OWN metric code through a C ABI.
 *
 * It compiles the reference's src/Point.h and src/Distance.h from where they lie (the build
 * recipe passes -I$(REF) to that directory; nothing is copied into this repository) against a minimal
 * stand-in for the only two CGAL names Distance.h mentions (src/Distance.h:4,14:
 * CGAL::Dimension_tag, CGAL::Kd_tree_rectangle with min_coord / max_coord).  CGAL's kd-tree search
 * itself is absent from this image, so the neighbour SEARCH stays unpinned; what this pins, bit
 * for bit, is everything the reference contributes to the arithmetic of the path:
 *   - Distance::transformed_distance(p, q)            src/Distance.h:6-11
 *   - Distance::min_distance_to_rectangle(p, b, d)    src/Distance.h:27-57
 *   - Distance::new_distance                          src/Distance.h:92-95
 *   - Distance::transformed_distance(d) / inverse     src/Distance.h:97,99
 *   - sizeof(Point) and its field offsets             src/Point.h:1-6
 * Output: oracle/_ref/libref_metric.so (git-ignored; built only where PT_REFERENCE_SRC is set).
 * Only tests/ may load it.
 */
#include <cmath>
#include <cstddef>
#include <string>
#include <vector>

namespace CGAL {
template <int N> struct Dimension_tag { static const int value = N; };
template <class FT, class D> struct Kd_tree_rectangle {
    FT lo[3], hi[3];
    FT min_coord(int i) const { return lo[i]; }
    FT max_coord(int i) const { return hi[i]; }
};
}  // namespace CGAL

#include "Point.h"      // the reference's, via -I$(REF)
#include "Distance.h"   // the reference's

extern "C" {

void ref_point_layout(int out[6])
{
    out[0] = (int)sizeof(Point);
    out[1] = (int)offsetof(Point, ver);
    out[2] = (int)offsetof(Point, normal);
    out[3] = (int)offsetof(Point, color);
    out[4] = (int)offsetof(Point, U);
    out[5] = (int)offsetof(Point, V);
}

double ref_transformed_distance(const void *p1, const void *p2)
{
    Distance d;
    return d.transformed_distance(*static_cast<const Point *>(p1), *static_cast<const Point *>(p2));
}

double ref_min_distance_to_rectangle(const void *p, const double lo[3], const double hi[3],
                                     double dists[3])
{
    Distance d;
    CGAL::Kd_tree_rectangle<double, CGAL::Dimension_tag<3> > b;
    for (int i = 0; i < 3; ++i) { b.lo[i] = lo[i]; b.hi[i] = hi[i]; }
    std::vector<double> v(dists, dists + 3);
    const double r = d.min_distance_to_rectangle(*static_cast<const Point *>(p), b, v);
    for (int i = 0; i < 3; ++i) dists[i] = v[i];
    return r;
}

double ref_new_distance(double dist, double old_off, double new_off)
{
    Distance d;
    return d.new_distance(dist, old_off, new_off, 0);
}

double ref_transformed_radius(double r)
{
    Distance d;
    return d.transformed_distance(r);
}

double ref_inverse_of_transformed_distance(double t)
{
    Distance d;
    return d.inverse_of_transformed_distance(t);
}

}  // extern "C"
