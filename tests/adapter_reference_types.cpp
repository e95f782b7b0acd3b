// Compiles include/rtb200_renderer.hpp against the REAL value types of the reference (triangle.h, materials.h, image.h,
// mat.h, vec.h, included from the original's tp2 directory, RTB200_REFERENCE, where they lie -- nothing is copied) and instantiates every templated
// member with them: the duck-typing the adapter relies on is checked against the reference's own declarations, not
// against stand-in structs.  CPU-only translation unit; built as an object file by tests/test_abi.py (no GPU, not run).
#include <vector>

#include "triangle.h"
#include "materials.h"
#include "image.h"
#include "mat.h"
#include "vec.h"
#include <QImage>          // oracle/qt_shim: the only Qt type the path touches

#include "rtb200_renderer.hpp"

// what QT/mainWindowThreads.cpp:39-65 and QT/mainwindow.cpp:108-312 do with a Renderer, type for type
void drive_with_reference_types(rtb200::Renderer& renderer, const std::vector<Triangle>& triangles, const Materials& materials,
                                const Image& map, const Image (&faces)[6], const Transform& transform, QImage& target)
{
    renderer.set_triangles(triangles);                       // std::vector<Triangle>, renderer.cpp:137
    renderer.set_materials(materials);                       // Materials, renderer.cpp:150
    renderer.set_ao_map(map);
    renderer.set_diffuse_map(map);
    renderer.set_normal_map(map);
    renderer.set_roughness_map(map);
    renderer.set_displacement_map(map);
    renderer.set_skysphere(map);
    renderer.set_skybox(faces);
    renderer.set_light_position(Point(3, 3, 2));
    renderer.set_camera_transform(transform);
    renderer.set_object_transform(Translation(Vector(0, -2, -4)) * transform);
    renderer.add_sphere(Point(0, 0, -3), 0.5f, 0);
    renderer.add_plane(Point(0, -2, 0), Vector(0, 1, 0), 0);
    renderer.change_render_size(1280, 720);
    renderer.change_camera_fov(80.0f);
    renderer.ray_trace();
    renderer.post_process();
    renderer.load_obj("data/Robot/robot.obj", nullptr);
    renderer.clear_image();
    renderer.raster_trace();
    renderer.post_process();
    renderer.copy_to(target);
}
