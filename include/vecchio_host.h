/*
 * vecchio_host.h -- C view of the host front end (vecchio_b200/host/vecchio.hpp) for callers
 * that cannot include C++ (the Python tests and bench.py).  It builds a scene with the
 * reference's scene API (src/scene.rs builders), builds the world BVH like src/main.rs:168,
 * lowers both to a vk_scene_desc, and steps the scene's camera iterator (src/main.rs:176).
 * Nothing here computes a hit or a colour.
 */
#ifndef VECCHIO_HOST_H
#define VECCHIO_HOST_H

#include "vecchio_gpu.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vkh_scene vkh_scene;

/* name: balls_demo | random_spheres_demo | perlin_demo | bowser_demo | cornell_box |
 *       final_scene | cornell_smoke | stress_spheres (param = grid side, 1000 => 1M spheres) |
 *       api_surface_demo (SpecDiffuse, sphere and box lights) |
 *       random_spheres_cover (random_spheres_demo without its light: sky-lit, legacy integrator only) |
 *       book1_cover (the book-1 final scene of sample/inoneweekend.png: grey ground, fixed camera; legacy only) |
 *       furnace_demo (param = 0 Lambertian | 1 Metal | 2 Dielectric | 3 white-medium sphere inside an emitting shell; closed form |
 *                     4 the Lambertian one in a shell 1000x as bright, samples above adaptive sampling's 255 clamp)
 * seed: seeds the host RNG standing in for rand::thread_rng() (scene + BVH axis choices).
 * assets_dir: directory holding earthmap.png etc. (NULL => "assets"). */
int vkh_scene_build(const char* name, uint64_t seed, const char* assets_dir, uint32_t param, vkh_scene** out);
void vkh_scene_free(vkh_scene* s);
const vk_scene_desc* vkh_scene_desc(const vkh_scene* s);
float vkh_scene_aspect_ratio(const vkh_scene* s);
/* cam_iter.next(): 1 = camera written, 0 = iterator exhausted */
int vkh_scene_next_camera(vkh_scene* s, vk_camera* out);
/* Camera::new (src/main.rs:71-109) */
void vkh_camera_new(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov,
                    float aspect_ratio, float aperture, float focus_dist, float time0, float time1,
                    vk_camera* out);
/* ImageTexture::new (src/material.rs:269-279): decoded RGB8 bytes; returns byte count or -1.
 * buf may be NULL to query the size. */
long vkh_decode_png(const char* path, uint8_t* buf, size_t buf_len, uint32_t* width, uint32_t* height);
/* Output conversion of src/main.rs:201-214 on the host: frame = W*H*3 linear floats, pixel i = y*W+x, row 0 =
 * bottom (what vk_render writes); out_rgb8 = the W*H*3 numbers of the reference's P3 file in file order
 * (row height-1 first), every channel through Vec3::to_color (src/vec3.rs:54-61: (256*clamp(sqrt(c),0,0.999))
 * as u32, NaN -> 0).  vk_render_rgb8 does the same on the device; this one serves frames that were summed on
 * the host (several GPUs in one process, merged checkpoints). */
void vkh_frame_to_rgb8(const float* frame, uint32_t width, uint32_t height, uint8_t* out_rgb8);
/* The file writer of src/main.rs:201-213: "P3", "W H", "255", then one "r g b" line per pixel in the order
 * of rgb8 (file order, as vk_render_rgb8 / vkh_frame_to_rgb8 produce it).  0 = OK, VK_ERR_INVALID on an I/O
 * failure (message in vkh_last_error) where the reference unwraps File::create. */
int vkh_write_ppm(const char* path, const uint8_t* rgb8, uint32_t width, uint32_t height);
/* A little-endian PFM of one frame plane: "PF" (channels 3) or "Pf" (channels 1), "W H", scale "-1.0" (the sign
 * says little-endian), then the W*H*channels floats row 0 first -- PFM stores rows bottom-to-top, the order of
 * vk_render's and vk_render_aov's planes, so nothing is flipped.  0 = OK, VK_ERR_INVALID for channels other than
 * 1 or 3, a null argument or an I/O failure (message in vkh_last_error). */
int vkh_write_pfm(const char* path, const float* data, uint32_t width, uint32_t height, uint32_t channels);
/* "output_{:04}.ppm" (src/main.rs:201) under dir (NULL or "" = current directory) into buf; returns the length
 * or -1 if buf is too small. */
int vkh_frame_filename(const char* dir, uint32_t file_idx, char* buf, size_t buf_len);
const char* vkh_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
