"""Host/shader shared POD layouts of the reference, as numpy dtypes.

Mirrors /root/reference/src/rendering_backend/glsl_common.h:31-99 byte for byte (sizes verified against
the header compiled with g++: PerFrameData 584, DirectionalLight 112, Vertex 56, Material 44,
Primitive 120, SVGFPushConstants 24, SSAOPushConstants 4). Matrices are glm column-major (m[c][r]).
"""
import numpy as np

MAT4 = (np.float32, (4, 4))  # stored [column][row], like glm

DirectionalLight = np.dtype([
    ("projview", *MAT4),
    ("direction", np.float32, 4),
    ("color", np.float32, 4),
    ("intensity", np.float32, 4),
])

PerFrameData = np.dtype([
    ("camera_view", *MAT4),
    ("camera_proj", *MAT4),
    ("camera_view_inverse", *MAT4),
    ("camera_proj_inverse", *MAT4),
    ("camera_viewproj_inverse", *MAT4),
    ("camera_view_prev_frame", *MAT4),
    ("camera_proj_prev_frame", *MAT4),
    ("directional_light", DirectionalLight),
    ("display_size", np.float32, 2),
    ("display_size_inverse", np.float32, 2),
    ("frame_index", np.uint32),
    ("blue_noise_texture_index", np.int32),
])

Vertex = np.dtype([
    ("pos", np.float32, 3),
    ("normal", np.float32, 3),
    ("tangent", np.float32, 4),
    ("uv0", np.float32, 2),
    ("uv1", np.float32, 2),
])

Material = np.dtype([
    ("base_color", np.float32, 4),
    ("base_color_texture", np.int32),
    ("metallic_roughness_texture", np.int32),
    ("normal_map", np.int32),
    ("metallic_factor", np.float32),
    ("roughness_factor", np.float32),
    ("alpha_mask", np.int32),
    ("alpha_cutoff", np.float32),
])

Primitive = np.dtype([
    ("transform", *MAT4),
    ("material", Material),
    ("vertex_offset", np.uint32),
    ("index_offset", np.uint32),
    ("index_count", np.uint32),
])

# vhr_shade_record (include/vhr_b200.h, vhr_debug_shade_hits): geometry index (texture kind: slot), primitive id, barycentrics of
# vertices 1 and 2 (texture kind: s, t), pixel (G-buffer kind)
ShadeRecord = np.dtype([("g", np.uint32), ("pid", np.uint32), ("u", np.float32), ("v", np.float32), ("x", np.int32), ("y", np.int32)])
SHADE_TEXTURE, SHADE_REFLECTION, SHADE_GBUFFER, SHADE_GBUFFER_ALPHA, SHADE_RAYTRACED, SHADE_RAYTRACED_ALPHA, SHADE_ANYHIT_ALPHA = range(7)
SHADE_OUT_WORDS = 8

SVGFPushConstants = np.dtype([
    ("integrated_shadow_and_ao", np.int32, 2),
    ("prev_frame_normals_and_object_ids", np.int32),
    ("shadow_and_ao_history", np.int32),
    ("shadow_and_ao_moments_history", np.int32),
    ("atrous_step", np.int32),
])

SSAOPushConstants = np.dtype([("radius", np.float32)])

SSRPushConstants = np.dtype([      # glsl_common.h:41-46
    ("ray_distance", np.float32),
    ("step_size", np.float32),
    ("thickness", np.float32),
    ("bsearch_steps", np.int32),
])

assert PerFrameData.itemsize == 584
assert DirectionalLight.itemsize == 112
assert Vertex.itemsize == 56
assert Material.itemsize == 44
assert Primitive.itemsize == 120
assert SVGFPushConstants.itemsize == 24
assert SSRPushConstants.itemsize == 16

# VkFormat values used on the hot path (hybrid_render_path.cpp:16-19,109-110,247-261)
VK_FORMAT_R8G8B8A8_UNORM = 37      # material textures (scene_loader.cpp:249-272)
VK_FORMAT_R8G8B8A8_SRGB = 43
VK_FORMAT_B8G8R8A8_UNORM = 44
VK_FORMAT_B8G8R8A8_SRGB = 50
VK_FORMAT_R16G16_SFLOAT = 83
VK_FORMAT_R16G16B16A16_SFLOAT = 97
VK_FORMAT_D32_SFLOAT = 126

FORMAT_TEXEL_BYTES = {
    VK_FORMAT_B8G8R8A8_UNORM: 4,
    VK_FORMAT_B8G8R8A8_SRGB: 4,
    VK_FORMAT_R16G16_SFLOAT: 4,
    VK_FORMAT_R16G16B16A16_SFLOAT: 8,
    VK_FORMAT_D32_SFLOAT: 4,
}
# (numpy dtype, channels) of the host-side view of each format
FORMAT_NUMPY = {
    VK_FORMAT_B8G8R8A8_UNORM: (np.uint8, 4),
    VK_FORMAT_B8G8R8A8_SRGB: (np.uint8, 4),
    VK_FORMAT_R16G16_SFLOAT: (np.float16, 2),
    VK_FORMAT_R16G16B16A16_SFLOAT: (np.float16, 4),
    VK_FORMAT_D32_SFLOAT: (np.float32, 1),
}
