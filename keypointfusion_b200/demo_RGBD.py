"""Drop-in for the per-frame numpy front end of the reference's demo_RGBD.py (Model_RGBD, demo_RGBD.py:65-173), batched on the
GPU: bbox -> centre, RGB / depth crops with the reference's exact integer geometry (comToBounds, cv2 INTER_NEAREST, centred
paste), depth normalisation, back-projection + 1024-point resample + clamp.  SURVEY.md 8f-3 / BASELINE.json config 5."""
import torch

from . import ops


class Model_RGBD(object):
    """Front end + (optionally) the network.  `net`: a keypointfusion_b200.model.model.KPFusion with backbones, or None when
    only the preprocessing is wanted.  `cam_para` = (fx, fy, fu, fv) as in demo_RGBD.py:585.

    Frames and hands: rgb [F,Hf,Wf,3], depth [F,Hf,Wf] and bbox [B,4], one box per hand; `frame_index` [B] says which frame box b
    is in (None: frame b, F == B), so a frame with two hands is uploaded and stored once.  See ops.frame_index_arg for how
    indices are checked."""

    def __init__(self, net=None, cam_para=(617.0, 617.0, 312.0, 241.0), cube=(250, 250, 250), img_size=128, sample_num=1024, seed=0):
        self.net, self.cam_para, self.cube, self.img_size, self.sample_num, self.seed = net, tuple(cam_para), list(cube), img_size, sample_num, seed
        self.flip = 1
        from .dataloader.loader import loader
        self.depthloader = loader(img_size=img_size)   # the geometry helper the reference passes to net() (demo_RGBD.py:111)
        self._consts = {}

    def _const(self, device):
        """cam (f64 and f32) and cube as device tensors, made once per device: no host-to-device copy inside a captured step."""
        c = self._consts.get(device)
        if c is None:
            c = self._consts[device] = dict(cam64=torch.tensor(self.cam_para, dtype=torch.float64, device=device),
                                            cam32=torch.tensor(self.cam_para, dtype=torch.float32, device=device),
                                            cube=torch.tensor(self.cube, dtype=torch.float32, device=device))
        return c

    # demo_RGBD.py:253-276 (batched: depth [F,Hf,Wf] uint16 on the GPU, bbx [B,4] xywh)
    def get_center_from_bbx(self, depth, bbx, upper=1500, lower=171, frame_index=None):
        return ops.center_from_bbox(depth, bbx, upper, lower, frame_index=frame_index)

    # demo_RGBD.py:464-517 + ToTensor()/255 (:87)
    def Crop_Image_deep_pp_RGB(self, rgb, com, size=None, dsize=None, paras=None, frame_index=None):
        size = self._const(rgb.device)["cube"] if size is None else size
        paras = self._const(rgb.device)["cam64"] if paras is None else paras
        return ops.crop_rgb(rgb, com, size, paras, (dsize or (self.img_size,))[0], frame_index=frame_index)

    # demo_RGBD.py:305-343
    def process_depth(self, cube_size, depth, center, frame_index=None):
        k = self._const(depth.device)
        img, M, com3d, cube = ops.crop_depth(depth, center, cube_size, k["cam64"], self.img_size, frame_index=frame_index)
        cam = k["cam32"].expand(img.shape[0], 4).contiguous()
        pcl, _ = ops.getpcl(img, com3d, cube, M, cam, self.sample_num, seed=self.seed, clamp=True, flip=self.flip)  # :319-332
        return img, pcl, com3d, M, cube

    def prepare_batch(self, rgb, depth, bbox, frame_index=None):
        """rgb [F,Hf,Wf,3] uint8 (BGR), depth [F,Hf,Wf] uint16, bbox [B,4] -> the nine tensors KPFusion.forward consumes, plus
        center_uvd and frame_index (None or the [B] int32 device tensor the crops used)."""
        fi = ops.frame_index_arg(frame_index, torch.as_tensor(bbox).numel() // 4, depth.shape[0], depth.device)
        center_uvd = self.get_center_from_bbx(depth, bbox, frame_index=fi)
        img_rgb = self.Crop_Image_deep_pp_RGB(rgb, center_uvd, frame_index=fi)
        img, pcl, com3d, M, cube = self.process_depth(self._const(depth.device)["cube"], depth, center_uvd, frame_index=fi)
        cam = self._const(depth.device)["cam32"].expand(img.shape[0], 4).contiguous()
        return dict(img_rgb=img_rgb, img=img, pcl=pcl, center=com3d, M=M, cube=cube, cam_para=cam, center_uvd=center_uvd, frame_index=fi)

    def to_frame(self, joints, batch):
        """Normalised joints [B,J,3] (any of the four sets KPFusion returns) -> (uvd_frame [B,J,3]: pixels of the frame and depth
        in mm, xyz_cam [B,J,3]: camera-space mm), the first half of the reference's post-processing (demo_RGBD.py:115-147,
        xyz_nl2uvdnl_tensor without the crop transform M)."""
        return ops.joints_to_frame(joints, batch["center"], batch["cube"], batch["cam_para"], self.flip)

    def estimate_pose_RGBD(self, rgb, depth, bbox, frame_index=None):
        """Batched demo_RGBD.py:65-131: returns (result list of KPFusion.forward, batch dict).  The batch dict also holds
        joints_uvd_frame and joints_xyz_cam, result[-1] in frame pixels and camera millimetres (to_frame)."""
        if self.net is None:
            raise RuntimeError("Model_RGBD was built without a network")
        b = self.prepare_batch(rgb, depth, bbox, frame_index)
        with torch.no_grad():
            result, spatial_weight, _ = self.net(b["img_rgb"], b["img"], b["pcl"], self.depthloader, b["center"], b["M"], b["cube"], b["cam_para"], 0.8)
            b["joints_uvd_frame"], b["joints_xyz_cam"] = self.to_frame(result[-1], b)
        return result, b
